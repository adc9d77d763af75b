#!/usr/bin/env python
"""bench.py — cache_aware routing decisions/sec on B200 (BASELINE.json metric, configs[1]).

  python bench.py --gpus N --steps K --warmup W            # smgx (CUDA) arm
  python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host cores (oracle port)

A "step" is one batch of B=4096 synthetic 512-token requests routed against a 64-worker fleet and a 1.0M-entry
GPU-resident positional KV index (event-driven cache_aware mode, SURVEY.md §8d config 2).
  value : whole-job decisions/s, request tokens already resident in HBM, CUDA events on the launching stream.
  e2e   : the same metric through the public C-ABI call with HOST (pinned) buffers — H2D of the tokens and D2H of
          the picks are inside the timed region (pipelined over the library's stream lanes).
Under torchrun every rank owns a full replica (fleet ≤ 512 workers ⇒ "replicas only", no data-path collective;
SURVEY §8e) and routes its own batches: weak scaling, value = all ranks' decisions ÷ max-over-ranks time.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cache_aware routing decisions/sec"
CFG = dict(cache_threshold=0.3, balance_abs_threshold=64, balance_rel_threshold=1.5, block_size=16)  # CLI defaults main.rs:156-165


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per DECISION of the dominant kernel pair, from the committed ncu --set full capture (profiles/roofline_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d["dram_bytes_per_launch_pair"] / d["decisions_per_launch_pair"]
        except Exception:  # noqa: BLE001
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_population(n_seq, T, seed):
    from smg_b200 import synth
    return synth.gen_sequences(n_seq, T, seed)


def algorithmic_bytes_per_decision(kinds, keeps, T, W, B, bs):
    """SURVEY §8d byte model for K2b + K3: 4·T tokens hashed + Pr·(32 + ceil(W/8)) index bytes + 16·W/B + 4,
    with Pr the probes the reference algorithm issues for that request (jump 64 ≥ P): full hit 2 (pos 0, pos P-1);
    novel 1; stored prefix of k blocks 2 + k (linear drain scans positions 1..k)."""
    entry = 32 + (W + 7) // 8
    pr = np.where(kinds == 0, 2, np.where(kinds == 1, 2 + keeps // bs, 1)).astype(np.float64)
    return float(4 * T + pr.mean() * entry + 16.0 * W / B + 4), float(pr.mean())


def gen_batch(seqs, B, seed, bs):
    """config-2 mix; returns tokens [B,T], kinds (0 full hit, 1 partial, 2 novel), keep (tokens kept for partials)."""
    rng = np.random.Generator(np.random.PCG64(seed + 2000))
    n_seq, T = seqs.shape
    P = T // bs
    kind_r = rng.random(B)
    pick = rng.integers(0, n_seq, size=B)
    out = rng.integers(0, 50000, size=(B, T), dtype=np.uint32)
    kinds = np.where(kind_r < 0.8, 0, np.where(kind_r < 0.9, 1, 2))
    keeps = rng.integers(1, P, size=B) * bs
    out[kinds == 0] = seqs[pick[kinds == 0]]
    for i in np.nonzero(kinds == 1)[0]:
        out[i, :keeps[i]] = seqs[pick[i], :keeps[i]]
    return out, kinds, keeps


def populate(pol, ix, seqs, W, bs):
    """31 250 sequences × 32 blocks → 1.0 M (position, content) entries, worker = i mod W (SURVEY §8d config 2)."""
    from smg_b200 import synth
    urls = synth.worker_urls(W)
    for u in urls:
        ix.intern_worker(u)
    n_seq, T = seqs.shape
    P = T // bs
    flat = np.ascontiguousarray(seqs.reshape(-1))
    hashes = np.zeros(n_seq * P, np.uint64)
    got = C.c_uint32()
    # content hashes of the whole population in a few kernel launches (convert_kv_block hashes token_ids, kv_event_monitor.rs:592)
    chunk = 4096 * T
    for off in range(0, flat.size, chunk):
        part = flat[off:off + chunk]
        nb = part.size // bs
        pol._h.call("smgx_content_hashes", part.ctypes.data_as(C.c_void_p), part.size, bs,
                    hashes[off // bs:].ctypes.data_as(C.c_void_p), nb, C.byref(got))
    seq_ids = np.arange(1, n_seq * P + 1, dtype=np.uint64)
    for s in range(n_seq):
        pol._h.call("smgx_indexer_apply_stored", ix.model, s % W, seq_ids[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p),
                    hashes[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p), P, None)
    return hashes


def populate_oracle(seqs, hashes, W, bs, jump):
    from oracle import orc
    from smg_b200 import synth
    urls = synth.worker_urls(W)
    op = orc.CacheAwarePolicy(eviction_interval_secs=0, **CFG)
    op.set_workers(urls)
    oix = orc.PositionalIndexer(jump)
    for u in urls:
        oix.intern_worker(u)
    n_seq, T = seqs.shape
    P = T // bs
    L = orc.lib()
    seq_ids = np.arange(1, n_seq * P + 1, dtype=np.uint64)
    for s in range(n_seq):
        L.orc_indexer_apply_stored(oix.h, s % W, seq_ids[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p),
                                   hashes[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p), P, 0, 0)
    op.attach_indexer("unknown", oix)
    op.set_kv_event_monitor(True)
    return op, oix


def oracle_hashes(seqs, bs):
    from oracle import orc
    n_seq, T = seqs.shape
    out = np.zeros(n_seq * (T // bs), np.uint64)
    L = orc.lib()
    for s in range(n_seq):
        row = np.ascontiguousarray(seqs[s])
        L.orc_request_content_hashes(row.ctypes.data_as(C.c_void_p), T, bs, out[s * (T // bs):].ctypes.data_as(C.c_void_p), T // bs)
    return out


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU algorithm on the box's host threads, same workload/metric.  The Rust crate cannot be built
    here (no cargo), so it is the oracle port — timed in its "port-tuned" form (oracle/tuned_event.h: flat open-addressed index, bitset
    worker sets, no per-block allocation, threads created before the clock starts; picks asserted equal to the plain port's), which is
    what `value` reports; the plain restatement's number is printed beside it.  Rank 0 only."""
    if rank != 0:
        return
    from smg_b200 import synth
    B, T, W, bs = args.batch, args.tokens, args.workers, 16
    seqs = build_population(args.sequences, T, 42)
    hashes = oracle_hashes(seqs, bs)
    op, oix = populate_oracle(seqs, hashes, W, bs, 64)
    loads = synth.poisson_loads(W, 8, 42)
    op.set_state(loads, [1] * W, [1] * W)
    batches = [synth.ragged(gen_batch(seqs, B, 42 + i, bs)[0]) for i in range(8)]
    batches = [(tk, off.astype(np.uint64)) for tk, off in batches]
    rel, ab = CFG["balance_rel_threshold"], CFG["balance_abs_threshold"]

    def tuned(steps, c):
        return op.tuned_select_steps_mt(oix, batches, steps, c, rel, ab, bs)

    # same picks from both variants on one batch before any timing is trusted
    want = op.select_batch_tokens(*batches[0])[0]
    got = op.tuned_select_steps_mt(oix, batches[:1], 1, 4, rel, ab, bs)[0]
    if not np.array_equal(want, got):
        print("reference arm: port-tuned picks differ from the plain port", file=sys.stderr)
        sys.exit(3)
    calib = {}
    if args.threads:
        cores = args.threads
    else:
        # "all the host threads it can use": SMT siblings / other tenants can make the full logical-CPU count slower than
        # fewer threads, so calibrate over {all, 1/2, 1/4, 1/8} logical CPUs on a short probe each and keep the fastest.
        ncpu = os.cpu_count() or 1
        cands = sorted({max(1, ncpu), max(1, ncpu // 2), max(1, ncpu // 4), max(1, ncpu // 8)}, reverse=True)
        best = None
        for c in cands:
            tuned(4, c)
            t_c = min(tuned(64, c)[1] for _ in range(2)) / 64
            calib[str(c)] = B / t_c
            if best is None or t_c < best[0]:
                best = (t_c, c)
        cores = best[1]
    tuned(args.warmup, cores)
    times = [tuned(args.steps, cores)[1] for _ in range(max(1, args.regions))]
    t = float(np.median(times))
    val = args.steps * B / t
    op.select_steps_mt(batches, args.warmup, cores)
    t_plain = op.select_steps_mt(batches, args.steps, cores)[1]
    # per-decision latency of the CPU path: one request on one thread (what a tokio task pays), plain and tuned
    one = [(batches[0][0][: T * 256], batches[0][1][:257])]
    per = []
    for _ in range(20):
        per.append(op.tuned_select_steps_mt(oix, one, 1, 1, rel, ab, bs)[1] / 256)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "decisions/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name(args), "batch": B, "tokens": T, "workers": W, "mode": "event_driven"},
            "cpu_baseline": {"value": val, "unit": "decisions/s", "cores": cores, "kind": "port-tuned",
                             "plain_port_value": args.steps * B / t_plain, "thread_calibration_decisions_per_s": calib,
                             "regions_s": times, "logical_cpus": os.cpu_count(),
                             "per_decision_latency_us": {"p50": float(np.percentile(per, 50) * 1e6), "p99": float(np.percentile(per, 99) * 1e6),
                                                         "what": "mean over 256 requests routed one after another on ONE thread, 20 repetitions"},
                             "sample": f"{args.steps} batches of {B} requests, read-only event-mode matching, each batch sharded over {cores} host threads created "
                                       f"before the clock starts (no barrier between steps); port-tuned = flat bitset index (oracle/tuned_event.h), picks equal to the plain port"},
            "e2e": {"value": val, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_name(args):
    return (f"config2: 1xB200 per rank, {args.workers} workers, {args.tokens}-token requests, {args.sequences * (args.tokens // 16)}-entry "
            f"positional KV index (event-driven cache_aware), batch={args.batch}, mix 80% full-hit / 10% partial / 10% novel")


def bind_numa(local_rank):
    """Pin this rank's threads + the pinned staging buffers it allocates next to the GPU's NUMA node (smgx_bind_numa)."""
    from smg_b200 import _lib
    L = _lib.load()
    node = C.c_int(-1)
    err = _lib.new_err()
    try:
        _lib.check(L.smgx_bind_numa(local_rank, C.byref(node), C.byref(err)), err)
    except Exception:  # noqa: BLE001
        return -1
    return int(node.value)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="smgx", choices=["smgx", "reference"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--tokens", type=int, default=512)
    ap.add_argument("--workers", type=int, default=64)
    ap.add_argument("--sequences", type=int, default=31250)
    ap.add_argument("--ring", type=int, default=32, help="distinct device-resident batches cycled through (ring × batch × tokens × 4 B > L2)")
    ap.add_argument("--lanes", type=int, default=4, help="stream lanes the timed steps are issued over (1 = strictly serial launches)")
    ap.add_argument("--regions", type=int, default=3, help="back-to-back timed regions of exactly --steps steps each; the median region is reported")
    ap.add_argument("--threads", type=int, default=0, help="--impl reference: host threads (0 = all cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-text-in", action="store_true", help="skip the text-in leg (GPU tokenize → pick) of the N=1 line")
    ap.add_argument("--no-per-request", action="store_true", help="skip the per-request front-end leg (smgx::Batcher, 32 blocking callers) of the N=1 line")
    ap.add_argument("--no-sharded", action="store_true", help="skip the worker-id-sharded config-4 sub-record of the N>1 line")
    ap.add_argument("--text-in", action="store_true", help="(kept for compatibility: the text-in leg is on by default at N=1)")
    ap.add_argument("--text-docs", type=int, default=8192)
    ap.add_argument("--text-bytes", type=int, default=2048)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the picks of the last timed step as DIR/picks.npy (float64, one per request of the batch; rank 0), "
                         "so that two builds can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "smgx":
        ap.error("--dump-outputs applies to --impl smgx")
    args.warmup = max(args.warmup, 3)

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    numa_node = bind_numa(local_rank)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl")

    from smg_b200 import BasicWorker, CacheAwareConfig, CacheAwarePolicy, synth
    from smg_b200 import _lib
    B, T, W, bs, R = args.batch, args.tokens, args.workers, 16, args.ring
    pol = CacheAwarePolicy(CacheAwareConfig(eviction_interval_secs=0, **CFG), device_id=local_rank, max_batch=B, max_tokens_per_request=T)
    h, L = pol._h, _lib.load()
    urls = synth.worker_urls(W)
    ws = [BasicWorker(u) for u in urls]
    loads = synth.poisson_loads(W, 8, 42)
    for w, l in zip(ws, loads):
        w.set_load(int(l))
    pol.init_workers(ws)
    mon = pol.kv_event_monitor(bs)
    ix = mon.create_indexer("unknown", 64)
    pol.set_kv_event_monitor(mon)
    seqs = build_population(args.sequences, T, 42)
    t0 = time.time()
    hashes = populate(pol, ix, seqs, W, bs)
    t_pop = time.time() - t0
    model = pol._push_fleet(ws)

    # ---- device-resident ring of distinct batches (ring × 8 MB > 126 MB L2) ----
    err = _lib.new_err()
    offsets = (np.arange(B + 1, dtype=np.uint64) * T).astype(np.uint32)
    d_off = L.smgx_device_alloc(h.p, offsets.nbytes, C.byref(err))
    h.call("smgx_memcpy_h2d", d_off, offsets.ctypes.data_as(C.c_void_p), offsets.nbytes)
    d_tok, d_out, host_batches, kinds_all, keeps_all = [], [], [], [], []
    for r in range(R):
        q, kinds, keeps = gen_batch(seqs, B, 42 + 1000 * rank + r, bs)
        kinds_all.append(kinds); keeps_all.append(keeps)
        flat = np.ascontiguousarray(q.reshape(-1))
        host_batches.append(flat)
        dt = L.smgx_device_alloc(h.p, flat.nbytes, C.byref(err))
        h.call("smgx_memcpy_h2d", dt, flat.ctypes.data_as(C.c_void_p), flat.nbytes)
        d_tok.append(dt)
        d_out.append(L.smgx_device_alloc(h.p, B * 4, C.byref(err)))
    alg_bytes, mean_pr = algorithmic_bytes_per_decision(np.concatenate(kinds_all), np.concatenate(keeps_all), T, W, B, bs)

    def barrier():
        h.call("smgx_synchronize")
        if dist is not None:
            import torch
            torch.cuda.synchronize()
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n_lanes = max(1, min(args.lanes, L.smgx_pipeline_depth(h.p)))

    def step_dev(i):
        # consecutive steps are issued round-robin over the library's stream lanes, as the host batcher does
        h.call("smgx_select_batch_tokens_device", model, i % n_lanes, d_tok[i % R], d_off, B, T, d_out[i % R], None)

    # ---- kernel-only (inputs resident in HBM) ----
    for i in range(args.warmup):
        step_dev(i)
    barrier()
    # the K timed steps are handed over in ONE C-ABI call (smgx_select_many_tokens_device): the host cost of a step is
    # then a C loop iteration, as it would be from the Rust batcher, not a Python→ctypes round trip (~5 µs)
    K = args.steps

    def region_args(reg):   # region `reg` walks the ring from a different start, so no region re-reads what the previous one left in L2
        order = [(args.warmup + reg * K + i) % R for i in range(K)]
        return (order, (C.c_void_p * K)(*[d_tok[j] for j in order]), (C.c_void_p * K)(*[d_off] * K), (C.c_void_p * K)(*[d_out[j] for j in order]),
                (C.c_uint32 * K)(*[B] * K))

    regions = [region_args(reg) for reg in range(max(1, args.regions))]
    for _ in range(2):   # warm the multi-batch path (scratch allocations, occupancy queries)
        _o, TOK, OFF, OUT, NS = regions[0]
        h.call("smgx_select_many_tokens_device", model, min(K, 32 * n_lanes), TOK, OFF, NS, T, OUT)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    region_ms, region_ms_ungated, gpu_launches = [], [], 0
    hold_us = int(100 + 2 * K)   # long enough for the host to enqueue the whole region behind the hold kernel
    for gated in (True, False):
      for order, TOK, OFF, OUT, NS in (regions if gated else regions[:1]):
        barrier()
        launches0 = pol.kernel_launches()
        ms = C.c_float()
        one_lane = False   # K steps are spread over all lanes: time across the lanes
        if gated and one_lane and os.environ.get("BENCH_WARM_BACK_TO_BACK", "0") == "1":
            # experiment: an untimed region of the same size runs immediately before the timed one (no idle gap on the GPU)
            _o2, TOK2, OFF2, OUT2, NS2 = regions[(regions.index((order, TOK, OFF, OUT, NS)) + 1) % len(regions)]
            h.call("smgx_stream_hold", 0, 2 * hold_us)
            h.call("smgx_select_many_tokens_device", model, K, TOK2, OFF2, NS2, T, OUT2)
            h.call("smgx_timer_start", 0)
        elif gated:
            h.call("smgx_timer_start_gated", 0, hold_us) if one_lane else h.call("smgx_timer_start_all_gated", hold_us)
        else:
            h.call("smgx_timer_start", 0) if one_lane else h.call("smgx_timer_start_all")
        if n_lanes == 1:
            for j in range(K):
                h.call("smgx_select_batch_tokens_device", model, 0, TOK[j], d_off, B, T, OUT[j], None)
        else:
            h.call("smgx_select_many_tokens_device", model, K, TOK, OFF, NS, T, OUT)
        h.call("smgx_timer_stop_ms", 0, C.byref(ms)) if one_lane else h.call("smgx_timer_stop_all_ms", C.byref(ms))
        (region_ms if gated else region_ms_ungated).append(float(ms.value))
        gpu_launches = pol.kernel_launches() - launches0   # the hold kernel is not counted: it is not part of the path
        last_slot = order[-1]
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        picks = np.zeros(B, np.int32)
        h.call("smgx_memcpy_d2h", picks.ctypes.data_as(C.c_void_p), d_out[last_slot], B * 4)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "picks.npy"), picks.astype(np.float64))
    ms_med = float(np.median(region_ms))
    t_dev = max_over_ranks(ms_med / 1e3)
    value = world * args.steps * B / t_dev

    # ---- parity at full scale: every batch of the last timed region against the oracle (same index, same fleet) ----
    parity = None
    if not args.no_cpu_baseline:
        o_hashes = oracle_hashes(seqs, bs)
        if not np.array_equal(o_hashes, hashes):
            print("PARITY FAILURE: GPU content hashes of the population differ from the oracle's", file=sys.stderr)
            sys.exit(3)
        op, _oix = populate_oracle(seqs, o_hashes, W, bs, 64)
        op.set_state(loads, [1] * W, [1] * W)
        order = regions[-1][0]
        checked, bad = 0, 0
        got = np.zeros(B, np.int32)
        off64 = offsets.astype(np.uint64)
        def check(dptr, j, what):
            h.call("smgx_memcpy_d2h", got.ctypes.data_as(C.c_void_p), dptr, B * 4)
            want = np.asarray(op.select_batch_tokens(host_batches[j], off64)[0])
            for r_ in np.nonzero(got != want)[0][:8]:
                print(f"PARITY: {what} ring batch {j} request {r_}: got {got[r_]} want {want[r_]}", file=sys.stderr)
            return int((got != want).sum())
        for j in sorted(set(order))[: (R if rank == 0 else 4)]:
            bad += check(d_out[j], j, f"{args.steps}-step timed region"); checked += B
        # branches + overlap scores of one batch through the info-carrying call
        info = (_lib.DecisionInfo * B)()
        d_info = L.smgx_device_alloc(h.p, C.sizeof(info), C.byref(err))
        h.call("smgx_select_batch_tokens_device", model, 0, d_tok[order[-1]], d_off, B, T, d_out[order[-1]], d_info)
        h.call("smgx_synchronize")
        h.call("smgx_memcpy_d2h", C.cast(info, C.c_void_p), d_info, C.sizeof(info))
        w_idx, w_br, w_ma, _ = op.select_batch_tokens(host_batches[order[-1]], off64)
        g_br = np.frombuffer(info, dtype=np.uint8).reshape(B, C.sizeof(_lib.DecisionInfo))[:, 8]
        g_ma = np.frombuffer(info, dtype=np.uint32).reshape(B, C.sizeof(_lib.DecisionInfo) // 4)[:, 0]
        bad_info = int((g_br != np.asarray(w_br)).sum() + (g_ma.astype(np.uint64) * bs != np.asarray(w_ma).astype(np.uint64)).sum())   # oracle reports the overlap in tokens
        parity = {"decisions": checked, "mismatches": bad, "branch_or_score_mismatches": bad_info,
                  "what": f"picks of {checked // B} timed batches (last region) + branches/overlap scores of one batch vs the oracle on the same "
                          f"{int(ix.entry_count())}-entry index"}
        bad_total = max_over_ranks(float(bad + bad_info))
        if bad_total:
            print(f"PARITY FAILURE: {bad} pick mismatches, {bad_info} branch/score mismatches vs the oracle", file=sys.stderr)
            sys.exit(3)
        del op, _oix
    else:
        out = np.zeros(B, np.int32)
        h.call("smgx_memcpy_d2h", out.ctypes.data_as(C.c_void_p), d_out[regions[-1][0][-1]], B * 4)
        assert out.min() >= 0 and out.max() < W

    # ---- end to end: public C-ABI call with pinned HOST buffers, H2D + D2H inside the timed region ----
    depth = L.smgx_pipeline_depth(h.p)
    nh = min(len(host_batches), 8)
    pin_tok, pin_out = [], []
    for r in range(nh):
        p = L.smgx_alloc_pinned(host_batches[r].nbytes)
        C.memmove(p, host_batches[r].ctypes.data, host_batches[r].nbytes)
        pin_tok.append(p)
    for r in range(depth):
        pin_out.append(L.smgx_alloc_pinned(B * 4))
    pin_off = L.smgx_alloc_pinned(offsets.nbytes)
    C.memmove(pin_off, offsets.ctypes.data, offsets.nbytes)
    tickets = [None] * depth

    def e2e_run(n_steps):
        for i in range(n_steps):
            slot = i % depth
            if tickets[slot] is not None:
                h.call("smgx_wait", tickets[slot])
            t = C.c_uint64()
            h.call("smgx_submit_tokens", model, pin_tok[i % nh], pin_off, B, pin_out[slot], None, C.byref(t))
            tickets[slot] = t.value
        for s in range(depth):
            if tickets[s] is not None:
                h.call("smgx_wait", tickets[s])
                tickets[s] = None

    e2e_run(max(args.warmup, depth))
    e2e_s = []
    for _ in range(max(1, args.regions)):
        barrier()
        t1 = time.perf_counter()
        e2e_run(args.steps)
        h.call("smgx_synchronize")
        e2e_s.append(time.perf_counter() - t1)
    t_e2e = max_over_ranks(float(np.median(e2e_s)))
    e2e_value = world * args.steps * B / t_e2e
    # per-decision latency = completion time of the batch the request rode in (depth-1 submission, no queueing);
    # kernel part = the same batch device-resident (submit → sync), the rest is the H2D of the tokens + D2H of the picks
    lat, lat_k = [], []
    for i in range(min(max(args.steps, 50), 200)):
        a = time.perf_counter()
        t = C.c_uint64()
        h.call("smgx_submit_tokens", model, pin_tok[i % nh], pin_off, B, pin_out[0], None, C.byref(t))
        h.call("smgx_wait", t.value)
        lat.append(time.perf_counter() - a)
    for i in range(min(max(args.steps, 50), 200)):
        a = time.perf_counter()
        h.call("smgx_select_batch_tokens_device", model, 0, d_tok[i % R], d_off, B, T, d_out[i % R], None)
        h.call("smgx_synchronize")
        lat_k.append(time.perf_counter() - a)
    p99_us, p50_us = float(np.percentile(lat, 99) * 1e6), float(np.percentile(lat, 50) * 1e6)
    k99_us, k50_us = float(np.percentile(lat_k, 99) * 1e6), float(np.percentile(lat_k, 50) * 1e6)

    peak, peak_src = measured_peak()
    path = os.environ.get("SMGX_EVENT_PATH", "split")   # the library's default: the pair (hash stream + balanced search)
    fused = path == "fused"
    kernels_per_launch = 2 if path == "split" else 1
    n_launch_groups = max(gpu_launches // kernels_per_launch, 1)
    achieved = alg_bytes * B * args.steps / (ms_med / 1e3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(args), "batch": B, "tokens": T, "workers": W, "block_size": bs, "jump_size": 64,
                   "index_entries": int(ix.entry_count()), "mode": "event_driven", "parallelism": f"replicas x{world} (no data-path collective)",
                   "l2_hygiene": f"ring of {R} distinct device-resident batches = {R * B * T * 4 / 2**20:.0f} MiB of tokens > L2, each timed region starts "
                                 f"at a different ring position; index ({ix.entry_count() * 32 / 2**20:.0f} MiB live slots) is the L2-resident working set",
                   "index_build_s": round(t_pop, 2), "numa_node": numa_node,
                   "timing": f"{len(region_ms)} back-to-back regions of exactly {K} steps each, CUDA events across the launching lanes, every region enqueued behind a "
                             f"{hold_us} us hold kernel so that the events bracket GPU execution only (region_ms); the same region with the start event recorded "
                             f"on an idle stream, i.e. including the host's launch latency, is region_ms_ungated; the median gated region is reported, max over ranks",
                   "issue": (f"K steps handed to smgx_select_many_tokens_device in one call: up to 32 batches per launch, launches alternate over "
                             f"{n_lanes} CUDA stream lanes") if n_lanes > 1 else "K launches, one batch each, on one stream"},
        "region_ms": region_ms, "region_ms_ungated": region_ms_ungated,
        "e2e": {"value": e2e_value, "unit": "decisions/s", "h2d_bytes_per_step": int(B * T * 4 + (B + 1) * 4), "d2h_bytes_per_step": int(B * 4),
                "pipeline_depth": int(depth), "regions_s": e2e_s,
                "timing": "host wall clock around K pipelined submit/wait calls (median of the regions), device synchronised on both sides"},
        "p50_decision_latency_us": p50_us, "p99_decision_latency_us": p99_us,
        "latency": {"batch": B, "host_buffers_p50_us": p50_us, "host_buffers_p99_us": p99_us, "device_resident_p50_us": k50_us, "device_resident_p99_us": k99_us,
                    "copies_p50_us": p50_us - k50_us,
                    "what": "one 4096-request batch, submit → wait; device_resident = kernel + launch + sync, copies = H2D of 8.4 MB tokens + D2H of 16 KB picks"},
        "gpu_launches": int(gpu_launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": (ncu_traffic() * B * args.steps / n_launch_groups) if ncu_traffic() else None,
                     "traffic_source": "per launch (pair) = DRAM bytes per decision of profiles/roofline_traffic.json (ncu --set full, dram__bytes_read + dram__bytes_write of the "
                                       "hash + search pair on one 20-batch call, cold L2: 2750 B/decision vs 2192 B algorithmic) x the decisions of one launch of this run; a "
                                       "committed capture, not measured in this run",
                     "kernel": ("event_fused_kernel<W1,16> (hash → jump search → argmax in one persistent kernel)" if fused else
                                "event_hs_kernel<16,2> (one launch: hash stream; the last CTA of every 256-request group runs search + argmax)" if path == "hs" else
                                "event_stream_kernel (one launch of persistent CTAs: bulk-copy token ring → XXH3 → jump search → argmax)" if path != "split" else
                                "hash_blocks_kernel<16> + event_search2_kernel (programmatic dependent launch; whole step: both kernels' time, the path's algorithmic bytes)"),
                     "batches_per_launch": args.steps / n_launch_groups,
                     "algorithmic_bytes_per_decision": alg_bytes, "mean_reference_probes": mean_pr,
                     "avg_launch_us": ms_med * 1e3 / n_launch_groups, "peak_source": peak_src},
        "clocks": clocks,
    }
    if parity is not None:
        line["parity_checked"] = parity
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(seqs, hashes, args, bs)
    # free the event leg's device memory before the secondary legs build their own policies
    for dptr in d_tok + d_out + [d_off]:
        L.smgx_device_free(h.p, dptr)
    if rank == 0 and world == 1 and not args.no_text_in:
        try:
            line["text_in"] = text_in_leg(args, local_rank)
        except Exception as e:  # noqa: BLE001
            line["text_in"] = {"error": str(e)[:300]}
    if rank == 0 and world == 1 and not args.no_per_request:
        line["per_request"] = per_request_leg(local_rank)
    if world > 1 and not args.no_sharded:
        try:
            sh = sharded_leg(args, rank, world, local_rank, dist)
        except Exception as e:  # noqa: BLE001
            sh = {"error": str(e)[:300]}
        if rank == 0:
            line["sharded"] = sh
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def per_request_leg(local_rank):
    """The reference's real call shape: LoadBalancingPolicy::select_worker is called once per request from many router tasks
    (policies/mod.rs:43-86, routers/grpc/common/stages/worker_selection.rs:157).  tests/cpp/test_batcher drives include/smgx_batcher.hpp —
    callers enqueue single requests, a group-commit dispatcher hands small batches to the zero-copy smgx_submit_tokens_mapped call, callers
    spin on the completion word — against a 640 k-entry index, and checks every pick against the oracle (checker only).  Two caller shapes:
    32 blocking callers (one request outstanding each: the latency-bound shape) and a 16-thread task pool with 512 requests outstanding."""
    exe = os.path.join(ROOT, "tests", "cpp", "test_batcher")
    if not os.path.exists(exe):
        return {"unavailable": "tests/cpp/test_batcher not built"}
    out = {}
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))
    for name, argv in (("blocking_32_callers", ["32", "4000", "1", "50", "1", "3", "0", "1500"]), ("task_pool_16x512", ["16", "16384", "512", "100", "1", "3", "0", "1500"])):
        try:
            r = subprocess.run([exe] + argv, capture_output=True, text=True, timeout=240, env=env)
            d = json.loads(r.stdout.strip().splitlines()[-1])
            out[name] = {k: d[k] for k in ("transport", "threads", "outstanding_per_thread", "requests", "decisions_per_s", "mean_batch", "p50_latency_us",
                                           "p99_latency_us", "p999_latency_us", "mismatches_vs_oracle")}
        except Exception as e:  # noqa: BLE001
            out[name] = {"error": str(e)[:200]}
    out["what"] = "per-request decisions through smgx::Batcher (include/smgx_batcher.hpp), every pick compared with the oracle; latency = enqueue → pick in the caller's hands"
    return out


def sharded_leg(args, rank, world, local_rank, dist):
    """BASELINE config 4: the fleet (512 workers per GPU) is sharded by worker id; every rank runs the candidate kernel on the FULL request
    batch against its own shard's index, pushes its 24 B/request candidates into every rank's gather buffer over NVLink (peer memory) and
    merges.  Strong-scaling of the FLEET, not of the requests: value = B · K / time, identical on every rank."""
    import torch
    from smg_b200 import CacheAwareConfig, _lib, synth
    from smg_b200.sharding import ShardedEventRouter
    Wg = 512 * world
    B, T, bs = args.batch, args.tokens, 16
    urls = synth.worker_urls(Wg)
    router = ShardedEventRouter(urls, rank, world, CacheAwareConfig(eviction_interval_secs=0, **CFG), jump_size=64, device_id=local_rank,
                                max_batch=B, max_tokens_per_request=T)
    n_seq = args.sequences
    seqs = synth.gen_sequences(n_seq, T, 44)
    flat = np.ascontiguousarray(seqs.reshape(-1))
    P = T // bs
    hashes = np.zeros(n_seq * P, np.uint64)
    got = C.c_uint32()
    hh = router.policy._h
    for off in range(0, flat.size, 4096 * T):
        part = flat[off:off + 4096 * T]
        hh.call("smgx_content_hashes", part.ctypes.data_as(C.c_void_p), part.size, bs, hashes[off // bs:].ctypes.data_as(C.c_void_p), part.size // bs, C.byref(got))
    ids = np.arange(1, n_seq * P + 1, dtype=np.uint64)
    for s in range(n_seq):
        g = s % Wg
        if router.owns(g):
            hh.call("smgx_indexer_apply_stored", router.indexer.model, router.local_id(g), ids[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p),
                    hashes[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p), P, None)
    loads = synth.poisson_loads(Wg, 8, 44)
    router.set_fleet_state(loads, np.ones(Wg, np.uint8))
    L = _lib.load()
    err = _lib.new_err()
    R = 8
    batches = [np.ascontiguousarray(gen_batch(seqs, B, 4400 + r, bs)[0].reshape(-1)) for r in range(R)]   # same stream on every rank (replicated requests)
    offsets = (np.arange(B + 1, dtype=np.uint64) * T).astype(np.uint32)
    d_off = L.smgx_device_alloc(hh.p, offsets.nbytes, C.byref(err))
    hh.call("smgx_memcpy_h2d", d_off, offsets.ctypes.data_as(C.c_void_p), offsets.nbytes)
    d_tok, d_out = [], []
    for r in range(R):
        dt = L.smgx_device_alloc(hh.p, batches[r].nbytes, C.byref(err))
        hh.call("smgx_memcpy_h2d", dt, batches[r].ctypes.data_as(C.c_void_p), batches[r].nbytes)
        d_tok.append(dt); d_out.append(L.smgx_device_alloc(hh.p, B * 4, C.byref(err)))

    def ag(arr):
        t = torch.from_numpy(arr.copy()).cuda()
        out = torch.empty(world * t.numel(), dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(out, t)
        return out.cpu().numpy()
    router.connect_peers(ag)
    for i in range(max(args.warmup, 4)):
        router.select_fused_device(d_tok[i % R], d_off, B, T, d_out[i % R])
    hh.call("smgx_synchronize"); torch.cuda.synchronize(); dist.barrier()
    K = args.steps
    times = []
    for _ in range(max(1, args.regions)):
        hh.call("smgx_synchronize"); dist.barrier()
        ms = C.c_float()
        hh.call("smgx_timer_start", 0)
        for i in range(K):
            router.select_fused_device(d_tok[i % R], d_off, B, T, d_out[i % R])
        hh.call("smgx_timer_stop_ms", 0, C.byref(ms))
        times.append(float(ms.value))
    hh.call("smgx_synchronize")
    t = torch.tensor([float(np.median(times)) / 1e3], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_s = float(t.item())
    picks = np.zeros(B, np.int32)
    last = (K - 1) % R
    hh.call("smgx_memcpy_d2h", picks.ctypes.data_as(C.c_void_p), d_out[last], B * 4)
    # every rank must hold the same picks; rank 0 checks them against the oracle run on the WHOLE fleet
    tp = torch.from_numpy(picks.copy()).cuda()
    allp = torch.empty(world * B, dtype=torch.int32, device="cuda")
    dist.all_gather_into_tensor(allp, tp)
    same = bool((allp.view(world, B) == tp.view(1, B)).all().item())
    res = None
    if rank == 0:
        from oracle import orc
        op = orc.CacheAwarePolicy(eviction_interval_secs=0, **CFG)
        op.set_workers(urls)
        oix = orc.PositionalIndexer(64)
        for u in urls:
            oix.intern_worker(u)
        OL = orc.lib()
        o_hashes = oracle_hashes(seqs, bs)
        for s in range(n_seq):
            OL.orc_indexer_apply_stored(oix.h, s % Wg, ids[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p), o_hashes[s * P:(s + 1) * P].ctypes.data_as(C.c_void_p), P, 0, 0)
        op.attach_indexer("unknown", oix)
        op.set_kv_event_monitor(True)
        op.set_state(loads, [1] * Wg, [1] * Wg)
        want = op.select_batch_tokens(batches[last], offsets.astype(np.uint64))[0]
        bad = int((want != picks).sum())
        res = {"workload": f"config4: {world}xB200, {Wg} workers sharded by worker id (512 per GPU), {n_seq * P}-entry index spread over the shards, "
                           f"batch={B} replicated to every rank, {T}-token requests",
               "value": K * B / t_s, "unit": "decisions/s", "ms_per_step": 1e3 * t_s / K, "steps": K, "region_ms": times,
               "comm": "peer-memory (CUDA IPC mappings over NVLink: 24 B/request/shard stored into every rank's gather buffer + release flags; no host sync, no NCCL on the data path)",
               "exchange_bytes_per_step_per_rank": int(24 * B * (world - 1)),
               "parity_checked": {"decisions": B, "mismatches": bad, "ranks_agree": same, "what": "last timed batch vs the oracle on the whole 512·N-worker fleet"}}
        if bad or not same:
            print(f"PARITY FAILURE (sharded): {bad} mismatches, ranks_agree={same}", file=sys.stderr)
            res["error"] = "parity failure"
    for dptr in d_tok + d_out + [d_off]:
        L.smgx_device_free(hh.p, dptr)
    return res


def text_corpus_docs(n_docs, target_bytes, seed):
    """Synthetic chat-like documents of ~target_bytes UTF-8 bytes built from source-code and prose lines available offline."""
    import glob
    rng = np.random.Generator(np.random.PCG64(seed))
    lines = []
    for f in sorted(glob.glob("/usr/lib/python3*/[a-z]*.py"))[:200]:
        try:
            lines += [ln for ln in open(f, encoding="utf-8", errors="ignore").read().split("\n") if 8 < len(ln) < 200]
        except OSError:
            pass
    if len(lines) < 1000:
        lines = ["the quick brown fox jumps over the lazy dog number %d" % i for i in range(5000)]
    docs = []
    for _ in range(n_docs):
        parts, size = ["<|im_start|>system\nYou are a helpful assistant.<|im_end|>\n<|im_start|>user\n"], 80
        while size < target_bytes:
            ln = lines[int(rng.integers(0, len(lines)))]
            parts.append(ln + "\n")
            size += len(ln.encode()) + 1
        docs.append("".join(parts) + "<|im_end|>\n<|im_start|>assistant\n")
    return docs, lines


def text_in_leg(args, local_rank):
    """The whole hot path from TEXT: tokenize (GPU BPE) → event-driven pick, through smgx_select_batch_text with host
    buffers.  Its own policy/index: N documents of ~2 KB, worker = i mod W, same 80/10/10 query mix."""
    import json as _json
    from smg_b200 import BasicWorker, CacheAwareConfig, CacheAwarePolicy, synth
    gold = os.path.join(ROOT, "tests", "golden")
    specials = _json.load(open(os.path.join(gold, "bpe_vectors.json")))["specials"]
    B, W, bs = args.batch, args.workers, 16
    pol = CacheAwarePolicy(CacheAwareConfig(eviction_interval_secs=0, **CFG), device_id=local_rank, max_batch=B, max_tokens_per_request=8192)
    tok = pol.load_tiktoken_tokenizer(os.path.join(gold, "synth_vocab.tiktoken"), specials)
    ws = [BasicWorker(u) for u in synth.worker_urls(W)]
    for w, l in zip(ws, synth.poisson_loads(W, 8, 42)):
        w.set_load(int(l))
    pol.init_workers(ws)
    mon = pol.kv_event_monitor(bs)
    ix = mon.create_indexer("unknown", 64)
    pol.set_kv_event_monitor(mon)
    n_docs = args.text_docs
    docs, lines = text_corpus_docs(n_docs, args.text_bytes, 42)
    for u in synth.worker_urls(W):
        ix.intern_worker(u)
    seq = 1
    n_tok_total = 0
    for s0 in range(0, n_docs, 2048):
        ids = tok.encode_batch(docs[s0:s0 + 2048])
        for k, t in enumerate(ids):
            nb = len(t) // bs
            n_tok_total += len(t)
            if nb:
                ix.apply_stored_tokens((s0 + k) % W, np.arange(seq, seq + nb, dtype=np.uint64), np.asarray(t[: nb * bs], np.uint32), bs)
                seq += nb
    rng = np.random.Generator(np.random.PCG64(777))
    batches = []
    for _ in range(4):
        texts = []
        for _i in range(B):
            u = rng.random()
            d = docs[int(rng.integers(0, n_docs))]
            if u < 0.8:
                texts.append(d)
            elif u < 0.9:
                cut = int(rng.integers(100, max(101, len(d) - 100)))
                texts.append(d[:cut] + " ".join(lines[int(rng.integers(0, len(lines)))] for _ in range(8)))
            else:
                texts.append("".join(lines[int(rng.integers(0, len(lines)))] + "\n" for _ in range(max(1, args.text_bytes // 60))))
        blob = [t.encode() for t in texts]
        offs = np.zeros(B + 1, np.uint32); np.cumsum([len(x) for x in blob], out=offs[1:])
        batches.append((texts, np.frombuffer(b"".join(blob), dtype=np.uint8).copy(), offs))
    h, L = pol._h, __import__("smg_b200")._lib.load()
    model = pol._push_fleet(ws)
    pins = []
    for texts, data, offs in batches:
        pd = L.smgx_alloc_pinned(data.nbytes); C.memmove(pd, data.ctypes.data, data.nbytes)
        po = L.smgx_alloc_pinned(offs.nbytes); C.memmove(po, offs.ctypes.data, offs.nbytes)
        pins.append((pd, po, int(offs[-1])))
    out = L.smgx_alloc_pinned(B * 4)
    cap = max(p[2] for p in pins) + 16
    otok = L.smgx_alloc_pinned(cap * 4)
    otoff = L.smgx_alloc_pinned((B + 1) * 4)

    def run(k, with_tokens):
        t0 = time.perf_counter()
        for i in range(k):
            pd, po, _ = pins[i % len(pins)]
            h.call("smgx_select_batch_text", model, pd, po, B, out, None, otok if with_tokens else None, otoff if with_tokens else None, cap)
        return time.perf_counter() - t0

    depth = L.smgx_pipeline_depth(h.p)
    outs = [L.smgx_alloc_pinned(B * 4) for _ in range(depth)]

    def run_pipelined(k):   # smgx_submit_text / smgx_wait over the library's stream lanes, like the tokens-in e2e leg
        tickets = [None] * depth
        t0 = time.perf_counter()
        for i in range(k):
            slot = i % depth
            if tickets[slot] is not None:
                h.call("smgx_wait", tickets[slot])
            pd, po, _ = pins[i % len(pins)]
            t = C.c_uint64()
            h.call("smgx_submit_text", model, pd, po, B, outs[slot], None, C.byref(t))
            tickets[slot] = t.value
        for s_ in range(depth):
            if tickets[s_] is not None:
                h.call("smgx_wait", tickets[s_])
        return time.perf_counter() - t0

    run(2 * len(pins), True)
    run(len(pins), False)
    run_pipelined(2 * depth)
    k = max(10, min(args.steps, 40))
    t_picks = run(k, False)
    t_full = run(k, True)
    t_pipe = run_pipelined(k)
    mean_bytes = float(np.mean([p[2] for p in pins])) / B
    res = {"unit": "decisions/s", "pipelined": {"value": k * B / t_pipe, "call": f"smgx_submit_text / smgx_wait, {depth} batches in flight"},
           "picks_only": {"value": k * B / t_picks}, "picks_and_tokens_to_host": {"value": k * B / t_full},
           "steps": k, "mean_text_bytes_per_request": mean_bytes, "mean_tokens_per_request": n_tok_total / n_docs,
           "bytes_per_token": args.text_bytes / max(1.0, n_tok_total / n_docs), "index_docs": n_docs, "index_entries": int(ix.entry_count()),
           "h2d_bytes_per_step": int(np.mean([p[2] for p in pins])) + (B + 1) * 4,
           "call": "smgx_select_batch_text (GPU BPE tokenize → hash → search → pick), one synchronous call per step, pinned host buffers"}
    try:
        import tiktoken
        from oracle import bpe_ref
        ranks = bpe_ref.load_tiktoken_bpe(os.path.join(gold, "synth_vocab.tiktoken"))
        enc = tiktoken.Encoding("synth", pat_str=bpe_ref.CL100K_BASE_PATTERN, mergeable_ranks=ranks, special_tokens=specials)
        nthreads = os.cpu_count() or 1
        texts = batches[0][0]
        enc.encode_batch(texts[:256], num_threads=nthreads, allowed_special="all")
        t0 = time.perf_counter()
        ids = enc.encode_batch(texts, num_threads=nthreads, allowed_special="all")
        dt = time.perf_counter() - t0
        res["cpu_tokenize_baseline"] = {"value": B / dt, "unit": "requests/s", "tokens_per_s": sum(len(x) for x in ids) / dt, "cores": nthreads,
                                        "kind": "tiktoken 0.12 (OpenAI Rust CoreBPE, the algorithm tiktoken-rs ports) encode_batch, tokenize step only"}
    except Exception as e:  # noqa: BLE001
        res["cpu_tokenize_baseline"] = {"unavailable": str(e)[:100]}
    return res


def cpu_baseline(seqs, hashes, args, bs):
    """The oracle (C++ restatement of the reference algorithm) on ONE host core, sequential reference semantics,
    bounded sample of the same workload."""
    from smg_b200 import synth
    B, T, W = args.batch, args.tokens, args.workers
    op, _ = populate_oracle(seqs, hashes, W, bs, 64)
    op.set_state(synth.poisson_loads(W, 8, 42), [1] * W, [1] * W)
    tk, off = synth.ragged(gen_batch(seqs, B, 42, bs)[0])
    off = off.astype(np.uint64)
    op.select_batch_tokens(tk, off)            # warm
    t, n = 0.0, 0
    while t < 8.0 and n < 400:
        t += op.select_batch_tokens(tk, off)[3]
        n += 1
    return {"value": n * B / t, "unit": "decisions/s", "cores": 1, "kind": "port",
            "sample": f"{n} passes over one batch of {B} requests (same index, same mix), single thread, {t:.1f} s of CPU work"}


if __name__ == "__main__":
    main()
