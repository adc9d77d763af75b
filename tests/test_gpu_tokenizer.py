"""GPU parity for K1 (tokenize): the CUDA BPE path through the C ABI against the golden vectors (Python tiktoken), the
oracle restatement, live tiktoken when importable, and the text-in pick (tokenize → cache-aware select in one call)."""
import json
import os
import random

import numpy as np
import pytest

from oracle import bpe_ref, orc
from smg_b200 import synth
from tests import random_vectors as RV

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
VOCAB = os.path.join(GOLD, "synth_vocab.tiktoken")


def _gold():
    return json.load(open(os.path.join(GOLD, "bpe_vectors.json")))


def _policy_and_tok(**cfg):
    from smg_b200 import CacheAwareConfig, CacheAwarePolicy
    g = _gold()
    pol = CacheAwarePolicy(CacheAwareConfig(eviction_interval_secs=0, **cfg))
    return pol, pol.load_tiktoken_tokenizer(VOCAB, g["specials"]), g


def test_golden_vectors_on_gpu():
    pol, tok, g = _policy_and_tok()
    texts = [c["text"] for c in g["cases"]]
    got = tok.encode_batch(texts)
    for c, ids in zip(g["cases"], got):
        assert ids == c["ids"], repr(c["text"][:80])
    assert tok.encode("") == [] and tok.encode("<|endoftext|>") == [g["specials"]["<|endoftext|>"]]


def random_tiktoken_texts():
    rng = random.Random(5)
    alphabet = "abcdefghij XYZ 0123\n\t\r'.,!?-_()<|>im_startend" + "éß你好\U0001f44b 　ſ"
    texts = ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, 300))) for _ in range(600)]
    texts += ["word " * 500, "x" * 3000, " " * 2000 + "end", "\n".join("line %d: the quick brown fox" % i for i in range(200))]
    return texts


def test_random_text_vs_oracle_and_live_tiktoken():
    """Against the oracle, the ids tiktoken gave for these texts (tests/golden/random_vectors.json, written by
    tests/golden/gen_random_vectors.py), and live tiktoken when it is importable."""
    pol, tok, g = _policy_and_tok()
    ranks = bpe_ref.load_tiktoken_bpe(VOCAB)
    enc = bpe_ref.CoreBPE(ranks, g["specials"])
    texts = random_tiktoken_texts()
    got = tok.encode_batch(texts)
    want = RV.load("tiktoken_gpu_texts")
    assert len(want) == len(texts)
    for t, ids, w in zip(texts, got, want):
        assert ids == enc.encode_with_special_tokens(t), repr(t[:80])
        assert RV.ids_digest(ids) == w, repr(t[:80])
    try:
        import tiktoken
    except ImportError:
        return
    live = tiktoken.Encoding("synth", pat_str=g["pattern"], mergeable_ranks=ranks, special_tokens=g["specials"])
    for t, ids in zip(texts, got):
        assert ids == live.encode(t, allowed_special="all"), repr(t[:80])


def test_text_in_pick_equals_tokens_in_pick_and_oracle():
    """tokenize → select on the device in one call == tokenize, then select == oracle policy on oracle tokens."""
    from smg_b200 import BasicWorker
    bs = 4
    cfg = dict(cache_threshold=0.3, balance_abs_threshold=64, balance_rel_threshold=1.5, block_size=bs)
    pol, tok, g = _policy_and_tok(**cfg)
    ranks = bpe_ref.load_tiktoken_bpe(VOCAB)
    enc = bpe_ref.CoreBPE(ranks, g["specials"])
    urls = synth.worker_urls(8)
    ws = [BasicWorker(u) for u in urls]
    pol.init_workers(ws)
    mon = pol.kv_event_monitor(bs)
    ix = mon.create_indexer("unknown", 8)
    pol.set_kv_event_monitor(mon)
    op = orc.CacheAwarePolicy(eviction_interval_secs=0, **cfg)
    op.set_workers(urls)
    oix = orc.PositionalIndexer(8)
    op.attach_indexer("unknown", oix)
    op.set_kv_event_monitor(True)
    rng = random.Random(9)
    lines = [c["text"] for c in g["cases"] if len(c["ids"]) >= 12]
    system = ["<|im_start|>system\n" + rng.choice(lines) + "<|im_end|>\n" for _ in range(6)]
    for u in urls:
        assert ix.intern_worker(u) == oix.intern_worker(u)
    seq = 1
    for k, sp in enumerate(system):                      # workers cache the system prompts (KV events carry token ids)
        ids = enc.encode_with_special_tokens(sp)
        nb = len(ids) // bs
        hs = orc.compute_request_content_hashes(ids, bs)
        blocks = [(seq + i, hs[i]) for i in range(nb)]
        seq += nb
        for w in (k % 8, (k + 3) % 8):
            ix.apply_stored(w, blocks)
            oix.apply_stored(w, blocks)
    loads = [rng.randint(0, 9) for _ in urls]
    for w, l in zip(ws, loads):
        w.set_load(l)
    op.set_state(loads, [1] * 8, [1] * 8)
    texts = [rng.choice(system) + "<|im_start|>user\n" + rng.choice(lines) + "<|im_end|>\n" for _ in range(200)] + [rng.choice(lines) for _ in range(56)]
    idx_text, info, toks = pol.select_worker_batch_text(ws, texts)
    assert toks == [enc.encode_with_special_tokens(t) for t in texts]
    idx_tok, _ = pol.select_worker_batch(ws, toks)
    assert np.array_equal(idx_text, idx_tok)
    flat = np.concatenate([np.asarray(t, np.uint32) for t in toks])
    offs = np.zeros(len(toks) + 1, np.uint64); np.cumsum([len(t) for t in toks], out=offs[1:])
    want, br, _, _ = op.select_batch_tokens(flat, offs)
    assert np.array_equal(idx_text, want)
    assert (np.asarray(br) == 2).sum() > 100      # most requests hit a cached system prompt
    # pipelined form: four sub-batches in flight over the stream lanes give the same picks
    import ctypes as C
    from smg_b200.policy import TiktokenTokenizer
    model = pol._push_fleet(ws)
    parts = [texts[i::4] for i in range(4)]
    bufs, tickets = [], []
    for part in parts:
        data, offsets = TiktokenTokenizer._ragged(part)
        out = np.full(len(part), -7, np.int32)
        t = C.c_uint64()
        pol._h.call("smgx_submit_text", model, data.ctypes.data_as(C.c_void_p), offsets.ctypes.data_as(C.c_void_p), len(part),
                    out.ctypes.data_as(C.c_void_p), None, C.byref(t))
        bufs.append((data, offsets, out)); tickets.append(t.value)
    for t in tickets:
        pol._h.call("smgx_wait", t)
    for i, (_, _, out) in enumerate(bufs):
        assert np.array_equal(out, idx_text[i::4])


# ---- HuggingFace tokenizer.json (byte-level BPE, Llama-3-style pre-tokenizer) -------------------------------------------------
@pytest.mark.parametrize("fixture", ["hf_llama3_style_tokenizer.json", "hf_plain_bpe_tokenizer.json"])
def test_hf_tokenizer_json_matches_tokenizers_crate(fixture):
    """tests/golden/hf_bpe_vectors.json was produced by the Python bindings of the `tokenizers` crate (the engine behind the
    reference's HuggingFaceTokenizer, huggingface.rs:310-316) from the committed tokenizer.json fixtures — one with
    ignore_merges (Llama 3), one without."""
    from smg_b200 import CacheAwareConfig, CacheAwarePolicy
    g = json.load(open(os.path.join(GOLD, "hf_bpe_vectors.json")))
    pol = CacheAwarePolicy(CacheAwareConfig(eviction_interval_secs=0))
    tok = pol.load_hf_tokenizer(os.path.join(GOLD, fixture))
    got = tok.encode_batch(g["texts"])
    for t, ids, want in zip(g["texts"], got, g["ids"][fixture]):
        assert ids == want, repr(t[:80])


def random_hf_texts():
    rng = random.Random(9)
    alphabet = "abcdefghij the quick XYZ 0123456789\n\t\r'.,!?-_(){}[]<|>eot_idbegin_of_text" + "éßüï你好世界\U0001f44b\U0001f30d ١٢٣"
    texts = ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, 400))) for _ in range(400)]
    texts += ["<|begin_of_text|>" + "hello world " * 50 + "<|eot_id|>", "don't DON'T I'LL we'Ve 'S", "   \n\n  \n x  \n", "12345678901234567890"]
    return texts


def test_hf_tokenizer_live_tokenizers_random_texts():
    """Against the ids the `tokenizers` package gave for these texts (tests/golden/random_vectors.json, written by
    tests/golden/gen_random_vectors.py), and against the live package when it is importable."""
    from smg_b200 import CacheAwareConfig, CacheAwarePolicy
    path = os.path.join(GOLD, "hf_llama3_style_tokenizer.json")
    pol = CacheAwarePolicy(CacheAwareConfig(eviction_interval_secs=0))
    tok = pol.load_hf_tokenizer(path)
    texts = random_hf_texts()
    got = tok.encode_batch(texts)
    want = RV.load("hf_llama3_style_texts")
    assert len(want) == len(texts)
    for t, a, b in zip(texts, got, want):
        assert RV.ids_digest(a) == b, repr(t[:80])
    try:
        import tokenizers
    except ImportError:
        return
    ref = tokenizers.Tokenizer.from_file(path)
    want = [e.ids for e in ref.encode_batch(texts, add_special_tokens=False)]
    for t, a, b in zip(texts, got, want):
        assert a == b, repr(t[:80])


def test_hf_loader_refuses_unsupported_tokenizer_json(tmp_path):
    from smg_b200 import CacheAwareConfig, CacheAwarePolicy
    j = json.load(open(os.path.join(GOLD, "hf_llama3_style_tokenizer.json")))
    j["normalizer"] = {"type": "NFC"}
    p = tmp_path / "tok.json"
    p.write_text(json.dumps(j))
    pol = CacheAwarePolicy(CacheAwareConfig(eviction_interval_secs=0))
    with pytest.raises(ValueError):
        pol.load_hf_tokenizer(str(p))


def test_piece_length_classes_vs_oracle():
    """Pieces of every length class take a different merge kernel (≤ 15 bytes: shared-memory columns; 16-32: one symbol per lane;
    33-256: linked list in shared memory; longer: in place in the global scratch) — all must agree with the oracle."""
    pol, tok, g = _policy_and_tok()
    ranks = bpe_ref.load_tiktoken_bpe(VOCAB)
    enc = bpe_ref.CoreBPE(ranks, g["specials"])
    rng = random.Random(17)
    texts = []
    for k in list(range(1, 70)) + [100, 127, 128, 129, 200, 255, 256, 257, 300, 1000]:
        texts += [" " * k + "x", "-" * k, "ab" * k, "".join(rng.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(k)),
                  "".join(rng.choice("éßü你好") for _ in range(k)), "=" * k + "\n" * (k % 5), "a" * k + " " + "b" * k]
    got = tok.encode_batch(texts)
    for t, ids in zip(texts, got):
        assert ids == enc.encode_with_special_tokens(t), (len(t), repr(t[:40]))
