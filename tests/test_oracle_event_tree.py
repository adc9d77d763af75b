"""Oracle pinned against the reference's own event_tree.rs unit tests (ported in scenarios_event_tree.py)
and XXH3 known answers.  CPU only."""
import json
import os
import struct

import pytest

from oracle import orc
from tests import random_vectors as RV
from tests import scenarios_event_tree as S

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("scenario", S.SCENARIOS, ids=lambda f: f.__name__)
def test_event_tree_scenarios(scenario):
    scenario(lambda jump: orc.PositionalIndexer(jump), orc)


def test_zero_jump_size_panics():  # event_tree.rs:1484
    with pytest.raises(ValueError, match="jump_size must be greater than 0"):
        orc.PositionalIndexer(0)


def test_request_content_hash_chunking():  # event_tree.rs:1062, :1520-1568
    h = orc.compute_request_content_hashes(list(range(1, 9)), 4)
    assert h == [orc.compute_content_hash([1, 2, 3, 4]), orc.compute_content_hash([5, 6, 7, 8])]
    assert orc.compute_request_content_hashes([1, 2, 3], 0) == []
    assert len(orc.compute_request_content_hashes(list(range(1, 11)), 4)) == 2
    assert orc.compute_request_content_hashes([1, 2, 3], 4) == []
    assert orc.compute_request_content_hashes([], 16) == []
    assert len(orc.compute_request_content_hashes(list(range(1, 7)), 2)) == 3
    h1 = orc.compute_request_content_hashes([10, 20, 30], 1)
    assert h1 == [orc.compute_content_hash([t]) for t in (10, 20, 30)]
    assert orc.compute_content_hash([]) == orc.compute_content_hash([])
    assert orc.compute_content_hash([42]) != orc.compute_content_hash([43])


def test_xxh3_known_answer_from_survey():
    # SURVEY.md §8c: xxh3_64(LE32[1,2,3,4], seed=1337) generated with Python xxhash 3.7.0
    assert orc.compute_content_hash([1, 2, 3, 4]) == 14643705804678351452


def test_xxh3_golden_vectors():
    """tests/golden/xxh3_vectors.json was produced by tests/golden/gen_golden.py with the independent Python
    `xxhash` package (XXH3 is a frozen public spec; the reference holds no literal digests, SURVEY §8c)."""
    vec = json.load(open(os.path.join(GOLD, "xxh3_vectors.json")))
    assert len(vec["cases"]) > 300
    for c in vec["cases"]:
        data = bytes.fromhex(c["hex"])
        assert orc.xxh3_64(data, c["seed"]) == int(c["digest"]), (len(data), c["seed"])


def xxh3_random_inputs():
    """Seeded random byte strings of every length 0..299 and a few long ones, then 16 token ids."""
    import random
    rng = random.Random(7)
    data = [bytes(rng.getrandbits(8) for _ in range(n)) for n in list(range(0, 300)) + [1023, 1024, 1025, 4096, 10000]]
    toks = [rng.getrandbits(32) for _ in range(16)]
    return data, toks


def test_xxh3_against_live_xxhash_if_present():
    """Against the digests Python `xxhash` gave for these inputs (tests/golden/random_vectors.json, written by
    tests/golden/gen_random_vectors.py), and against the live package when it is importable."""
    data, toks = xxh3_random_inputs()
    want = RV.load("xxh3_seed1337")
    assert [orc.xxh3_64(d, 1337) for d in data] == [int(x) for x in want["digests"]]
    assert orc.compute_content_hash(toks) == int(want["content_hash"])
    try:
        import xxhash
    except ImportError:
        return
    for d in data:
        assert orc.xxh3_64(d, 1337) == xxhash.xxh3_64_intdigest(d, seed=1337)
    assert orc.compute_content_hash(toks) == xxhash.xxh3_64_intdigest(struct.pack("<16I", *toks), seed=1337)


def test_apply_kv_events_reference_cases():
    """orc.apply_kv_events restates KvEventMonitor::apply_event; pinned by the reference's tests (kv_event_monitor.rs:629-760)."""
    def blk(h, toks):
        return {"block_hash": h, "token_ids": toks, "block_size": len(toks)}
    ix = orc.PositionalIndexer(64)
    w = ix.intern_worker("http://w1:8000")
    assert orc.apply_kv_events(ix, w, [{"stored": {"blocks": [blk(1, [10, 20, 30, 40]), blk(2, [50, 60, 70, 80])], "parent_block_hash": None}}]) == 0
    assert ix.current_size() == 2                                                        # test_apply_stored_no_parent
    ix = orc.PositionalIndexer(64)
    w = ix.intern_worker("http://w1:8000")
    orc.apply_kv_events(ix, w, [{"stored": {"blocks": [blk(1, [10, 20, 30, 40])], "parent_block_hash": None}}])
    assert orc.apply_kv_events(ix, w, [{"stored": {"blocks": [blk(2, [50, 60, 70, 80])], "parent_block_hash": 1}}]) == 0
    assert ix.current_size() == 2                                                        # test_apply_stored_with_parent
    ix = orc.PositionalIndexer(64)
    w = ix.intern_worker("http://new-worker:8000")
    assert orc.apply_kv_events(ix, w, [{"stored": {"blocks": [blk(1, [10, 20, 30, 40])], "parent_block_hash": 999}}]) == 1
    assert ix.current_size() == 1                                                        # test_apply_stored_fallback_on_worker_not_tracked
    orc.apply_kv_events(ix, w, [{"stored": {"blocks": [blk(-1, [1, 2])], "parent_block_hash": 1}}])      # −1 ≡ u64::MAX (:643)
    assert orc.apply_kv_events(ix, w, [{"stored": {"blocks": [blk(5, [3, 4])], "parent_block_hash": 2**64 - 1}}]) == 0
    orc.apply_kv_events(ix, w, [{"removed": {"block_hashes": [5]}}])
    assert ix.current_size() == 2
    orc.apply_kv_events(ix, w, [{"cleared": {}}])
    assert ix.current_size() == 0
