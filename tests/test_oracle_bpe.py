"""BPE oracle (oracle/bpe_ref.py) pinned against the golden vectors produced by Python tiktoken (OpenAI's Rust CoreBPE)
and, when importable, against live tiktoken on random text.  CPU only."""
import json
import os
import random

from oracle import bpe_ref
from tests import random_vectors as RV

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _load():
    g = json.load(open(os.path.join(GOLD, "bpe_vectors.json")))
    ranks = bpe_ref.load_tiktoken_bpe(os.path.join(GOLD, "synth_vocab.tiktoken"))
    return g, ranks


def test_pattern_is_the_reference_pattern():
    g, _ = _load()
    assert g["pattern"] == bpe_ref.CL100K_BASE_PATTERN   # crates/tokenizer/src/tiktoken.rs:28


def test_oracle_matches_golden_vectors():
    g, ranks = _load()
    enc = bpe_ref.CoreBPE(ranks, g["specials"])
    assert len(g["cases"]) > 300
    for c in g["cases"]:
        assert enc.encode_with_special_tokens(c["text"]) == c["ids"], c["text"][:80]


def random_texts():
    rng = random.Random(3)
    alphabet = "abcdefghij XYZ 0123\n\t\r'.,!?-_()<|>im_startend" + "éß你好\U0001f44b 　"
    return ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, 160))) for _ in range(400)]


def test_oracle_matches_live_tiktoken_on_random_text():
    """Against the ids tiktoken gave for these texts (tests/golden/random_vectors.json, written by
    tests/golden/gen_random_vectors.py), and against live tiktoken when it is importable."""
    g, ranks = _load()
    enc = bpe_ref.CoreBPE(ranks, g["specials"])
    texts = random_texts()
    want = RV.load("tiktoken_oracle_texts")
    assert len(want) == len(texts)
    for t, ids in zip(texts, want):
        assert RV.ids_digest(enc.encode_with_special_tokens(t)) == ids, repr(t)
    try:
        import tiktoken
    except ImportError:
        return
    live = tiktoken.Encoding("synth", pat_str=g["pattern"], mergeable_ranks=ranks, special_tokens=g["specials"])
    for t in texts:
        assert enc.encode_with_special_tokens(t) == live.encode(t, allowed_special="all"), repr(t)
