"""Generates tests/golden/random_vectors.json: what the independent Python packages compute on the seeded random inputs of
the tests that compare against them (tests/test_oracle_event_tree.py, tests/test_oracle_bpe.py, tests/test_gpu_tokenizer.py),
so that those comparisons also run where the packages are not installed.  Token ids are stored as digests (tests/random_vectors.py).
  * xxh3_seed1337 — `xxhash` (C reference implementation of the XXH3 spec)
  * tiktoken_oracle_texts, tiktoken_gpu_texts — `tiktoken` (OpenAI's Rust CoreBPE) over tests/golden/synth_vocab.tiktoken
  * hf_llama3_style_texts — `tokenizers` (the HuggingFace Rust crate) over tests/golden/hf_llama3_style_tokenizer.json
Run from the repo root: python tests/golden/gen_random_vectors.py"""
import json
import os
import struct
import sys

import tiktoken
import tokenizers
import xxhash

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import bpe_ref  # noqa: E402
from tests.random_vectors import ids_digest  # noqa: E402
from tests.test_gpu_tokenizer import random_hf_texts, random_tiktoken_texts  # noqa: E402
from tests.test_oracle_bpe import random_texts  # noqa: E402
from tests.test_oracle_event_tree import xxh3_random_inputs  # noqa: E402


def main():
    data, toks = xxh3_random_inputs()
    g = json.load(open(os.path.join(HERE, "bpe_vectors.json")))
    ranks = bpe_ref.load_tiktoken_bpe(os.path.join(HERE, "synth_vocab.tiktoken"))
    enc = tiktoken.Encoding("synth", pat_str=g["pattern"], mergeable_ranks=ranks, special_tokens=g["specials"])
    hf = tokenizers.Tokenizer.from_file(os.path.join(HERE, "hf_llama3_style_tokenizer.json"))
    out = {
        "generators": {"xxhash": xxhash.VERSION, "tiktoken": tiktoken.__version__, "tokenizers": tokenizers.__version__},
        "xxh3_seed1337": {"digests": [str(xxhash.xxh3_64_intdigest(d, seed=1337)) for d in data],
                          "content_hash": str(xxhash.xxh3_64_intdigest(struct.pack("<16I", *toks), seed=1337))},
        "tiktoken_oracle_texts": [ids_digest(enc.encode(t, allowed_special="all")) for t in random_texts()],
        "tiktoken_gpu_texts": [ids_digest(enc.encode(t, allowed_special="all")) for t in random_tiktoken_texts()],
        "hf_llama3_style_texts": [ids_digest(e.ids) for e in hf.encode_batch(random_hf_texts(), add_special_tokens=False)],
    }
    json.dump(out, open(os.path.join(HERE, "random_vectors.json"), "w"), separators=(",", ":"))


if __name__ == "__main__":
    main()
    print("ok")
