"""Shared loader for tests/golden/random_vectors.json (made by tests/golden/gen_random_vectors.py).  Token id lists are stored
as 64-bit BLAKE2b digests of their little-endian u32 bytes, which keeps the file small."""
import hashlib
import json
import os
import struct

PATH = os.path.join(os.path.dirname(__file__), "golden", "random_vectors.json")


def ids_digest(ids):
    return hashlib.blake2b(struct.pack(f"<{len(ids)}I", *ids), digest_size=8).hexdigest()


def load(key):
    return json.load(open(PATH))[key]
