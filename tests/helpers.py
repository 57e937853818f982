"""Test-side wiring: loads the checkers (oracle restatement, reference build) and the product."""
import hashlib
import json
import os
import random

from edlib_b200._ffi import EdlibLib, REPO, product_path

ORACLE_SO = os.path.join(REPO, "oracle", "liboracle.so")
REF_SO = os.path.join(REPO, "oracle", "_ref", "libedlib_ref.so")

_cache = {}


def oracle():
    if "oracle" not in _cache:
        _cache["oracle"] = EdlibLib(ORACLE_SO, prefix="oracle")
    return _cache["oracle"]


def have_ref():
    return os.path.exists(REF_SO)


def ref():
    if "ref" not in _cache:
        _cache["ref"] = EdlibLib(REF_SO, prefix="edlib")
    return _cache["ref"]


def product():
    if "product" not in _cache:
        _cache["product"] = EdlibLib(product_path(), prefix="edlib", has_batch=True)
    return _cache["product"]


def digest(value):
    """Short fingerprint of a result dict, a string or None, as stored in tests/golden/ref_digests.json (bytes fields are
    hashed as hex, dict keys in sorted order)."""
    if isinstance(value, dict):
        value = {k: (v.hex() if isinstance(v, bytes) else v) for k, v in value.items()}
    text = json.dumps(value, sort_keys=True, default=int)
    return hashlib.sha256(text.encode()).hexdigest()[:8]


def golden_digests():
    """tests/golden/ref_digests.json: fingerprints of the reference build's answers (tests/golden/make_ref_digests.py)."""
    if "golden" not in _cache:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")) as f:
            _cache["golden"] = json.load(f)
    return _cache["golden"]


def rand_seq(rng, n, alphabet):
    return bytes(rng.choice(alphabet) for _ in range(n))


def mutate(rng, s, rate, alphabet):
    """Substitution / insertion / deletion, one third each, per-base probability `rate`."""
    out = bytearray()
    for ch in s:
        if rng.random() < rate:
            kind = rng.randrange(3)
            if kind == 0:
                out.append(rng.choice(alphabet))
            elif kind == 1:
                out.append(ch)
                out.append(rng.choice(alphabet))
            # kind == 2: deletion
        else:
            out.append(ch)
    return bytes(out)
