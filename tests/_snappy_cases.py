"""Seeded snappy inputs of the tests that compare with the reference's vendored snappy 1.1.3, and what the reference returned
for them (tests/golden/snappy_ref_results.json, written by tests/golden/gen_snappy_ref_results.py): the tests regenerate the
inputs from their seeds and compare the device's results with the stored ones."""
import hashlib
import json
import os

from _traffic import rnd62

HERE = os.path.dirname(os.path.abspath(__file__))
T62 = b"abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789"


def digest(b):
    return None if b is None else hashlib.sha256(bytes(b)).hexdigest()


def ref_results():
    with open(os.path.join(HERE, "golden", "snappy_ref_results.json")) as f:
        return json.load(f)


def corrupted_blobs(rng, seeds, count=400):
    """truncations, bit flips, appended bytes and overwritten bytes of the streams in `seeds`"""
    out = []
    for _ in range(count):
        b = bytearray(rng.choice(seeds)); c = rng.random()
        if c < 0.3: del b[rng.randrange(len(b)):]
        elif c < 0.7:
            for _k in range(rng.randrange(1, 4)): b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
        elif c < 0.85: b += bytes(rng.randrange(256) for _k in range(rng.randrange(1, 5)))
        else: b[rng.randrange(len(b))] = rng.randrange(256)
        out.append(bytes(b))
    return out


def warp_raws(rng, long):
    text = b" ".join(rng.choice([b"echo", b"brpc", b"socket", b"iobuf", b"x" * 30]) for _ in range(4000))
    if long:
        return [b"", b"a", b"abcd" * 10, rnd62(rng, 100), rnd62(rng, 5000), text, text * 5, b"\x00" * 70000, rnd62(rng, 70000), (rnd62(rng, 37) * 3000)[:100000]]
    return [b"", b"a", b"abcd" * 10, rnd62(rng, 100), rnd62(rng, 3000), text[:20000], b"\x00" * 9000, (rnd62(rng, 37) * 300)[:9000], rnd62(rng, 70000)[:20000]]


def warp_corruption(rng, comp):
    b = bytearray(comp)
    c = rng.random()
    if c < 0.3: del b[rng.randrange(len(b)):]
    elif c < 0.8: b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
    else: b += bytes(rng.getrandbits(8) for _ in range(3))
    return bytes(b)


def warp_corruptions_per_raw(long):
    return 30 if long else 12


LEAF_SIZES = [0, 1, 7, 47, 48, 100, 1027, 4099, 70001, 300000]


def leaf_raw(rng, n):
    raw = bytes(rng.choice(T62) for _ in range(min(n, 5000))) * (n // 5000 + 1)
    return raw[:n]
