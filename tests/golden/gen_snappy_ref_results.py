#!/usr/bin/env python
"""Generate tests/golden/snappy_ref_results.json: what the reference's vendored snappy 1.1.3 and crc32c.cc (compiled unmodified into
oracle/_ref/libref_leaf.so by oracle/Makefile) return for the seeded inputs of tests/_snappy_cases.py, as SHA-256 digests:
  gpu_corruptions  RawUncompress of the 400 corrupted streams of test_gpu_snappy (null = the reference rejects the stream)
  warp.{short,long} RawCompress of test_device_warp_host's inputs, and [GetUncompressedLength, RawUncompress verdict, output]
                   of their corruptions (default and B2_LONG_TESTS=1 sizes)
  leaf             crc32c, MaxCompressedLength and RawCompress of test_gpu_leaf_signatures' inputs
Run where the reference sources are present; the JSON is committed."""
import ctypes as C
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
import _snappy_cases as S  # noqa: E402
from _traffic import SEED  # noqa: E402

ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_leaf.so"))
ref.ref_crc32c_extend.restype = C.c_uint32; ref.ref_crc32c_extend.argtypes = [C.c_uint32, C.c_char_p, C.c_size_t]
ref.ref_snappy_max_compressed_length.restype = C.c_size_t; ref.ref_snappy_max_compressed_length.argtypes = [C.c_size_t]
ref.ref_snappy_compress.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.POINTER(C.c_size_t)]
ref.ref_snappy_uncompress.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
ref.ref_snappy_uncompressed_length.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]


def compress(raw):
    cap = ref.ref_snappy_max_compressed_length(len(raw)); out = C.create_string_buffer(cap); n = C.c_size_t(cap)
    ref.ref_snappy_compress(raw, len(raw), out, C.byref(n))
    return out.raw[:n.value]


def uncompressed_length(b):
    ul = C.c_size_t()
    return ul.value if ref.ref_snappy_uncompressed_length(b, len(b), C.byref(ul)) else None


def uncompress(b, cap):
    out = C.create_string_buffer(max(1, cap)); got = C.c_size_t()
    return out.raw[:got.value] if ref.ref_snappy_uncompress(b, len(b), out, cap, C.byref(got)) else None


def gpu_corruptions():
    vec = json.load(open(os.path.join(HERE, "snappy_vectors.json")))
    seeds = [bytes.fromhex(v["comp_hex"]) for v in vec]
    seeds = [b for b in seeds if 0 < len(b) < 5000]
    res = []
    for b in S.corrupted_blobs(random.Random(SEED), seeds):
        ul = uncompressed_length(b)
        res.append(S.digest(uncompress(b, ul)) if ul is not None and ul <= 32 * len(b) + 64 else None)
    return res


def warp(long):
    rng = random.Random(SEED + 972)
    comp, corrupt = [], []
    for raw in S.warp_raws(rng, long):
        c = compress(raw)
        comp.append(S.digest(c))
        for _ in range(S.warp_corruptions_per_raw(long)):
            if not c:
                break
            b = S.warp_corruption(rng, c)
            ul = uncompressed_length(b)
            if ul is None or ul > 32 * len(b) + 64 or ul > (1 << 20):
                corrupt.append([ul, None, None])
                continue
            out = uncompress(b, ul)
            corrupt.append([ul, out is not None, S.digest(out)])
    return {"compress": comp, "corrupt": corrupt}


def leaf():
    rng = random.Random(20260921)
    res = []
    for n in S.LEAF_SIZES:
        raw = S.leaf_raw(rng, n)
        res.append({"n": n, "crc32c": ref.ref_crc32c_extend(0, raw, n), "max_compressed_length": ref.ref_snappy_max_compressed_length(n),
                    "compressed": S.digest(compress(raw))})
    return res


def main():
    out = {"gpu_corruptions": gpu_corruptions(), "warp": {"short": warp(False), "long": warp(True)}, "leaf": leaf()}
    path = os.path.join(HERE, "snappy_ref_results.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0)
    print("wrote", path, os.path.getsize(path))


if __name__ == "__main__":
    main()
