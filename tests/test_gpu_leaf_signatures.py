"""GPU: the reference-signature leaves of seam 4 (b2_crc32c_extend, b2_snappy_raw_compress / _raw_uncompress, ...) against what the
reference's own crc32c.cc and vendored snappy return for the same inputs (tests/golden/snappy_ref_results.json)."""
import ctypes as C
import random

import pytest

import _snappy_cases as S

pytestmark = pytest.mark.gpu


def test_reference_signature_leaves_match_the_reference_build():
    import brpc_b200
    lib = brpc_b200.lib
    rng = random.Random(20260921)
    want = S.ref_results()["leaf"]
    assert [w["n"] for w in want] == S.LEAF_SIZES
    for w in want:
        n = w["n"]
        raw = S.leaf_raw(rng, n)
        # Extend chains: crc(a + b) == Extend(Extend(0, a), b)
        cut = n // 3
        got = lib.b2_crc32c_extend(lib.b2_crc32c_extend(0, raw[:cut], cut), raw[cut:], n - cut)
        assert got == w["crc32c"] == lib.b2_crc32c_extend(0, raw, n), n
        cap = lib.b2_snappy_max_compressed_length(n)
        assert cap == w["max_compressed_length"]
        b = C.create_string_buffer(cap + 16); bn = C.c_size_t(0)
        lib.b2_snappy_raw_compress(raw, n, b, C.byref(bn))
        comp = b.raw[:bn.value]
        assert S.digest(comp) == w["compressed"], "snappy bytes differ at n=%d" % n
        ul = C.c_size_t(0)
        assert lib.b2_snappy_get_uncompressed_length(comp, len(comp), C.byref(ul)) == 1 and ul.value == n
        out = C.create_string_buffer(n + 16)
        assert lib.b2_snappy_raw_uncompress(comp, len(comp), out) == 1 and out.raw[:n] == raw
    assert lib.b2_snappy_raw_uncompress(b"\x05abc", 4, C.create_string_buffer(64)) == 0       # malformed stream: false, like the reference
