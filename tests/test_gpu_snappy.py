"""GPU: snappy decode (a10).  (1) the leaf b2_snappy_uncompress_batch against the golden vectors
produced by the reference's vendored snappy (tests/golden/snappy_vectors.json, patterns of
test/brpc_snappy_compress_unittest.cpp:80-255) and against the reference decoder's results on
corrupted streams (tests/golden/snappy_ref_results.json); (2) snappy-compressed baidu_std requests
through the whole path vs the oracle (the compress x checksum matrix of test/brpc_server_unittest.cpp:1690-1880 restricted to
{none, snappy} x {none, crc32c})."""
import json
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

import _oracle as O  # noqa: E402
from _compare import assert_same  # noqa: E402
from _traffic import SEED, echo_frame, rnd62  # noqa: E402
import _snappy_cases as S  # noqa: E402


def _pattern(n):
    t = b"abcdefghijklmnopqrstuvwxyz0123456789"
    return (t * (n // len(t) + 1))[:n]


def test_snappy_golden_vectors_and_corruptions():
    import brpc_b200
    ctx = brpc_b200.Context(device=0, max_batch_bytes=32 << 20, max_msgs=1 << 16, max_runs=16, max_resp_bytes=64 << 20)
    vec = json.load(open(os.path.join(HERE, "golden", "snappy_vectors.json")))
    blobs, want = [], []
    for v in vec:
        comp = bytes.fromhex(v["comp_hex"])
        raw = bytes.fromhex(v["raw_hex"]) if "raw_hex" in v else _pattern(v["raw_len"])
        assert len(raw) == v["raw_len"]
        blobs.append(comp); want.append(raw)
    # corruptions: truncations, bit flips, bad offsets; expectation = the reference decoder's verdict (digest of its output)
    rng = random.Random(SEED)
    seeds = [b for b in blobs if 0 < len(b) < 5000]
    blobs += S.corrupted_blobs(rng, seeds)
    buf = bytearray(); offs = []; lens = []
    for b in blobs:
        buf += b"\x00" * rng.randrange(0, 5); offs.append(len(buf)); lens.append(len(b)); buf += b
    got = ctx.snappy_uncompress_batch(np.frombuffer(bytes(buf), np.uint8), offs, lens, 48 << 20)
    want = [S.digest(w) for w in want] + S.ref_results()["gpu_corruptions"]
    assert len(want) == len(blobs)
    bad = [i for i in range(len(blobs)) if S.digest(got[i]) != want[i]]
    assert not bad, "mismatch at %s (want None? %s)" % (bad[:5], [want[i] is None for i in bad[:5]])
    assert sum(w is None for w in want) > 50 and sum(w is not None for w in want[len(vec):]) > 5


def test_snappy_requests_through_the_path():
    import brpc_b200
    rng = random.Random(SEED + 1)
    ms = [dict(brpc_b200.ECHO_METHOD, response_checksum_type=rng.choice([0, 1]))]
    for tile in (512, 8192):
        ctx = brpc_b200.Context(device=0, max_batch_bytes=64 << 20, max_msgs=1 << 18, max_runs=4096, tile_bytes=tile, methods=ms)
        cfg = O.make_config(methods=ms)
        streams = []
        for s in range(60):
            fr = []
            for i in range(rng.randrange(1, 12)):
                n = rng.choice([0, 1, 10, 100, 1000, 5000, 70000])
                msg = rng.choice([_pattern(n), rnd62(rng, n), b"r" * n, (rnd62(rng, 50) * (n // 50 + 1))[:n]])
                f = echo_frame(rng, i, msg, compress_type=rng.choice([0, 1, 1, 1]), checksum_type=rng.choice([0, 0, 1]),
                               attachment=rng.choice([b"", b"", rnd62(rng, 37)]))
                if rng.random() < 0.15:                      # corrupt the compressed body / checksum
                    f = bytearray(f); f[-1 - rng.randrange(max(1, min(40, len(f) - 60)))] ^= 0x41; f = bytes(f)
                fr.append(f)
            streams.append(b"".join(fr))
        data, runs = brpc_b200.make_runs(streams)
        dev = ctx.process_batch(data, runs)
        orc = O.process_batch(cfg, data, runs)
        assert_same(dev, orc, "tile=%d" % tile)
        st = dev[1]["status"]
        assert (st == 0).sum() > 50 and (st == 1).sum() > 3


def test_snappy_encoder_bit_exact_golden():
    """Compressed bytes must equal what the reference's vendored snappy 1.1.3 produces (golden vectors
    generated through oracle/_ref), for every pattern of brpc_snappy_compress_unittest.cpp plus mixes."""
    import brpc_b200
    ctx = brpc_b200.Context(device=0, max_batch_bytes=32 << 20, max_msgs=1 << 16, max_runs=16, max_resp_bytes=64 << 20)
    vec = json.load(open(os.path.join(HERE, "golden", "snappy_vectors.json")))
    raws, want = [], []
    for v in vec:
        raws.append(bytes.fromhex(v["raw_hex"]) if "raw_hex" in v else _pattern(v["raw_len"])); want.append(bytes.fromhex(v["comp_hex"]))
    buf = bytearray(); offs = []; lens = []
    rng = random.Random(3)
    for r in raws:
        buf += b"\x00" * rng.randrange(0, 7); offs.append(len(buf)); lens.append(len(r)); buf += r
    got = ctx.snappy_compress_batch(np.frombuffer(bytes(buf), np.uint8), offs, lens, 48 << 20)
    bad = [(vec[i]["name"], len(got[i]), len(want[i])) for i in range(len(raws)) if got[i] != want[i]]
    assert not bad, bad[:6]
    # and the device decoder inverts the device encoder
    buf2 = bytearray(); offs2 = []; lens2 = []
    for g in got:
        offs2.append(len(buf2)); lens2.append(len(g)); buf2 += g
    back = ctx.snappy_uncompress_batch(np.frombuffer(bytes(buf2), np.uint8), offs2, lens2, 48 << 20)
    assert back == raws


def test_snappy_replies_through_the_path():
    """cntl->set_response_compress_type(COMPRESS_TYPE_SNAPPY) on the echo method, with and without crc32c."""
    import brpc_b200
    rng = random.Random(SEED + 2)
    for cks in (0, 1):
        ms = [dict(brpc_b200.ECHO_METHOD, response_compress_type=1, response_checksum_type=cks)]
        ctx = brpc_b200.Context(device=0, max_batch_bytes=64 << 20, max_msgs=1 << 18, max_runs=4096, methods=ms)
        cfg = O.make_config(methods=ms)
        streams = []
        for s in range(40):
            fr = []
            for i in range(rng.randrange(1, 10)):
                n = rng.choice([0, 1, 14, 15, 16, 100, 1000, 5000, 70000, 140000])
                msg = rng.choice([_pattern(n), rnd62(rng, n), b"r" * n, (rnd62(rng, 50) * (n // 50 + 1))[:n]])
                fr.append(echo_frame(rng, i, msg, compress_type=rng.choice([0, 0, 1]), checksum_type=rng.choice([0, 1]),
                                     attachment=rng.choice([b"", rnd62(rng, 37)])))
            streams.append(b"".join(fr))
        data, runs = brpc_b200.make_runs(streams)
        dev = ctx.process_batch(data, runs)
        orc = O.process_batch(cfg, data, runs)
        assert_same(dev, orc, "cks=%d" % cks)
        assert (dev[1]["status"] == 0).sum() > 50


def test_streaming_frames_with_snappy_payloads():
    """BASELINE configs[4] shape: streaming_rpc DATA frames whose payloads the application snappy-compressed
    (policy::SnappyCompress), cut + meta-decoded + decompressed on the device, interleaved with baidu_std calls."""
    import brpc_b200
    rng = random.Random(SEED + 3)
    ctx = brpc_b200.Context(device=0, max_batch_bytes=64 << 20, max_msgs=1 << 16, max_runs=256, stream_handler=1)
    cfg = O.make_config(stream_handler=1)
    streams = []
    for s in range(48):
        fr = []
        for i in range(rng.randrange(1, 8)):
            n = rng.choice([0, 10, 1000, 70000, 262144])
            raw = rng.choice([_pattern(n), rnd62(rng, min(n, 30000)), (rnd62(rng, 64) * (n // 64 + 1))[:n]])
            comp = O.snappy_compress(raw)
            if rng.random() < 0.15 and len(comp) > 4:
                comp = bytearray(comp); comp[rng.randrange(len(comp))] ^= 0x10; comp = bytes(comp)
            fr.append(O.pack_stream_frame(1000 + s, 2000 + s, rng.choice([3, 3, 3, 4, 1]), rng.choice([None, False]), comp))
            if rng.random() < 0.3:
                fr.append(echo_frame(rng, i, rnd62(rng, 100)))
        streams.append(b"".join(fr))
    data, runs = brpc_b200.make_runs(streams)
    dev = ctx.process_batch(data, runs)
    orc = O.process_batch(cfg, data, runs)
    assert_same(dev, orc, "streaming")
    m = dev[1]
    assert ((m["status"] == 4) & (m["resp_len"] > 100000)).sum() > 3 and ((m["status"] == 4) & (m["error_code"] == 1003)).sum() > 0
