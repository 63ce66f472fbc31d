"""CPU: the WARP-cooperative device code of the hot path — warp_crc32c_update, warp_snappy_decode / _compress, pack_one — on an emulated 32-lane
warp (tests/cpp/warp_emul_prelude.h: 32 host threads, every __shfl / __ballot / __syncwarp a barrier plus an exchange), out of the generated
host-compilable copy of b2_kernels.cuh.  CRC against the oracle (which the reference's crc32c.cc pins), snappy against what the reference's
vendored snappy returned for the same inputs (tests/golden/snappy_ref_results.json), and whole batches — decode_one per message, slot scan,
pack_one per message — against the oracle's descriptors and reply bytes for every kind of message (errors, CRC32C, snappy and gzip / zlib requests, snappy replies, attachments, client sockets, stream frames)."""
import ctypes as C
import os
import random
import subprocess
import sys
import zlib

import numpy as np
import pytest

LONG = os.environ.get("B2_LONG_TESTS") == "1"      # the full sizes: ~18 minutes on 8 cores (every warp collective is a 32-thread barrier)

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
import _oracle as O  # noqa: E402
from _traffic import SEED, echo_frame, echo_pb, mixed_frames, raw_request_frame, rnd62, split_runs  # noqa: E402
from brpc_b200.abi import ECHO_METHOD, MSG_DT  # noqa: E402
from brpc_b200.messenger import make_runs  # noqa: E402
from _compare import MSG_FIELDS  # noqa: E402
import _snappy_cases as S  # noqa: E402


@pytest.fixture(scope="module")
def wh():
    cpp = os.path.join(HERE, "cpp")
    so = os.path.join(cpp, "libwarp_host.so")
    deps = [os.path.join(cpp, f) for f in ("gen_kernels_host.py", "warp_emul_prelude.h", "warp_host.cc")] + \
           [os.path.join(ROOT, "brpc_b200", "csrc", f) for f in ("b2_kernels.cuh", "b2_core.cuh", "b2_inflate.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call([sys.executable, os.path.join(cpp, "gen_kernels_host.py")])
        subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-w", "-pthread", "-I", os.path.join(cpp, "stub"), "-I", os.path.join(ROOT, "include"),
                               "-o", so, os.path.join(cpp, "warp_host.cc")])
    lib = C.CDLL(so)
    lib.wh_crc32c_extend.restype = C.c_uint32
    lib.wh_crc32c_extend.argtypes = [C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.wh_snappy_uncompress.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.wh_snappy_compress.restype = C.c_uint32
    lib.wh_snappy_compress.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p]
    lib.wh_create.restype = C.c_void_p
    lib.wh_create.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_char_p]
    lib.wh_destroy.argtypes = [C.c_void_p]
    lib.wh_add_method.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.wh_process.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
    return lib


def test_warp_crc32c_against_the_oracle(wh):
    rng = random.Random(SEED + 971)
    agree = C.c_uint32()
    assert wh.wh_crc32c_extend(0, (b"\x00" * 32 + b"pad"), 32, C.byref(agree)) == 0x8a9136aa and agree.value       # RFC 3720 B.4
    base = np.frombuffer(bytes(rng.getrandbits(8) for _ in range(70000)) + bytes(64), np.uint8).copy()
    sizes = list(range(0, 130)) + [255, 256, 257, 511, 512, 513, 1023, 1024, 1027, 4095, 4096, 5000, 65536, 69999] if LONG else \
        list(range(0, 70)) + [100, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024, 1027, 2048, 4099, 9000, 20011]
    for n in sizes:
        for lead in ((0, 1, 5, 15, 16) if LONG else (0, 1, 5, 15)):
            init = rng.choice([0, 0xffffffff, rng.getrandbits(32)])
            got = wh.wh_crc32c_extend(init, base.ctypes.data + 16 + lead, n, C.byref(agree))
            assert agree.value and got == O.crc32c(bytes(base[16 + lead:16 + lead + n]), init), (n, lead)


def test_warp_snappy_against_the_reference_library(wh):
    want = S.ref_results()["warp"]["long" if LONG else "short"]
    corrupt = iter(want["corrupt"])
    rng = random.Random(SEED + 972)
    for raw, want_comp in zip(S.warp_raws(rng, LONG), want["compress"]):
        out = C.create_string_buffer(len(raw) + len(raw) // 6 + 96)
        n = wh.wh_snappy_compress(raw, len(raw), out)
        assert S.digest(out.raw[:n]) == want_comp, len(raw)                                      # bit-exact with the vendored snappy 1.1.3
        back = C.create_string_buffer(max(1, len(raw))); prod = C.c_uint32()
        assert wh.wh_snappy_uncompress(out.raw[:n], n, back, len(raw), C.byref(prod)) == 1 and back.raw[:prod.value] == raw
        for _ in range(S.warp_corruptions_per_raw(LONG)):                                       # corrupted streams: the reference's verdict
            if not n: break
            b = S.warp_corruption(rng, out.raw[:n])
            ul, ok_ref, want_out = next(corrupt)
            if ok_ref is None:
                continue
            dbuf = C.create_string_buffer(max(1, ul)); prod = C.c_uint32()
            ok_dev = wh.wh_snappy_uncompress(b, len(b), dbuf, ul, C.byref(prod))
            assert ok_dev == (1 if ok_ref else 0), (len(raw), len(b))
            if ok_ref:
                assert S.digest(dbuf.raw[:prod.value]) == want_out
    assert next(corrupt, None) is None


def _process(wh, k, cfg, chunks, flags=0):
    data, runs = make_runs(chunks)
    runs["flags"] = flags
    rs, msgs, resp = O.process_batch(cfg, data, runs, resp_cap=64 << 20)
    n = len(msgs)
    if n == 0:
        return 0
    buf = np.concatenate([np.asarray(data, np.uint8), np.zeros(1024, np.uint8)])
    fo = (msgs["frame_off"].astype(np.uint32) | ((0 if flags & 4 else 1) * (msgs["protocol"] != 1).astype(np.uint32) << 31)).astype(np.uint32)
    run_of = msgs["run_idx"].astype(np.uint32)
    dmsgs = np.zeros(n, MSG_DT); cap = int(len(data) * 3 + n * 256 + (1 << 20)); dresp = np.zeros(cap, np.uint8); used = C.c_uint32()
    rc = wh.wh_process(k, buf.ctypes.data, runs.ctypes.data, len(runs), fo.ctypes.data, run_of.ctypes.data, n, dmsgs.ctypes.data, dresp.ctypes.data, cap, C.byref(used))
    assert rc == 0
    for f in MSG_FIELDS:
        if f in ("resp_off",):
            continue
        assert np.array_equal(dmsgs[f], msgs[f]), (f, [(i, int(dmsgs[f][i]), int(msgs[f][i])) for i in range(n) if dmsgs[f][i] != msgs[f][i]][:5])
    for i in range(n):
        if int(msgs["status"][i]) == 7:
            continue                                                                             # client result reported in place (batch offsets)
        a, b = int(dmsgs["resp_off"][i]), int(msgs["resp_off"][i]); ln = int(msgs["resp_len"][i])
        assert bytes(dresp[a:a + ln]) == bytes(resp[b:b + ln]), (i, int(msgs["status"][i]), ln)
    return n


def _make(wh, methods, identity=None, stream_handler=0):
    k = wh.wh_create(0, (1 << 1) | (1 << 2), stream_handler, identity)
    for m in methods:
        wh.wh_add_method(k, m["service_full_name"], m["service_name"], m["method_name"], m["request_type_name"], m["handler"], m["echo_attachment"],
                         m["response_checksum_type"], m["response_compress_type"])
    return k


def test_decode_and_pack_of_whole_batches_on_the_emulated_warp(wh):
    rng = random.Random(SEED + 973)
    total = 0
    for r_cks, r_cmp, identity in [(0, 0, None), (1, 0, b"10.0.0.1:8000"), (0, 1, None), (1, 1, None)]:
        ms = [dict(ECHO_METHOD, response_checksum_type=r_cks, response_compress_type=r_cmp)]
        k = _make(wh, ms, identity); cfg = O.make_config(methods=ms, server_identity=identity)
        streams = [mixed_frames(rng, rng.randrange(10, 60) if LONG else 25, big=LONG) for _ in range(6 if LONG else 4)]
        total += _process(wh, k, cfg, split_runs(rng, streams))
        # snappy / gzip / zlib requests, with and without CRC32C, some corrupted
        fr = []
        for i in range(60 if LONG else 32):
            msg = rng.choice([rnd62(rng, rng.choice([0, 10, 1000, 20000] if LONG else [0, 10, 1000, 4000])), b"r" * rng.choice([1, 5000, 70000] if LONG else [1, 3000])])
            kind = rng.choice(["snappy", "gzip", "zlib", "plain"])
            if kind in ("gzip", "zlib"):
                c = zlib.compressobj(rng.choice([0, 1, 6]), zlib.DEFLATED, 31 if kind == "gzip" else 15)
                body = c.compress(echo_pb(msg)) + c.flush()
                if rng.random() < 0.2 and body:
                    b = bytearray(body); b[rng.randrange(len(b))] ^= 0x10; body = bytes(b)
                f = raw_request_frame(body, 7000 + i, compress_type=2 if kind == "gzip" else 3, attachment=rng.choice([b"", rnd62(rng, 33)]))
            else:
                f = echo_frame(rng, i, msg, compress_type=1 if kind == "snappy" else 0, checksum_type=rng.choice([0, 1]), attachment=rng.choice([b"", rnd62(rng, 33)]))
                if rng.random() < 0.15:
                    b = bytearray(f); b[-1 - rng.randrange(min(40, len(b) - 50))] ^= 0x41; f = bytes(b)
            fr.append(f)
        total += _process(wh, k, cfg, [b"".join(fr[i::4]) for i in range(4)])
        wh.wh_destroy(k)
    assert total > (900 if LONG else 400)


def test_client_sockets_and_stream_payloads_on_the_emulated_warp(wh):
    rng = random.Random(SEED + 974)
    ms = [dict(ECHO_METHOD, response_compress_type=1, response_checksum_type=1)]
    k = _make(wh, ms); cfg = O.make_config(methods=ms)
    streams = [mixed_frames(rng, 60 if LONG else 30) for _ in range(6 if LONG else 4)]
    data, runs = make_runs(split_runs(rng, streams, cut_tail=False))
    rs, msgs, resp = O.process_batch(cfg, data, runs)
    replies = [bytes(resp[int(m["resp_off"]):int(m["resp_off"]) + int(m["resp_len"])]) for m in msgs if int(m["resp_len"]) and int(m["status"]) in (0, 1)]
    n = _process(wh, k, cfg, [b"".join(replies[i::5]) for i in range(5)], flags=1)       # the server's (snappy + CRC) replies as client-side input
    assert n > (200 if LONG else 60)
    wh.wh_destroy(k)
    k = _make(wh, [dict(ECHO_METHOD)], stream_handler=1); cfg = O.make_config(stream_handler=1)
    frames = []
    n_frames = 40 if LONG else 18
    for i in range(n_frames):
        raw = rng.choice([rnd62(rng, rng.choice([0, 100, 30000] if LONG else [0, 100, 4000])), b"z" * (5000 if LONG else 1500)])
        payload = O.snappy_compress(raw)
        if rng.random() < 0.2 and payload:
            b = bytearray(payload); b[rng.randrange(len(b))] ^= 4; payload = bytes(b)
        frames.append(O.pack_stream_frame(1000 + i, -1, 3, None, payload))
    assert _process(wh, k, cfg, [b"".join(frames[i::3]) for i in range(3)]) == n_frames
    wh.wh_destroy(k)
