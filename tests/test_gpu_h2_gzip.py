"""GPU: b2_h2_decompress_requests (the GzipDecompress step of ProcessHttpRequest, k_h2_inflate) against the oracle
(orc_h2_decompress, itself pinned to the system zlib in tests/test_oracle_h2_gzip.py): status, slot placement and every inflated byte,
for the gzip stream families and the header-rule table, through b2_h2_process_batch with 64 connections per batch; the 1 MiB
limits; NO_ROOM in message order; the argument checks; echo by reference (B2_H2_RESP_BODY_IN_UNZ); a live grpcio gzip client;
and b2::GpuH2Messenger through the C++ driver tests/cpp/h2_gzip_messenger_test.cc."""
import gzip
import os
import random
import subprocess
import threading

import numpy as np
import pytest

import _h2gzip as Z
import _oracle as O
import _oracle_h2gzip as OZ

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_CONNS = 64


def make_ctx(stream_bytes=4096 + (256 << 10), max_resp_bytes=64 << 20, pending=64):
    import brpc_b200
    ctx = brpc_b200.Context(device=0, max_batch_bytes=32 << 20, max_msgs=1 << 14, max_runs=256, max_resp_bytes=max_resp_bytes)
    ctx.h2_configure(max_conns=N_CONNS, max_pending=pending, stream_bytes=stream_bytes)
    for i in range(N_CONNS):
        ctx.h2_conn_reset(i)
    return ctx


def _merged_oracle(conn_bytes):
    """every connection through its own oracle H2Conn; the messages re-based onto one blob, in run order (as the device lists them)"""
    msgs, blobs, at = [], [], 0
    orc = []
    for b in conn_bytes:
        c = O.H2Conn(); orc.append(c)
        err, cons, m, ctrl, blob, _, _ = c.consume(b)
        assert err == 2 and cons == len(b)
        m = m.copy()
        for f in ("headers_off", "body_off", "msg_off", "path_off"):
            m[f] += at
        msgs.append(m); blobs.append(blob.tobytes()); at += len(blob)
    return np.concatenate(msgs), b"".join(blobs), orc


def _device(ctx, conn_bytes, out_cap=32 << 20, unz_cap=16 << 20):
    import brpc_b200
    data, runs = brpc_b200.make_runs(conn_bytes)
    runs["socket_id"] = np.arange(len(conn_bytes), dtype=np.uint64)
    rs, msgs, out = ctx.h2_process_batch(data, runs, msg_cap=1 << 14, out_cap=out_cap)
    assert all(int(s["parse_error"]) == 2 and int(s["consumed"]) == len(b) for s, b in zip(rs, conn_bytes))
    res, unz = ctx.h2_decompress_requests(msgs, out_cap=unz_cap)
    return data, msgs, out, res, unz


def _compare(ctx, calls_per_conn, chunk=None, unz_cap=16 << 20):
    conn_bytes = [Z.connection(calls, seed=i, chunk=chunk) for i, calls in enumerate(calls_per_conn)]
    data, dmsgs, dout, dres, dunz = _device(ctx, conn_bytes, unz_cap=unz_cap)
    omsgs, oblob, orc = _merged_oracle(conn_bytes)
    assert len(dmsgs) == len(omsgs) == sum(len(c) for c in calls_per_conn)
    ores, ounz = OZ.h2_decompress(omsgs, oblob, out_cap=unz_cap)
    for f in ("status", "out_off", "out_len"):
        assert list(dres[f]) == list(ores[f]), f
    ok = dres["status"] == Z.OK
    end = int((dres["out_off"][ok].astype(np.int64) + dres["out_len"][ok]).max()) if ok.any() else 0
    assert dunz[:end].tobytes() == ounz
    return dres, data, dmsgs, dout, dunz, orc


@pytest.mark.parametrize("chunk", [None, 1000], ids=["one-data-frame", "split-data-frames"])
def test_device_equals_oracle_on_every_family(chunk):
    fams = Z.stream_families(random.Random(21), corrupt_limit=2048)
    rng = random.Random(22)
    calls = []
    for k, (_, s) in enumerate(fams):
        grpc = k % 3 != 0
        calls.append((s, grpc, 1, [(b"grpc-encoding", b"gzip")] if grpc else [(b"content-encoding", b"gzip")]))
    for _, grpc, flag, headers, _ in Z.HEADER_RULES:
        calls.append((gzip.compress(Z.text(rng, 3000), mtime=0), grpc, flag, headers))
    ctx = make_ctx()
    per_batch = N_CONNS * 24
    n_ok = 0
    for at in range(0, len(calls), per_batch):
        part = calls[at:at + per_batch]
        conns = [part[i::N_CONNS] for i in range(N_CONNS)]
        res = _compare(ctx, [c for c in conns if c], chunk=chunk)[0]
        n_ok += int((res["status"] == Z.OK).sum())
        for i in range(N_CONNS):
            ctx.h2_conn_reset(i)
    assert n_ok > len(fams) // 2


def test_one_mebibyte_limits():
    rng = random.Random(31)
    big_in = gzip.compress(bytes(rng.getrandbits(8) for _ in range((1 << 20) + 4096)), mtime=0)
    assert len(big_in) > 1 << 20
    calls = [(gzip.compress(bytes(1 << 20), mtime=0), True, 1, [(b"grpc-encoding", b"gzip")]),           # exactly kGzMaxOut
             (gzip.compress(bytes((1 << 20) + 1), mtime=0), True, 1, [(b"grpc-encoding", b"gzip")]),     # one byte more
             (big_in, True, 1, [(b"grpc-encoding", b"gzip")]),                                        # input over 1 MiB
             (gzip.compress(b"small", mtime=0), False, 0, [(b"content-encoding", b"gzip")])]
    ctx = make_ctx(stream_bytes=4096 + (2 << 20), pending=8)
    res = _compare(ctx, [calls[:2], calls[2:]], unz_cap=4 << 20)[0]
    assert list(res["status"]) == [Z.OK, Z.HOST, Z.HOST, Z.OK]
    assert int(res["out_len"][0]) == 1 << 20 and int(res["out_len"][3]) == 5


def test_no_room_in_message_order_and_nothing_past_out_cap():
    payloads = [gzip.compress(bytes([65 + k]) * (1000 * (k + 1)), mtime=0) for k in range(6)]
    calls = [(p, True, 1, [(b"grpc-encoding", b"gzip")]) for p in payloads]
    ctx = make_ctx()
    import brpc_b200
    data, runs = brpc_b200.make_runs([Z.connection(calls)])
    rs, msgs, out = ctx.h2_process_batch(data, runs, out_cap=4 << 20)
    cap = 1000 + 2000 + 3000 + 3999
    buf = np.full(cap + 4096, 0xA5, np.uint8)
    res, _ = ctx.h2_decompress_requests(msgs, out=buf[:cap])
    assert list(res["status"]) == [Z.OK] * 3 + [Z.NO_ROOM] * 3
    assert list(res["out_off"][:3]) == [0, 1000, 3000]
    assert (buf[cap:] == 0xA5).all() and (buf[6000:cap] == 0xA5).all()          # only the inflated bytes are written
    assert buf[:6000].tobytes() == b"A" * 1000 + b"B" * 2000 + b"C" * 3000
    ores, ounz = OZ.h2_decompress(*_merged_oracle([Z.connection(calls)])[:2], out_cap=cap)
    assert list(ores["status"]) == list(res["status"]) and ounz == buf[:6000].tobytes()


def test_invalid_arguments():
    import brpc_b200
    ctx = make_ctx()
    with pytest.raises(brpc_b200.B2Error) as e:                                  # no batch on this context yet
        ctx.h2_decompress_requests(np.zeros(1, brpc_b200.abi.H2_MSG_DT))
    assert e.value.code == -1
    calls = [(gzip.compress(b"valid", mtime=0), True, 1, [(b"grpc-encoding", b"gzip")])] * 2
    data, runs = brpc_b200.make_runs([Z.connection(calls)])
    rs, msgs, out = ctx.h2_process_batch(data, runs, out_cap=1 << 20)
    res, unz = ctx.h2_decompress_requests(msgs)
    assert list(res["status"]) == [Z.OK, Z.OK]
    for field, value in [("headers_off", 1 << 20), ("headers_len", 1 << 20), ("body_off", data.nbytes), ("msg_len", 1 << 21)]:
        bad = msgs.copy(); bad[1][field] = value
        with pytest.raises(brpc_b200.B2Error) as e:
            ctx.h2_decompress_requests(bad)
        assert e.value.code == -1, field
    ctx.h2_decompress_requests(msgs)                                             # the batch is still live


def test_echo_by_reference_from_the_inflated_message():
    """process -> decompress -> b2_h2_pack_responses with B2_H2_RESP_BODY_IN_UNZ: the frames equal the oracle's pack_response of the
    inflated message, over several batches (the HPACK encoder tables and windows carry over)"""
    from brpc_b200.abi import H2_RESPONSE_DT
    rng = random.Random(41)
    ctx = make_ctx()
    orc = [O.H2Conn() for _ in range(N_CONNS)]
    encs = [Z.T.HpackEncoder(random.Random(i)) for i in range(N_CONNS)]
    sid = [1] * N_CONNS
    import brpc_b200
    n_echo = 0
    for rnd in range(4):
        conn_bytes, plain = [], []
        for i in range(N_CONNS):
            b = (Z.T.PREFACE + Z.T.settings()) if rnd == 0 else b""
            for _ in range(rng.choice([1, 2, 3])):
                m = Z.text(rng, rng.choice([0, 10, 4096, 20000, 70000]))
                compressed = rng.random() < 0.8
                payload = gzip.compress(m, mtime=0) if compressed else m
                b += Z.request(encs[i], sid[i], payload, compressed=int(compressed), headers=[(b"grpc-encoding", b"gzip")],
                               chunk=rng.choice([None, 3000]))
                sid[i] += 2; plain.append(m)
            conn_bytes.append(b)
        data, runs = brpc_b200.make_runs(conn_bytes)
        runs["socket_id"] = np.arange(N_CONNS, dtype=np.uint64)
        rs, msgs, out = ctx.h2_process_batch(data, runs, msg_cap=1 << 12, out_cap=32 << 20)
        res, unz = ctx.h2_decompress_requests(msgs, out_cap=16 << 20)
        resps = np.zeros(len(msgs), H2_RESPONSE_DT); expect = []; k = 0
        for i in range(N_CONNS):
            e, cons, omsgs, octrl, oblob, _, _ = orc[i].consume(conn_bytes[i])
            st = rs[i]
            assert bytes(out[st["ctrl_off"]:st["ctrl_off"] + st["ctrl_len"]]) == octrl
            for m in msgs[st["first_msg"]:st["first_msg"] + st["n_msgs"]]:
                r = res[k]
                hb = bytes(out[m["headers_off"]:m["headers_off"] + m["headers_len"]])
                ct = dict(O.parse_header_records(hb))[b"content-type"]
                ct_off = int(m["headers_off"]) + hb.index(ct)
                if r["status"] == Z.OK:
                    body = unz[r["out_off"]:r["out_off"] + r["out_len"]].tobytes()
                    resps[k] = (i, m["stream_id"], 200, 1 | 8 | 16, ct_off, len(ct), r["out_off"], r["out_len"], 0, 0, 0, 0)
                    n_echo += 1
                else:
                    assert r["status"] == Z.NONE and not (m["flags"] & 4)
                    src = data if (m["flags"] & 16) else out
                    body = bytes(src[m["msg_off"]:m["msg_off"] + m["msg_len"]])
                    resps[k] = (i, m["stream_id"], 200, 1 | 8 | (2 if (m["flags"] & 16) else 4), ct_off, len(ct), m["msg_off"], m["msg_len"], 0, 0, 0, 0)
                assert body == plain[k]
                expect.append(orc[i].pack_response(int(m["stream_id"]), body, 200, ct, True, 0, b""))
                k += 1
        got = ctx.h2_pack_responses(None, resps)
        assert got == expect
    assert n_echo > 200


class DeviceGzipEngine:
    """b2_h2_process_batch -> b2_h2_decompress_requests -> b2_h2_pack_responses: a compressed Echo call is answered from its inflated
    message on the device (B2_H2_RESP_BODY_IN_UNZ), uncompressed."""
    def __init__(self, ctx):
        import brpc_b200
        from brpc_b200.abi import H2_RESPONSE_DT
        self.ctx, self.b2, self.RDT = ctx, brpc_b200, H2_RESPONSE_DT
        self.lock = threading.Lock()
        self.calls = self.inflated = 0

    def open(self, cid):
        with self.lock:
            self.ctx.h2_conn_reset(cid)

    def feed(self, cid, buf):
        with self.lock:
            data, runs = self.b2.make_runs([buf]); runs["socket_id"] = cid
            rs, msgs, out = self.ctx.h2_process_batch(data, runs, msg_cap=1024, out_cap=16 << 20)
            ctrl = bytes(out[int(rs["ctrl_off"][0]):int(rs["ctrl_off"][0]) + int(rs["ctrl_len"][0])])
            reply = b""
            if len(msgs):
                res, _ = self.ctx.h2_decompress_requests(msgs, out_cap=16 << 20)
                ct = b"application/grpc"; gm = b"unimplemented"
                unz = res["status"] == Z.OK
                ok = ((msgs["flags"] & 3) == 3) & (msgs["method_idx"] >= 0) & (unz | (res["status"] == Z.NONE))
                r = np.zeros(len(msgs), self.RDT)
                r["conn"] = cid; r["stream_id"] = msgs["stream_id"]; r["status_code"] = 200
                r["flags"] = 1 | np.where(ok, np.where(unz, 16, np.where(msgs["flags"] & 16, 2, 4)), 0)
                r["content_type_off"] = 0; r["content_type_len"] = len(ct)
                r["body_off"] = np.where(ok, np.where(unz, res["out_off"], msgs["msg_off"]), 0)
                r["body_len"] = np.where(ok, np.where(unz, res["out_len"], msgs["msg_len"]), 0)
                r["grpc_status"] = np.where(ok, 0, 12)
                r["grpc_message_off"] = len(ct); r["grpc_message_len"] = np.where(ok, 0, len(gm))
                reply = b"".join(self.ctx.h2_pack_responses(np.frombuffer(ct + gm + bytes(16), np.uint8), r))
                self.calls += len(msgs); self.inflated += int(unz.sum())
            return int(rs["consumed"][0]), ctrl + reply, int(rs["parse_error"][0]), len(msgs)


def test_live_grpcio_gzip_client_against_the_device():
    grpc = pytest.importorskip("grpc")
    from _h2loop import H2LoopServer
    from test_oracle_h2_grpcio import _channel, _echo
    import brpc_b200
    ctx = brpc_b200.Context(device=0, max_batch_bytes=16 << 20, max_msgs=1 << 14, max_runs=64, max_resp_bytes=64 << 20)
    ctx.h2_configure(max_conns=16, max_pending=192, stream_bytes=4096 + (256 << 10))
    eng = DeviceGzipEngine(ctx)
    srv = H2LoopServer(eng)
    rng = random.Random(51)
    try:
        with _channel(srv.port) as ch:
            call = _echo(ch)
            sizes = [0, 1, 100, 4096, 16384, 65000]
            msgs = [Z.text(rng, sizes[i % len(sizes)] if i % 3 else rng.randrange(0, 66000)) for i in range(1000)]
            for m in msgs[:100]:
                assert call(m, timeout=30, compression=grpc.Compression.Gzip) == m
            gate = threading.BoundedSemaphore(128)
            futs = []
            for m in msgs[100:]:
                gate.acquire()
                f = call.future(m, timeout=120, compression=grpc.Compression.Gzip)
                f.add_done_callback(lambda _f: gate.release())
                futs.append((m, f))
            for m, f in futs:
                try:
                    got = f.result()
                except grpc.RpcError as e:
                    raise AssertionError("call failed: %s; server loop errors: %r" % (e, srv.errors))
                assert got == m
        assert eng.calls == 1000 and not srv.errors, srv.errors
        assert eng.inflated > 700, eng.inflated
    finally:
        srv.close()


def test_gpu_h2_messenger_with_gzip_calls_cpp(tmp_path):
    exe = str(tmp_path / "h2_gzip_messenger_test")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-Wall", "-o", exe, os.path.join(ROOT, "tests", "cpp", "h2_gzip_messenger_test.cc"),
                           "-L" + os.path.join(ROOT, "brpc_b200"), "-lb2rpc", "-L" + os.path.join(ROOT, "oracle"), "-loracle_h2gzip", "-loracle", "-lz",
                           "-Wl,-rpath," + os.path.join(ROOT, "brpc_b200"), "-Wl,-rpath," + os.path.join(ROOT, "oracle")])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "h2 gzip messenger ok" in out.stdout
