"""CPU: the GzipDecompress step of ProcessHttpRequest (policy/http_rpc_protocol.cpp:1646-1683) in the oracle (orc_h2_decompress).
(1) what it inflates equals GzipDecompressBase (gzip_compress.cpp:138-176) driving the system zlib call for call
    (tests/_gzipdecompress.py), for every family of gzip-labelled bytes, and that restatement says the one-block body never fails;
(2) the header rules, case by case (the table in tests/_h2gzip.py);
(3) a live grpcio client with gzip compression against the oracle's h2 loop: every call is echoed."""
import gzip
import random
import threading

import pytest

import _gzipdecompress as GD
import _gzipstream as G
import _h2gzip as Z
import _oracle as O
import _oracle_h2gzip as OZ


def _decompress_all(calls, chunk=None):
    """one oracle connection per 32 calls; returns [(status, inflated bytes or None)] in call order"""
    got = []
    for at in range(0, len(calls), 32):
        part = calls[at:at + 32]
        c = O.H2Conn()
        err, cons, msgs, ctrl, blob, _, _ = c.consume(Z.connection(part, seed=at, chunk=chunk))
        assert err == 2 and len(msgs) == len(part)
        res, out = OZ.h2_decompress(msgs, blob, out_cap=64 << 20)
        for r in res:
            got.append((int(r["status"]), out[r["out_off"]:r["out_off"] + r["out_len"]] if r["status"] == Z.OK else None))
    return got


@pytest.mark.parametrize("grpc", [True, False], ids=["grpc-message", "h2-body"])
def test_oracle_equals_gzip_decompress_base_on_every_family(grpc):
    fams = Z.stream_families(random.Random(11))
    hdr = [(b"grpc-encoding", b"gzip")] if grpc else [(b"content-encoding", b"gzip")]
    calls = [(s, grpc, 1, hdr) for _, s in fams]
    got = _decompress_all(calls)
    n_nonempty = 0
    for (label, s), (st, b) in zip(fams, got):
        if not grpc and not s:
            assert st == Z.NONE, label                   # an empty body is never decompressed
            continue
        ok, want = GD.gzip_decompress_base(s)
        assert ok, label                                 # one block: GzipDecompressBase never fails (DESIGN §5)
        assert st == Z.OK and b == want, label
        n_nonempty += bool(want)
    assert n_nonempty > 1000


def test_gzip_decompress_base_on_one_block_is_the_gzip_input_stream():
    """the pin itself: for one-block bodies GzipDecompressBase hands over exactly what GzipInputStream yields"""
    for label, s in Z.stream_families(random.Random(12))[:80]:
        assert GD.gzip_decompress_base(s) == (True, G.gzip_input_stream(s, G.GZIP)), label


@pytest.mark.parametrize("case", Z.HEADER_RULES, ids=[c[0] for c in Z.HEADER_RULES])
def test_header_rules(case):
    _, grpc, flag, headers, want = case
    payload = gzip.compress(b"header rule " * 50, mtime=0)
    c = O.H2Conn()
    err, cons, msgs, ctrl, blob, _, _ = c.consume(Z.connection([(payload, grpc, flag, headers)]))
    assert len(msgs) == 1
    res, out = OZ.h2_decompress(msgs, blob)
    assert int(res[0]["status"]) == want
    if want == Z.OK:
        assert out[res[0]["out_off"]:res[0]["out_off"] + res[0]["out_len"]] == b"header rule " * 50
    else:
        assert res[0]["out_len"] == 0


def test_empty_body_and_bad_prefix_are_not_decompressed():
    payload = gzip.compress(b"x" * 100, mtime=0)
    enc = Z.T.HpackEncoder(random.Random(3))
    hdr = [(b"grpc-encoding", b"gzip")]
    conn = Z.T.PREFACE + Z.T.settings() + Z.request(enc, 1, b"", body=b"") + \
        Z.request(enc, 3, payload, body=b"\x01" + (len(payload) + 1).to_bytes(4, "big") + payload, headers=hdr)
    err, cons, msgs, ctrl, blob, _, _ = O.H2Conn().consume(conn)
    assert len(msgs) == 2 and not (msgs[1]["flags"] & 2)
    res, _ = OZ.h2_decompress(msgs, blob)
    assert list(res["status"]) == [Z.NONE, Z.NONE]


def test_no_room_follows_message_order():
    payloads = [gzip.compress(bytes([65 + k]) * (1000 * (k + 1)), mtime=0) for k in range(5)]
    calls = [(p, True, 1, [(b"grpc-encoding", b"gzip")]) for p in payloads]
    err, cons, msgs, ctrl, blob, _, _ = O.H2Conn().consume(Z.connection(calls))
    res, out = OZ.h2_decompress(msgs, blob, out_cap=1000 + 2000 + 3000 + 10)
    assert list(res["status"]) == [Z.OK, Z.OK, Z.OK, Z.NO_ROOM, Z.NO_ROOM]
    assert list(res["out_off"][:3]) == [0, 1000, 3000] and len(out) == 6000


def test_live_grpcio_gzip_client_against_the_oracle():
    grpc = pytest.importorskip("grpc")
    from _h2loop import H2LoopServer
    from test_oracle_h2_grpcio import _channel, _echo
    rng = random.Random(5)
    eng = Z.OracleGzipEngine()
    srv = H2LoopServer(eng)
    try:
        with _channel(srv.port) as ch:
            call = _echo(ch)
            sizes = [0, 1, 100, 4096, 16384, 70000, 200000]
            msgs = [Z.text(rng, sizes[i % len(sizes)] if i % 3 else rng.randrange(0, 200000)) for i in range(300)]
            for m in msgs[:100]:
                assert call(m, timeout=30, compression=grpc.Compression.Gzip) == m
            gate = threading.BoundedSemaphore(64)
            futs = []
            for m in msgs[100:]:
                gate.acquire()
                f = call.future(m, timeout=120, compression=grpc.Compression.Gzip)
                f.add_done_callback(lambda _f: gate.release())
                futs.append((m, f))
            for m, f in futs:
                assert f.result() == m
        assert eng.calls == 300 and not srv.errors, srv.errors
        assert eng.compressed_calls > 200, eng.compressed_calls   # C-core sends a message uncompressed when gzip would not shrink it
    finally:
        srv.close()
