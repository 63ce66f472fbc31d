"""gzip-compressed h2 / gRPC requests for the tests of the GzipDecompress step of ProcessHttpRequest
(policy/http_rpc_protocol.cpp:1646-1683): the header-rule table, the families of gzip streams, and client connections that carry
them (tests only)."""
import gzip
import random
import zlib

import _h2traffic as T
import _oracle as O
import _oracle_h2gzip as OZ
from test_oracle_gzip import _gzip_with_header

NONE, OK, NO_ENCODING, NOT_GZIP, FAILED, HOST, NO_ROOM = range(7)
GRPC_CT, JSON_CT = b"application/grpc", b"application/json"

# (id, gRPC?, compressed flag of the 5-byte prefix, extra header fields in order, expected status).  GetHeader sees the value
# HttpHeader::AppendHeader built (http_header.cpp:100-116): names case-insensitive, a repeated field folded with "," onto a
# non-empty value and overwriting an empty one; only the exact string "gzip" is inflated.
HEADER_RULES = [
    ("grpc-missing", True, 1, [], NO_ENCODING),
    ("grpc-gzip", True, 1, [(b"grpc-encoding", b"gzip")], OK),
    ("grpc-GZIP", True, 1, [(b"grpc-encoding", b"GZIP")], NOT_GZIP),
    ("grpc-gzip-space", True, 1, [(b"grpc-encoding", b"gzip ")], NOT_GZIP),
    ("grpc-deflate", True, 1, [(b"grpc-encoding", b"deflate")], NOT_GZIP),
    ("grpc-identity", True, 1, [(b"grpc-encoding", b"identity")], NOT_GZIP),
    ("grpc-duplicated", True, 1, [(b"grpc-encoding", b"gzip"), (b"grpc-encoding", b"gzip")], NOT_GZIP),
    ("grpc-empty-then-gzip", True, 1, [(b"grpc-encoding", b""), (b"grpc-encoding", b"gzip")], OK),
    ("grpc-gzip-then-empty", True, 1, [(b"grpc-encoding", b"gzip"), (b"grpc-encoding", b"")], NOT_GZIP),
    ("grpc-empty", True, 1, [(b"grpc-encoding", b"")], NOT_GZIP),
    ("grpc-mixed-case-name", True, 1, [(b"Grpc-Encoding", b"gzip")], OK),
    ("grpc-flag0-with-header", True, 0, [(b"grpc-encoding", b"gzip")], NONE),
    ("grpc-flag0-no-header", True, 0, [], NONE),
    ("grpc-content-encoding-ignored", True, 1, [(b"content-encoding", b"gzip")], NO_ENCODING),
    ("grpc-both", True, 1, [(b"content-encoding", b"identity"), (b"grpc-encoding", b"gzip")], OK),
    ("http-content-encoding", False, 0, [(b"content-encoding", b"gzip")], OK),
    ("http-missing", False, 0, [], NONE),
    ("http-grpc-encoding-ignored", False, 0, [(b"grpc-encoding", b"gzip")], NONE),
    ("http-deflate", False, 0, [(b"content-encoding", b"deflate")], NOT_GZIP),
    ("http-duplicated", False, 0, [(b"content-encoding", b"gzip"), (b"content-encoding", b"gzip")], NOT_GZIP),
    ("http-mixed-case-name", False, 0, [(b"Content-Encoding", b"gzip")], OK),
]


def text(rng, n):
    words = [b"echo", b"brpc", b"socket", b"message", b"iobuf", b"attachment", b"gzip", b"stream", b"\n"]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words) + b" "
    return bytes(out[:n])


def _raw_deflate(data):
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    return c.compress(data) + c.flush()


def stream_families(rng, corrupt_limit=2048):
    """(label, gzip-labelled bytes) covering what GzipDecompress meets: gzip at levels 0-9, header fields, concatenated members,
    zlib-wrapped and raw-deflate streams, the empty body, truncation at every byte and bit flips of streams up to corrupt_limit."""
    out = [("empty", b"")]
    for lvl in range(10):
        for n in (0, 1, 700, 5000):
            out.append(("level%d-%d" % (lvl, n), gzip.compress(text(rng, n), compresslevel=lvl, mtime=0)))
    d = text(rng, 3000)
    for kw in [dict(extra=b"\x01\x02abcd"), dict(name=b"file.bin"), dict(comment=b"a comment"), dict(hcrc=True),
               dict(extra=b"x" * 300, name=b"n" * 100, comment=b"c" * 50, hcrc=True)]:
        out.append(("header-" + "-".join(sorted(kw)), _gzip_with_header(d, **kw)))
    out.append(("concatenated", gzip.compress(b"first member ", mtime=0) + gzip.compress(text(rng, 2000), mtime=0)))
    out.append(("concatenated-garbage", gzip.compress(b"member", mtime=0) + b"garbage after"))
    out.append(("zlib-wrapped", zlib.compress(d)))
    out.append(("raw-deflate", _raw_deflate(d)))
    out.append(("random", bytes(rng.getrandbits(8) for _ in range(300))))
    out.append(("incompressible", gzip.compress(bytes(rng.getrandbits(8) for _ in range(9000)), mtime=0)))
    base = [gzip.compress(text(rng, 300), mtime=0), gzip.compress(text(rng, 6000), mtime=0), gzip.compress(bytes(range(256)) * 4, 0, mtime=0)]
    for k, s in enumerate(base):
        assert len(s) <= corrupt_limit
        for cut in range(len(s)):
            out.append(("cut%d-%d" % (k, cut), s[:cut]))
        for pos in range(len(s)):
            b = bytearray(s); b[pos] ^= 1 << (pos % 8)
            out.append(("flip%d-%d" % (k, pos), bytes(b)))
    return out


def body_of(payload, grpc, compressed):
    if not grpc:
        return payload
    return bytes([compressed]) + len(payload).to_bytes(4, "big") + payload


def request(enc, sid, payload, grpc=True, compressed=1, headers=((b"grpc-encoding", b"gzip"),), chunk=None, body=None,
            path=b"/example.EchoService/Echo"):
    """HEADERS + DATA frames of one call.  chunk: DATA payload size (None = one frame when it fits); body overrides the framing of
    payload (e.g. a prefix whose length does not match)."""
    fields = [enc.field(b":method", b"POST"), enc.field(b":scheme", b"http"), enc.field(b":path", path),
              enc.field(b":authority", b"127.0.0.1:8010"), enc.field(b"content-type", GRPC_CT if grpc else JSON_CT)]
    fields += [enc.field(n, v) for n, v in headers]
    body = body_of(payload, grpc, compressed) if body is None else body
    frames = [T.frame(1, 0x4 | (0 if body else 0x1), sid, b"".join(fields))]
    step = min(chunk or 16000, 16000)
    pieces = [body[i:i + step] for i in range(0, len(body), step)]
    for j, pc in enumerate(pieces):
        frames.append(T.frame(0, 0x1 if j == len(pieces) - 1 else 0, sid, pc))
    return b"".join(frames)


def connection(calls, seed=0, chunk=None):
    """calls: [(payload, grpc, compressed, headers)] -> the client's bytes: preface, SETTINGS, one stream per call in order."""
    rng = random.Random(seed)
    enc = T.HpackEncoder(rng)
    parts = [T.PREFACE, T.settings()]
    for k, (payload, grpc, compressed, headers) in enumerate(calls):
        parts.append(request(enc, 1 + 2 * k, payload, grpc, compressed, headers, chunk=chunk))
    return b"".join(parts)


class OracleGzipEngine:
    """The oracle's h2 server loop with the GzipDecompress step: a compressed call to Echo is answered with its inflated message,
    uncompressed (the echo service sets no response_compress_type).  compressed_calls counts the calls whose prefix flag was set."""
    def __init__(self):
        self.conns = {}
        self.compressed_calls = 0
        self.calls = 0

    def open(self, cid):
        self.conns[cid] = O.H2Conn()

    def feed(self, cid, buf):
        c = self.conns[cid]
        err, cons, msgs, ctrl, blob, _, _ = c.consume(buf)
        out = [ctrl]
        if len(msgs):
            res, unz = OZ.h2_decompress(msgs, blob, buf, out_cap=64 << 20)
            for m, r in zip(msgs, res):
                self.calls += 1; self.compressed_calls += bool(m["flags"] & 4)
                ok = (m["flags"] & 3) == 3 and m["method_idx"] >= 0 and r["status"] in (NONE, OK)
                if not ok:
                    body = b""
                elif r["status"] == OK:
                    body = unz[r["out_off"]:r["out_off"] + r["out_len"]]
                else:
                    body = bytes(blob[m["msg_off"]:m["msg_off"] + m["msg_len"]])
                out.append(c.pack_response(int(m["stream_id"]), body, grpc_status=0 if ok else 12, grpc_message=b"" if ok else b"unimplemented"))
        return cons, b"".join(out), err, len(msgs)
