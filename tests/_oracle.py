"""ctypes binding of oracle/liboracle.so (CPU ORACLE — tests only)."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = C.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))


class Span(C.Structure):
    _fields_ = [("off", C.c_uint32), ("len", C.c_uint32)]


class RpcMeta(C.Structure):
    _fields_ = [("has", C.c_uint32),
                ("has_service_name", C.c_int), ("has_method_name", C.c_int),
                ("service_name", Span), ("method_name", Span), ("request_id", Span),
                ("log_id", C.c_int64), ("trace_id", C.c_int64), ("span_id", C.c_int64), ("parent_span_id", C.c_int64),
                ("has_span_id", C.c_int), ("has_parent_span_id", C.c_int),
                ("timeout_ms", C.c_int32),
                ("has_error_code", C.c_int), ("has_error_text", C.c_int),
                ("error_code", C.c_int32), ("error_text", Span),
                ("compress_type", C.c_int32), ("correlation_id", C.c_int64), ("attachment_size", C.c_int32),
                ("chunk_has_stream_id", C.c_int), ("chunk_has_chunk_id", C.c_int),
                ("authentication_data", Span),
                ("ss_has_stream_id", C.c_int), ("ss_stream_id", C.c_int64),
                ("ss_need_feedback", C.c_int), ("ss_writable", C.c_int),
                ("ss_n_extra", C.c_uint32), ("n_user_fields", C.c_uint32),
                ("content_type", C.c_int32), ("checksum_type", C.c_int32), ("checksum_value", Span)]


class StreamMeta(C.Structure):
    _fields_ = [("has", C.c_uint32), ("stream_id", C.c_int64), ("source_stream_id", C.c_int64),
                ("consumed_size", C.c_int64), ("frame_type", C.c_int32), ("feedback_has_consumed_size", C.c_int)]


class Method(C.Structure):
    _fields_ = [("service_full_name", C.c_char_p), ("service_name", C.c_char_p), ("method_name", C.c_char_p),
                ("request_type_name", C.c_char_p), ("handler", C.c_int32), ("echo_attachment", C.c_int32),
                ("response_checksum_type", C.c_int32), ("response_compress_type", C.c_int32)]


class Config(C.Structure):
    _fields_ = [("max_body_size", C.c_uint64), ("server_identity", C.c_char_p),
                ("methods", C.POINTER(Method)), ("n_methods", C.c_uint32), ("stream_handler", C.c_int), ("protocols", C.c_uint32)]


class RequestSpec(C.Structure):
    _fields_ = [("service_name", C.c_char_p), ("method_name", C.c_char_p),
                ("has_log_id", C.c_int), ("log_id", C.c_int64), ("correlation_id", C.c_int64),
                ("compress_type", C.c_int32), ("checksum_type", C.c_int32), ("content_type", C.c_int32),
                ("message", C.c_char_p), ("message_len", C.c_uint32),
                ("attachment", C.c_char_p), ("attachment_len", C.c_uint32),
                ("has_trace", C.c_int), ("trace_id", C.c_int64), ("span_id", C.c_int64), ("parent_span_id", C.c_int64),
                ("request_id", C.c_char_p), ("timeout_ms", C.c_int32)]


RUN_DT = np.dtype([("socket_id", "<u8"), ("offset", "<u4"), ("length", "<u4"),
                   ("preferred_proto", "<i4"), ("flags", "<u4")])
RUN_STATUS_DT = np.dtype([("consumed", "<u4"), ("parse_error", "<u4"), ("n_msgs", "<u4"), ("first_msg", "<u4"),
                          ("preferred_proto", "<i4"), ("n_unanswered", "<u4"), ("resp_off", "<u4"), ("resp_bytes", "<u4")])
MSG_DT = np.dtype([("run_idx", "<u4"), ("frame_off", "<u4"), ("body_size", "<u4"), ("meta_size", "<u4"),
                   ("correlation_id", "<i8"), ("log_id", "<i8"),
                   ("attachment_size", "<i4"), ("compress_type", "<i4"), ("checksum_type", "<i4"), ("error_code", "<i4"),
                   ("has_bits", "<u2"), ("protocol", "u1"), ("content_type", "u1"),
                   ("method_idx", "<i2"), ("status", "<u2"), ("resp_off", "<u4"), ("resp_len", "<u4")])
assert RUN_DT.itemsize == 24 and RUN_STATUS_DT.itemsize == 32 and MSG_DT.itemsize == 64

lib.orc_crc32c_extend.restype = C.c_uint32
lib.orc_crc32c_extend.argtypes = [C.c_uint32, C.c_char_p, C.c_size_t]
lib.orc_crc32c_mask.restype = C.c_uint32; lib.orc_crc32c_mask.argtypes = [C.c_uint32]
lib.orc_crc32c_unmask.restype = C.c_uint32; lib.orc_crc32c_unmask.argtypes = [C.c_uint32]
lib.orc_parse_rpc_meta.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(RpcMeta)]
lib.orc_parse_stream_meta.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(StreamMeta)]
lib.orc_parse_echo_request.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(Span)]
lib.orc_pack_echo_request.restype = C.c_size_t
lib.orc_pack_echo_request.argtypes = [C.POINTER(RequestSpec), C.c_void_p, C.c_size_t]
lib.orc_pack_stream_frame.restype = C.c_size_t
lib.orc_pack_stream_frame.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_void_p, C.c_size_t]
lib.orc_process_batch.argtypes = [C.POINTER(Config), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p,
                                  C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
lib.orc_snappy_max_compressed_length.restype = C.c_size_t; lib.orc_snappy_max_compressed_length.argtypes = [C.c_size_t]
lib.orc_snappy_compress.restype = C.c_size_t; lib.orc_snappy_compress.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p]
lib.orc_snappy_uncompressed_length.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
lib.orc_snappy_uncompress.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]


lib.orc_gzip_input_stream.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
lib.orc_free.argtypes = [C.c_void_p]


lib.orc_pack_response.restype = C.c_size_t
lib.orc_pack_response.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t]


def pack_response(reply, data):
    """reply: one REPLY_DT record (numpy, offsets into data).  The frame SendRpcResponse writes; b"" = not packable."""
    import numpy as np
    r = np.ascontiguousarray(reply).reshape(1)
    cap = int(r["body_len"][0]) * 2 + len(data) + 4096
    out = C.create_string_buffer(cap)
    n = lib.orc_pack_response(r.ctypes.data, bytes(data), out, cap)
    assert n != (1 << 64) - 1
    return out.raw[:n]


def gzip_input_stream(b, fmt):
    """What GzipInputStream(fmt = 2 gzip | 3 zlib) hands to the parser for the body `b` (oracle/b2_oracle_gzip.c)."""
    out = C.c_void_p(); n = C.c_size_t()
    assert lib.orc_gzip_input_stream(bytes(b), len(b), fmt, C.byref(out), C.byref(n)) == 0
    r = C.string_at(out, n.value)
    lib.orc_free(out)
    return r


def snappy_compress(b):
    """RawCompress of the reference's snappy 1.1.3 (the oracle's restatement, pinned by tests/golden/snappy_vectors.json)."""
    out = C.create_string_buffer(lib.orc_snappy_max_compressed_length(len(b)))
    n = lib.orc_snappy_compress(bytes(b), len(b), out)
    return out.raw[:n]


def snappy_uncompressed_length(b):
    """GetUncompressedLength: the announced length, or None when the preamble is malformed."""
    n = C.c_size_t()
    return n.value if lib.orc_snappy_uncompressed_length(bytes(b), len(b), C.byref(n)) else None


def snappy_uncompress(b, cap):
    """RawUncompress: the bytes, or None when the stream is invalid or announces more than cap bytes."""
    out = C.create_string_buffer(max(1, cap)); got = C.c_size_t()
    return out.raw[:got.value] if lib.orc_snappy_uncompress(bytes(b), len(b), out, cap, C.byref(got)) else None


def crc32c(b, init=0):
    return lib.orc_crc32c_extend(init, bytes(b), len(b))


def parse_rpc_meta(b):
    m = RpcMeta()
    ok = lib.orc_parse_rpc_meta(bytes(b), len(b), C.byref(m))
    return bool(ok), m


def parse_stream_meta(b):
    m = StreamMeta()
    ok = lib.orc_parse_stream_meta(bytes(b), len(b), C.byref(m))
    return bool(ok), m


def parse_echo_request(b):
    s = Span()
    ok = lib.orc_parse_echo_request(bytes(b), len(b), C.byref(s))
    return bool(ok), (s.off, s.len)


def pack_echo_request(service=b"example.EchoService", method=b"Echo", log_id=None, correlation_id=0,
                      compress_type=0, checksum_type=0, content_type=0, message=b"", attachment=b"",
                      trace=None, request_id=None, timeout_ms=0):
    s = RequestSpec()
    s.service_name, s.method_name = service, method
    s.has_log_id, s.log_id = (0, 0) if log_id is None else (1, log_id)
    s.correlation_id = correlation_id
    s.compress_type, s.checksum_type, s.content_type = compress_type, checksum_type, content_type
    s.message, s.message_len = message, len(message)
    s.attachment, s.attachment_len = attachment, len(attachment)
    if trace:
        s.has_trace, s.trace_id, s.span_id, s.parent_span_id = 1, trace[0], trace[1], trace[2]
    s.request_id = request_id
    s.timeout_ms = timeout_ms
    cap = 2048 + len(message) + len(message) // 5 + len(attachment)
    buf = C.create_string_buffer(cap)
    n = lib.orc_pack_echo_request(C.byref(s), buf, cap)
    assert n > 0, "orc_pack_echo_request failed"
    return buf.raw[:n]


def pack_stream_frame(stream_id, source_stream_id=-1, frame_type=3, has_continuation=None, data=b""):
    cap = 128 + len(data)
    buf = C.create_string_buffer(cap)
    n = lib.orc_pack_stream_frame(stream_id, source_stream_id, frame_type,
                                  0 if has_continuation is None else 1, 1 if has_continuation else 0,
                                  data, len(data), buf, cap)
    assert n > 0
    return buf.raw[:n]


ECHO_METHOD = dict(service_full_name=b"example.EchoService", service_name=b"EchoService", method_name=b"Echo",
                   request_type_name=b"example.EchoRequest", handler=1, echo_attachment=1,
                   response_checksum_type=0, response_compress_type=0)


def make_config(methods=None, max_body_size=0, server_identity=None, stream_handler=0, protocols=0):
    methods = [ECHO_METHOD] if methods is None else methods
    arr = (Method * max(1, len(methods)))()
    for i, m in enumerate(methods):
        for k, v in m.items():
            setattr(arr[i], k, v)
    cfg = Config(max_body_size, server_identity, arr, len(methods), stream_handler, protocols)
    cfg._keep = arr
    return cfg


def process_batch(cfg, data, runs, msg_cap=None, resp_cap=None):
    """data: bytes/np.uint8 array; runs: np array RUN_DT.  Returns (run_status, msgs, resp)."""
    data = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
    runs = np.ascontiguousarray(runs)
    n_runs = len(runs)
    msg_cap = msg_cap or (len(data) // 12 + 16)
    resp_cap = resp_cap or (len(data) * 2 + 4096 * max(1, msg_cap // 8) + (1 << 16))
    rs = np.zeros(n_runs, dtype=RUN_STATUS_DT)
    msgs = np.zeros(msg_cap, dtype=MSG_DT)
    resp = np.zeros(resp_cap, dtype=np.uint8)
    nm, rb = C.c_uint32(0), C.c_uint32(0)
    rc = lib.orc_process_batch(C.byref(cfg), data.ctypes.data, len(data), runs.ctypes.data, n_runs, rs.ctypes.data,
                               msgs.ctypes.data, msg_cap, C.byref(nm), resp.ctypes.data, resp_cap, C.byref(rb))
    assert rc == 0, "oracle capacity exceeded"
    return rs, msgs[:nm.value], resp[:rb.value]


# ---- HPACK / h2 (a15) ----
H2_FRAME_DT = np.dtype([("type", "u1"), ("flags", "u1"), ("pad", "<u2"), ("stream_id", "<u4"), ("payload_off", "<u4"), ("payload_len", "<u4")])
lib.orc_hpack_new.restype = C.c_void_p; lib.orc_hpack_new.argtypes = [C.c_uint32]
lib.orc_hpack_free.argtypes = [C.c_void_p]
lib.orc_hpack_decode_block.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
lib.orc_h2_scan.restype = C.c_uint32
lib.orc_h2_scan.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]


def parse_header_records(buf):
    out, o = [], 0
    while o < len(buf):
        nl = buf[o] | (buf[o + 1] << 8); vl = buf[o + 2] | (buf[o + 3] << 8)
        out.append((bytes(buf[o + 4:o + 4 + nl]), bytes(buf[o + 4 + nl:o + 4 + nl + vl]))); o += 4 + nl + vl
    return out


class HPack:
    def __init__(self, max_table_size=4096):
        self.h = lib.orc_hpack_new(max_table_size)

    def decode_block(self, b):
        cap = 1 << 20
        out = C.create_string_buffer(cap); ol, nh = C.c_uint32(), C.c_uint32()
        st = lib.orc_hpack_decode_block(self.h, bytes(b), len(b), out, cap, C.byref(ol), C.byref(nh))
        return st, parse_header_records(out.raw[:ol.value])

    def __del__(self):
        lib.orc_hpack_free(self.h)


def h2_scan(b, max_frame_size=16384):
    cap = len(b) // 9 + 2
    fr = np.zeros(cap, H2_FRAME_DT); consumed, err = C.c_uint32(), C.c_uint32()
    n = lib.orc_h2_scan(bytes(b), len(b), max_frame_size, fr.ctypes.data, cap, C.byref(consumed), C.byref(err))
    return fr[:n], consumed.value, err.value


# ---- h2 server-side parser (a15) ----
H2_MSG_DT = np.dtype([("run_idx", "<u4"), ("stream_id", "<u4"), ("headers_off", "<u4"), ("headers_len", "<u4"), ("n_headers", "<u4"),
                      ("body_off", "<u4"), ("body_len", "<u4"), ("http_method", "<u4"), ("content_type", "<u4"), ("flags", "<u4"),
                      ("method_idx", "<i4"), ("msg_off", "<u4"), ("msg_len", "<u4"), ("path_off", "<u4"), ("path_len", "<u4"), ("reserved", "<u4")])
H2_RESPONSE_DT = np.dtype([("conn", "<u4"), ("stream_id", "<u4"), ("status_code", "<i4"), ("flags", "<u4"), ("content_type_off", "<u4"),
                           ("content_type_len", "<u4"), ("body_off", "<u4"), ("body_len", "<u4"), ("grpc_status", "<i4"),
                           ("grpc_message_off", "<u4"), ("grpc_message_len", "<u4"), ("reserved", "<u4")])
lib.orc_h2_pack_response.restype = C.c_uint32
lib.orc_h2_pack_response.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p]
H2_REQUEST_DT = np.dtype([("conn", "<u4"), ("flags", "<u4"), ("path_off", "<u4"), ("path_len", "<u4"), ("authority_off", "<u4"),
                          ("authority_len", "<u4"), ("content_type_off", "<u4"), ("content_type_len", "<u4"), ("body_off", "<u4"),
                          ("body_len", "<u4"), ("extra_off", "<u4"), ("extra_len", "<u4")])          # == b2_h2_request, 48 bytes
lib.orc_h2_pack_request.restype = C.c_int32
lib.orc_h2_pack_request.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
lib.orc_h2_conn_set_next_stream_id.argtypes = [C.c_void_p, C.c_uint32]
lib.orc_h2_conn_peer_update.argtypes = [C.c_void_p, C.c_void_p]
H2_PEER_UPDATE_DT = np.dtype([("set", "<u4"), ("header_table_size", "<u4"), ("max_frame_size", "<u4"), ("stream_window_size", "<u4"), ("conn_window_add", "<i8")])
lib.orc_h2_conn_new.restype = C.c_void_p
lib.orc_h2_conn_free.argtypes = [C.c_void_p]
lib.orc_h2_consume.restype = C.c_uint32
lib.orc_h2_consume.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                               C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                               C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]


def h2_extra_records(extra):
    return b"".join(len(n).to_bytes(2, "little") + len(v).to_bytes(2, "little") + bytes(n) + bytes(v) for n, v in extra)


def h2_request_blob(calls):
    """calls: (conn, flags, path, authority, content_type, body, extra headers) -> (blob bytes, H2_REQUEST_DT array)."""
    parts = []; r = np.zeros(len(calls), H2_REQUEST_DT); at = 0
    for i, (conn, flags, path, authority, ct, body, extra) in enumerate(calls):
        ex = h2_extra_records(extra); offs = []
        for piece in (path, authority, ct, body, ex):
            offs.append(at); parts.append(bytes(piece)); at += len(piece)
        r[i] = (conn, flags, offs[0], len(path), offs[1], len(authority), offs[2], len(ct), offs[3], len(body), offs[4], len(ex))
    return b"".join(parts) + b"\0", r


class H2Conn:
    """One server-side H2Context of the oracle."""
    def __init__(self, cfg=None):
        self._h = lib.orc_h2_conn_new(); self.cfg = cfg or make_config()

    def consume(self, b):
        """Returns (parse_error, consumed, msgs, ctrl bytes, blob, remote_max_frame_size, remote_stream_window_size)."""
        b = bytes(b)
        msgs = np.zeros(256, H2_MSG_DT); ctrl = np.zeros(len(b) * 3 + 4096, np.uint8); blob = np.zeros(len(b) * 8 + (1 << 18), np.uint8)
        cons, nm, cl, bl, mfs, sws = (C.c_uint32() for _ in range(6))
        err = lib.orc_h2_consume(self._h, C.byref(self.cfg), b, len(b), C.byref(cons), msgs.ctypes.data, len(msgs), C.byref(nm),
                                 ctrl.ctypes.data, len(ctrl), C.byref(cl), blob.ctypes.data, len(blob), C.byref(bl), C.byref(mfs), C.byref(sws))
        assert nm.value <= len(msgs)
        return err, cons.value, msgs[:nm.value], ctrl[:cl.value].tobytes(), blob[:bl.value], mfs.value, sws.value

    def pack_response(self, stream_id, body=b"", status=200, content_type=b"application/grpc", grpc=True, grpc_status=0, grpc_message=b""):
        blob = bytes(content_type) + bytes(body) + bytes(grpc_message)
        r = np.zeros(1, H2_RESPONSE_DT)
        r[0] = (0, stream_id, status, 1 if grpc else 0, 0, len(content_type), len(content_type), len(body), grpc_status,
                len(content_type) + len(body), len(grpc_message), 0)
        out = np.zeros(len(body) * 2 + 4096, np.uint8)
        n = lib.orc_h2_pack_response(self._h, r.ctypes.data, blob, out.ctypes.data)
        return out[:n].tobytes()

    def pack_request(self, path, authority, body=b"", content_type=b"application/grpc", flags=1 | 8 | 16, extra=()):
        """Client side (H2UnsentRequest).  Returns (status, stream_id, bytes)."""
        blob, r = h2_request_blob([(0, flags, path, authority, content_type, body, extra)])
        out = np.zeros(len(body) * 2 + 8192, np.uint8); ol, sid = C.c_uint32(), C.c_uint32()
        st = lib.orc_h2_pack_request(self._h, r.ctypes.data, blob, out.ctypes.data, C.byref(ol), C.byref(sid))
        return st, sid.value, out[:ol.value].tobytes()

    def peer_update(self, header_table_size=None, max_frame_size=None, stream_window_size=None, conn_window_add=None):
        u = np.zeros(1, H2_PEER_UPDATE_DT)
        vals = (header_table_size, max_frame_size, stream_window_size, conn_window_add)
        u[0] = (sum(1 << i for i, v in enumerate(vals) if v is not None), *(0 if v is None else v for v in vals))
        return lib.orc_h2_conn_peer_update(self._h, u.ctypes.data)

    def set_next_stream_id(self, sid):
        lib.orc_h2_conn_set_next_stream_id(self._h, sid)

    def __del__(self):
        if self._h:
            lib.orc_h2_conn_free(self._h); self._h = None
