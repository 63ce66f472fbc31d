"""ctypes binding of include/b2rpc.h (brpc_b200/libb2rpc.so)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
lib_path = os.environ.get("B2RPC_LIB") or os.path.join(_HERE, "libb2rpc.so")      # (B2RPC_LIB: A/B builds of the same library for tuning runs)

B2_OK, B2_E_INVAL, B2_E_NO_DEVICE, B2_E_CUDA, B2_E_CAPACITY, B2_E_NOMEM = 0, -1, -2, -3, -4, -5

RUN_DT = np.dtype([("socket_id", "<u8"), ("offset", "<u4"), ("length", "<u4"),
                   ("preferred_proto", "<i4"), ("flags", "<u4")])
RUN_STATUS_DT = np.dtype([("consumed", "<u4"), ("parse_error", "<u4"), ("n_msgs", "<u4"), ("first_msg", "<u4"),
                          ("preferred_proto", "<i4"), ("n_unanswered", "<u4"), ("resp_off", "<u4"), ("resp_bytes", "<u4")])
H2_FRAME_DT = np.dtype([("type", "u1"), ("flags", "u1"), ("pad", "<u2"), ("stream_id", "<u4"), ("payload_off", "<u4"), ("payload_len", "<u4")])
HPACK_BLOCK_DT = np.dtype([("conn", "<u4"), ("offset", "<u4"), ("length", "<u4"), ("reserved", "<u4")])
H2_RUN_STATUS_DT = np.dtype([("consumed", "<u4"), ("parse_error", "<u4"), ("n_msgs", "<u4"), ("first_msg", "<u4"), ("ctrl_off", "<u4"), ("ctrl_len", "<u4"),
                             ("remote_max_frame_size", "<u4"), ("remote_stream_window_size", "<u4")])
REQUEST_DT = np.dtype([("kind", "<u4"), ("flags", "<u4"), ("method_idx", "<i4"), ("timeout_ms", "<i4"), ("correlation_id", "<i8"), ("log_id", "<i8"),
                       ("compress_type", "<i4"), ("checksum_type", "<i4"), ("frame_type", "<i4"), ("payload_off", "<u4"), ("payload_len", "<u4"),
                       ("attachment_off", "<u4"), ("attachment_len", "<u4"), ("reserved", "<u4")])
REPLY_DT = np.dtype([("flags", "<u4"), ("error_code", "<i4"), ("correlation_id", "<i8"), ("compress_type", "<i4"), ("checksum_type", "<i4"),
                     ("content_type", "<i4"), ("error_text_off", "<u4"), ("error_text_len", "<u4"), ("body_off", "<u4"), ("body_len", "<u4"),
                     ("attachment_off", "<u4"), ("attachment_len", "<u4"), ("checksum_value_off", "<u4"), ("checksum_value_len", "<u4"),
                     ("extra_streams_off", "<u4"), ("n_extra_streams", "<u4"), ("user_fields_off", "<u4"), ("n_user_fields", "<u4"),
                     ("reserved", "<u4"), ("stream_id", "<i8")])          # == b2_reply, 88 bytes
H2_RESPONSE_DT = np.dtype([("conn", "<u4"), ("stream_id", "<u4"), ("status_code", "<i4"), ("flags", "<u4"), ("content_type_off", "<u4"),
                           ("content_type_len", "<u4"), ("body_off", "<u4"), ("body_len", "<u4"), ("grpc_status", "<i4"),
                           ("grpc_message_off", "<u4"), ("grpc_message_len", "<u4"), ("reserved", "<u4")])
H2_REQUEST_DT = np.dtype([("conn", "<u4"), ("flags", "<u4"), ("path_off", "<u4"), ("path_len", "<u4"), ("authority_off", "<u4"),
                          ("authority_len", "<u4"), ("content_type_off", "<u4"), ("content_type_len", "<u4"), ("body_off", "<u4"),
                          ("body_len", "<u4"), ("extra_off", "<u4"), ("extra_len", "<u4")])          # == b2_h2_request, 48 bytes
H2_PEER_UPDATE_DT = np.dtype([("set", "<u4"), ("header_table_size", "<u4"), ("max_frame_size", "<u4"), ("stream_window_size", "<u4"), ("conn_window_add", "<i8")])
H2_REQUEST_RESULT_DT = np.dtype([("status", "<i4"), ("stream_id", "<u4"), ("out_off", "<u4"), ("out_len", "<u4")])
H2_UNZ_RESULT_DT = np.dtype([("status", "<u4"), ("out_off", "<u4"), ("out_len", "<u4"), ("reserved", "<u4")])        # == b2_h2_unz_result
H2_UNZ_NONE, H2_UNZ_OK, H2_UNZ_NO_ENCODING, H2_UNZ_NOT_GZIP, H2_UNZ_FAILED, H2_UNZ_HOST, H2_UNZ_NO_ROOM = range(7)
H2_MSG_DT = np.dtype([("run_idx", "<u4"), ("stream_id", "<u4"), ("headers_off", "<u4"), ("headers_len", "<u4"), ("n_headers", "<u4"),
                      ("body_off", "<u4"), ("body_len", "<u4"), ("http_method", "<u4"), ("content_type", "<u4"), ("flags", "<u4"),
                      ("method_idx", "<i4"), ("msg_off", "<u4"), ("msg_len", "<u4"), ("path_off", "<u4"), ("path_len", "<u4"), ("reserved", "<u4")])
MSG_DT = np.dtype([("run_idx", "<u4"), ("frame_off", "<u4"), ("body_size", "<u4"), ("meta_size", "<u4"),
                   ("correlation_id", "<i8"), ("log_id", "<i8"),
                   ("attachment_size", "<i4"), ("compress_type", "<i4"), ("checksum_type", "<i4"), ("error_code", "<i4"),
                   ("has_bits", "<u2"), ("protocol", "u1"), ("content_type", "u1"),
                   ("method_idx", "<i2"), ("status", "<u2"), ("resp_off", "<u4"), ("resp_len", "<u4")])
assert RUN_DT.itemsize == 24 and RUN_STATUS_DT.itemsize == 32 and MSG_DT.itemsize == 64


class Method(C.Structure):
    _fields_ = [("service_full_name", C.c_char_p), ("service_name", C.c_char_p), ("method_name", C.c_char_p),
                ("request_type_name", C.c_char_p), ("handler", C.c_int32), ("echo_attachment", C.c_int32),
                ("response_checksum_type", C.c_int32), ("response_compress_type", C.c_int32)]


class Options(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_batch_bytes", C.c_uint32), ("max_msgs", C.c_uint32),
                ("max_runs", C.c_uint32), ("max_resp_bytes", C.c_uint32), ("tile_bytes", C.c_uint32),
                ("max_body_size", C.c_uint64)]


class BatchResult(C.Structure):
    _fields_ = [("runs", C.c_void_p), ("n_runs", C.c_uint32),
                ("msgs", C.c_void_p), ("n_msgs", C.c_uint32),
                ("resp", C.c_void_p), ("resp_bytes", C.c_uint32),
                ("kernel_ms", C.c_float), ("n_launches", C.c_uint32), ("refs", C.c_void_p), ("iov", C.c_void_p)]


REF_DT = np.dtype([("prefix_len", "<u4"), ("src_off", "<u4"), ("src_len", "<u4"), ("reserved", "<u4")])
IOVEC_DT = np.dtype([("base", "<u8"), ("len", "<u8")])          # struct iovec
INPUT_COPY, INPUT_PULL, RESP_COPY, RESP_BY_REF, RESP_IOVEC = 0, 1, 0, 1, 2


class B2Error(RuntimeError):
    def __init__(self, code, text):
        super().__init__("b2rpc error %d: %s" % (code, text))
        self.code = code


def _load():
    if not os.path.exists(lib_path):
        raise ImportError("brpc_b200/libb2rpc.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a).  There is no CPU fallback.")
    l = C.CDLL(lib_path)
    l.b2_last_error.restype = C.c_char_p
    l.b2_version.restype = C.c_char_p
    l.b2_ctx_create.argtypes = [C.POINTER(Options), C.POINTER(C.c_void_p)]
    l.b2_ctx_destroy.argtypes = [C.c_void_p]
    l.b2_register_method.argtypes = [C.c_void_p, C.POINTER(Method)]
    l.b2_set_server_identity.argtypes = [C.c_void_p, C.c_char_p]
    l.b2_set_stream_handler.argtypes = [C.c_void_p, C.c_int]
    l.b2_set_protocols.argtypes = [C.c_void_p, C.c_uint32]
    l.b2_block_alloc.restype = C.c_void_p; l.b2_block_alloc.argtypes = [C.c_size_t]
    l.b2_block_free.argtypes = [C.c_void_p]
    l.b2_block_pool_host_allocs.restype = C.c_uint64
    l.b2_set_modes.argtypes = [C.c_void_p, C.c_int, C.c_int]
    l.b2_ring_start.argtypes = [C.c_void_p]; l.b2_ring_stop.argtypes = [C.c_void_p]
    l.b2_ring_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
    l.b2_ring_wait.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(BatchResult)]
    l.b2_ring_launches.restype = C.c_uint64; l.b2_ring_launches.argtypes = [C.c_void_p]
    l.b2_ring_phase_ns.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    l.b2_latency_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    l.b2_process_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(BatchResult)]
    l.b2_batch_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
    l.b2_batch_collect.argtypes = [C.c_void_p, C.POINTER(BatchResult)]
    l.b2_batch_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32]
    l.b2_batch_execute.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]
    l.b2_batch_execute_many.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_uint32)]
    l.b2_batch_launch.argtypes = [C.c_void_p]
    l.b2_batch_wait.argtypes = [C.c_void_p]
    l.b2_elapsed_ms.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
    l.b2_batch_download.argtypes = [C.c_void_p, C.POINTER(BatchResult)]
    l.b2_batch_info.argtypes = [C.c_void_p, C.c_void_p]
    l.b2_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
    l.b2_stage_times.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.c_int]
    l.b2_crc32c_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    l.b2_snappy_uncompress_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                             C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    l.b2_snappy_compress_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                           C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    l.b2_crc32c_extend.restype = C.c_uint32; l.b2_crc32c_extend.argtypes = [C.c_uint32, C.c_char_p, C.c_size_t]
    l.b2_snappy_max_compressed_length.restype = C.c_size_t; l.b2_snappy_max_compressed_length.argtypes = [C.c_size_t]
    l.b2_snappy_raw_compress.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_size_t)]
    l.b2_snappy_get_uncompressed_length.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
    l.b2_snappy_raw_uncompress.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p]
    l.b2_hpack_reset.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    l.b2_hpack_decode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
    l.b2_h2_scan_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    l.b2_h2_conn_reset.argtypes = [C.c_void_p, C.c_uint32]
    l.b2_h2_configure.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
    l.b2_h2_process_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                      C.POINTER(C.c_uint32), C.c_void_p, C.c_uint32]
    l.b2_h2_pack_requests.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]
    l.b2_h2_conn_set_next_stream_id.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    l.b2_h2_conn_peer_update.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    l.b2_h2_pack_responses.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    l.b2_h2_decompress_requests.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]
    l.b2_pack_requests.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    l.b2_pack_responses.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    l.b2_counters_read.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    l.b2_counters_device_ptr.restype = C.c_void_p; l.b2_counters_device_ptr.argtypes = [C.c_void_p]
    return l


lib = _load()

# every symbol include/b2rpc.h declares (tests check the library exports them)
ABI_SYMBOLS = ["b2_ctx_create", "b2_ctx_destroy", "b2_last_error", "b2_version", "b2_register_method",
               "b2_set_server_identity", "b2_set_stream_handler", "b2_set_protocols", "b2_block_alloc", "b2_block_free", "b2_block_pool_host_allocs", "b2_set_modes", "b2_ring_start", "b2_ring_stop", "b2_ring_submit", "b2_ring_wait", "b2_ring_launches", "b2_ring_phase_ns", "b2_latency_probe", "b2_process_batch", "b2_batch_submit", "b2_batch_collect", "b2_batch_upload",
               "b2_batch_execute", "b2_batch_execute_many", "b2_batch_download", "b2_batch_launch", "b2_batch_wait",
               "b2_elapsed_ms", "b2_batch_info", "b2_device_pci_bus_id", "b2_stage_times", "b2_crc32c_batch", "b2_crc32c_extend", "b2_snappy_max_compressed_length", "b2_snappy_raw_compress", "b2_snappy_get_uncompressed_length", "b2_snappy_raw_uncompress", "b2_snappy_uncompress_batch", "b2_snappy_compress_batch", "b2_hpack_reset", "b2_hpack_decode_batch", "b2_pack_requests", "b2_pack_responses", "b2_h2_scan_batch", "b2_h2_conn_reset", "b2_h2_configure", "b2_h2_process_batch", "b2_h2_pack_responses", "b2_counters_read",
               "b2_counters_device_ptr", "b2_counters_allreduce", "b2_h2_pack_requests", "b2_h2_conn_set_next_stream_id", "b2_h2_conn_peer_update",
               "b2_h2_decompress_requests"]

ECHO_METHOD = dict(service_full_name=b"example.EchoService", service_name=b"EchoService", method_name=b"Echo",
                   request_type_name=b"example.EchoRequest", handler=1, echo_attachment=1,
                   response_checksum_type=0, response_compress_type=0)


def _check(rc):
    if rc < 0:
        raise B2Error(rc, (lib.b2_last_error() or b"").decode("utf-8", "replace"))
    return rc


class PinnedBuffer:
    """Host memory from b2_block_alloc (cudaHostAlloc), viewed as a numpy uint8 array."""

    def __init__(self, nbytes):
        self.ptr = lib.b2_block_alloc(nbytes)
        if not self.ptr:
            raise B2Error(B2_E_NOMEM, "b2_block_alloc failed")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            lib.b2_block_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """b2_ctx: one per GPU."""

    def __init__(self, device=0, max_batch_bytes=64 << 20, max_msgs=1 << 20, max_runs=4096, max_resp_bytes=0,
                 tile_bytes=0, max_body_size=0, methods=(ECHO_METHOD,), server_identity=None, stream_handler=0):
        opt = Options(device, max_batch_bytes, max_msgs, max_runs, max_resp_bytes, tile_bytes, max_body_size)
        h = C.c_void_p()
        _check(lib.b2_ctx_create(C.byref(opt), C.byref(h)))
        self._h = h
        self._keep = []
        for m in methods:
            self.register_method(**m)
        if server_identity:
            _check(lib.b2_set_server_identity(self._h, server_identity))
        if stream_handler:
            _check(lib.b2_set_stream_handler(self._h, stream_handler))

    def close(self):
        if getattr(self, "_h", None):
            lib.b2_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def register_method(self, **kw):
        m = Method(**kw)
        self._keep.append(m)
        return _check(lib.b2_register_method(self._h, C.byref(m)))

    @staticmethod
    def _views(res):
        runs = np.ctypeslib.as_array((C.c_uint8 * (32 * res.n_runs)).from_address(res.runs)).view(RUN_STATUS_DT) \
            if res.n_runs else np.zeros(0, RUN_STATUS_DT)
        msgs = np.ctypeslib.as_array((C.c_uint8 * (64 * res.n_msgs)).from_address(res.msgs)).view(MSG_DT) \
            if res.n_msgs else np.zeros(0, MSG_DT)
        resp = np.ctypeslib.as_array((C.c_uint8 * res.resp_bytes).from_address(res.resp)) \
            if res.resp_bytes else np.zeros(0, np.uint8)
        return runs, msgs, resp

    @staticmethod
    def _info(res):
        refs = None
        if res.refs and res.n_msgs:
            refs = np.ctypeslib.as_array((C.c_uint8 * (16 * res.n_msgs)).from_address(res.refs)).view(REF_DT)
        iov = None
        if res.iov and res.n_msgs:
            iov = np.ctypeslib.as_array((C.c_uint8 * (32 * res.n_msgs)).from_address(res.iov)).view(IOVEC_DT)
        return {"kernel_ms": res.kernel_ms, "n_launches": res.n_launches, "refs": refs, "iov": iov}

    # ---- the persistent latency kernel (b2_ring_*) ----
    def ring_start(self):
        _check(lib.b2_ring_start(self._h))

    def ring_stop(self):
        _check(lib.b2_ring_stop(self._h))

    def ring_submit(self, data, runs, ptr=None, nbytes=None):
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        if ptr is None:
            data = np.ascontiguousarray(data, dtype=np.uint8); ptr, nbytes = data.ctypes.data, data.nbytes
            self._ring_keep = data
        t = C.c_uint32(0)
        _check(lib.b2_ring_submit(self._h, ptr, nbytes, runs.ctypes.data, len(runs), C.byref(t)))
        return t.value

    def ring_wait(self, ticket):
        res = BatchResult()
        _check(lib.b2_ring_wait(self._h, ticket, C.byref(res)))
        rs, msgs, resp = self._views(res)
        return rs, msgs, resp, self._info(res)

    def latency_probe(self, ptr, nbytes, runs, iters, use_ring):
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        us = np.zeros(iters, np.float32)
        _check(lib.b2_latency_probe(self._h, ptr, nbytes, runs.ctypes.data, len(runs), iters, 1 if use_ring else 0, us.ctypes.data))
        return us

    def ring_phase_ns(self, ticket):
        out = (C.c_uint64 * 4)()
        _check(lib.b2_ring_phase_ns(self._h, ticket, out))
        return list(out)

    def ring_launches(self):
        return int(lib.b2_ring_launches(self._h))

    def set_protocols(self, mask):
        _check(lib.b2_set_protocols(self._h, mask))

    def set_modes(self, input_mode=INPUT_COPY, resp_mode=RESP_COPY):
        _check(lib.b2_set_modes(self._h, input_mode, resp_mode))

    def process_batch(self, data, runs):
        """Host buffers in, host (pinned) views out: (run_status, msgs, resp, info)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        res = BatchResult()
        _check(lib.b2_process_batch(self._h, data.ctypes.data, data.nbytes, runs.ctypes.data, len(runs), C.byref(res)))
        rs, msgs, resp = self._views(res)
        return rs, msgs, resp, self._info(res)

    def upload(self, data, runs):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        _check(lib.b2_batch_upload(self._h, data.ctypes.data, data.nbytes, runs.ctypes.data, len(runs)))

    def upload_ptr(self, ptr, nbytes, runs):
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        _check(lib.b2_batch_upload(self._h, ptr, nbytes, runs.ctypes.data, len(runs)))

    def execute(self):
        ms, n = C.c_float(0), C.c_uint32(0)
        _check(lib.b2_batch_execute(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def execute_many(self, steps):
        ms, n = C.c_float(0), C.c_uint32(0)
        _check(lib.b2_batch_execute_many(self._h, steps, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def launch(self):
        _check(lib.b2_batch_launch(self._h))

    def wait(self):
        _check(lib.b2_batch_wait(self._h))

    def elapsed_ms_to(self, other):
        ms = C.c_float(0)
        _check(lib.b2_elapsed_ms(self._h, other._h, C.byref(ms)))
        return ms.value

    def download(self):
        res = BatchResult()
        _check(lib.b2_batch_download(self._h, C.byref(res)))
        rs, msgs, resp = self._views(res)
        return rs, msgs, resp, self._info(res)

    def process_batch_ptr(self, ptr, nbytes, runs):
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        res = BatchResult()
        _check(lib.b2_process_batch(self._h, ptr, nbytes, runs.ctypes.data, len(runs), C.byref(res)))
        rs, msgs, resp = self._views(res)
        return rs, msgs, resp, self._info(res)

    def submit_ptr(self, ptr, nbytes, runs):
        runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        self._submitted_runs = runs           # keep alive until collect
        _check(lib.b2_batch_submit(self._h, ptr, nbytes, runs.ctypes.data, len(runs)))

    def collect(self):
        res = BatchResult()
        _check(lib.b2_batch_collect(self._h, C.byref(res)))
        rs, msgs, resp = self._views(res)
        return rs, msgs, resp, self._info(res)

    def batch_info(self):
        out = (C.c_uint32 * 4)()
        _check(lib.b2_batch_info(self._h, out))
        return {"tile_bytes": out[0], "n_tiles": out[1], "spec_k": out[2], "fused": bool(out[3])}

    def stage_times(self):
        names = (C.c_char_p * 16)()
        ms = (C.c_float * 16)()
        n = lib.b2_stage_times(self._h, names, ms, 16)
        return [(names[i].decode(), ms[i]) for i in range(max(0, min(n, 16)))]

    def crc32c_batch(self, data, offs, lens):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint32)
        lens = np.ascontiguousarray(lens, dtype=np.uint32)
        out = np.zeros(len(offs), dtype=np.uint32)
        _check(lib.b2_crc32c_batch(self._h, data.ctypes.data, data.nbytes, offs.ctypes.data, lens.ctypes.data,
                                   len(offs), out.ctypes.data))
        return out

    def snappy_uncompress_batch(self, data, offs, lens, out_cap):
        """Returns (list of bytes or None) for each slice."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint32); lens = np.ascontiguousarray(lens, dtype=np.uint32)
        n = len(offs)
        out = np.zeros(out_cap, dtype=np.uint8); ooffs = np.zeros(n, dtype=np.uint32); olens = np.zeros(n, dtype=np.int32)
        _check(lib.b2_snappy_uncompress_batch(self._h, data.ctypes.data, data.nbytes, offs.ctypes.data, lens.ctypes.data, n,
                                              out.ctypes.data, out_cap, ooffs.ctypes.data, olens.ctypes.data))
        return [None if olens[i] < 0 else out[ooffs[i]:ooffs[i] + olens[i]].tobytes() for i in range(n)]

    def snappy_compress_batch(self, data, offs, lens, out_cap):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint32); lens = np.ascontiguousarray(lens, dtype=np.uint32)
        n = len(offs)
        out = np.zeros(out_cap, dtype=np.uint8); ooffs = np.zeros(n, dtype=np.uint32); olens = np.zeros(n, dtype=np.uint32)
        _check(lib.b2_snappy_compress_batch(self._h, data.ctypes.data, data.nbytes, offs.ctypes.data, lens.ctypes.data, n,
                                            out.ctypes.data, out_cap, ooffs.ctypes.data, olens.ctypes.data))
        return [out[ooffs[i]:ooffs[i] + olens[i]].tobytes() for i in range(n)]

    def hpack_reset(self, conn, max_table_size=4096):
        _check(lib.b2_hpack_reset(self._h, conn, max_table_size))

    def hpack_decode_batch(self, data, blocks, per_block_cap=4096):
        """blocks: list of (conn, offset, length).  Returns [(status, [(name, value), ...]), ...]."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        b = np.zeros(len(blocks), HPACK_BLOCK_DT)
        for i, (c, o, n) in enumerate(blocks):
            b[i] = (c, o, n, 0)
        n = len(blocks)
        out = np.zeros(max(1, n * per_block_cap), np.uint8); ol = np.zeros(n, np.uint32); st = np.zeros(n, np.int32); nh = np.zeros(n, np.uint32)
        _check(lib.b2_hpack_decode_batch(self._h, data.ctypes.data, data.nbytes, b.ctypes.data, n, out.ctypes.data, per_block_cap,
                                         ol.ctypes.data, st.ctypes.data, nh.ctypes.data))
        res = []
        for i in range(n):
            buf = out[i * per_block_cap:i * per_block_cap + ol[i]]; o = 0; hs = []
            while o < len(buf):
                nl = int(buf[o]) | (int(buf[o + 1]) << 8); vl = int(buf[o + 2]) | (int(buf[o + 3]) << 8)
                hs.append((buf[o + 4:o + 4 + nl].tobytes(), buf[o + 4 + nl:o + 4 + nl + vl].tobytes())); o += 4 + nl + vl
            assert len(hs) == nh[i]
            res.append((int(st[i]), hs))
        return res

    def h2_scan_batch(self, data, runs, max_frame_size=16384, cap_per_run=256):
        data = np.ascontiguousarray(data, dtype=np.uint8); runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        n = len(runs)
        frames = np.zeros(max(1, n * cap_per_run), H2_FRAME_DT); nf = np.zeros(n, np.uint32); cons = np.zeros(n, np.uint32); err = np.zeros(n, np.uint32)
        _check(lib.b2_h2_scan_batch(self._h, data.ctypes.data, data.nbytes, runs.ctypes.data, n, max_frame_size, frames.ctypes.data, cap_per_run,
                                    nf.ctypes.data, cons.ctypes.data, err.ctypes.data))
        return [frames[i * cap_per_run:i * cap_per_run + min(int(nf[i]), cap_per_run)] for i in range(n)], nf, cons, err

    def h2_configure(self, max_conns=1024, max_pending=8, stream_bytes=69632):
        _check(lib.b2_h2_configure(self._h, max_conns, max_pending, stream_bytes))

    def h2_conn_reset(self, conn):
        _check(lib.b2_h2_conn_reset(self._h, conn))

    def h2_process_batch(self, data, runs, msg_cap=None, out_cap=None, out=None):
        """runs[i].socket_id = h2 connection index.  Returns (run_status, msgs, out)."""
        data = np.ascontiguousarray(data, dtype=np.uint8); runs = np.ascontiguousarray(runs, dtype=RUN_DT)
        n = len(runs)
        msg_cap = msg_cap or max(64, 64 * n)
        out_cap = out_cap or max(1 << 16, n * (1 << 17))
        rs = np.zeros(n, H2_RUN_STATUS_DT); msgs = np.zeros(msg_cap, H2_MSG_DT); nm = C.c_uint32(0)
        if out is None:
            out = np.empty(out_cap, np.uint8)       # (pass a PinnedBuffer's array to keep the copies off pageable memory)
        out_cap = out.nbytes
        _check(lib.b2_h2_process_batch(self._h, data.ctypes.data, data.nbytes, runs.ctypes.data, n, rs.ctypes.data, msgs.ctypes.data, msg_cap,
                                       C.byref(nm), out.ctypes.data, out_cap))
        return rs, msgs[:nm.value], out

    def h2_pack_responses(self, data, resps, out_cap=None, raw=False, out=None):
        """resps: H2_RESPONSE_DT array (offsets into data).  Returns the packed bytes of every response."""
        resps = np.ascontiguousarray(resps, dtype=H2_RESPONSE_DT)
        n = len(resps)
        out_cap = out_cap or int(resps["body_len"].astype(np.int64).sum() * 2 + n * 2048 + 4096)
        offs = np.zeros(n, np.uint32); lens = np.zeros(n, np.uint32)
        if out is None:
            out = np.empty(out_cap, np.uint8)
        out_cap = out.nbytes
        if data is None:                 # every field uses a zero-copy source (B2_H2_RESP_*_IN_INPUT / _IN_OUT)
            ptr, nb = None, 0
        else:
            data = np.ascontiguousarray(data, dtype=np.uint8); ptr, nb = data.ctypes.data, data.nbytes
        _check(lib.b2_h2_pack_responses(self._h, ptr, nb, resps.ctypes.data, n, out.ctypes.data, out_cap, offs.ctypes.data, lens.ctypes.data))
        if raw:
            return out, offs, lens
        return [out[offs[i]:offs[i] + lens[i]].tobytes() for i in range(n)]

    def h2_decompress_requests(self, msgs, out_cap=None, out=None):
        """GzipDecompress of ProcessHttpRequest for messages of the last h2_process_batch (its H2_MSG_DT records, in the order to
        serve them).  Returns (H2_UNZ_RESULT_DT per message, out): an inflated message is out[out_off:out_off + out_len]."""
        msgs = np.ascontiguousarray(msgs, dtype=H2_MSG_DT)
        n = len(msgs)
        if out is None:
            out = np.empty(out_cap or (4 << 20), np.uint8)
        res = np.zeros(n, H2_UNZ_RESULT_DT)
        _check(lib.b2_h2_decompress_requests(self._h, msgs.ctypes.data, n, out.ctypes.data, out.nbytes, res.ctypes.data))
        return res, out

    def h2_pack_requests(self, data, reqs, out_cap=None):
        """Client side of h2 (H2UnsentRequest): reqs is an H2_REQUEST_DT array (offsets into data).  Returns (results, [bytes per request])."""
        data = np.ascontiguousarray(data, dtype=np.uint8); reqs = np.ascontiguousarray(reqs, dtype=H2_REQUEST_DT)
        n = len(reqs)
        out_cap = out_cap or int(reqs["body_len"].astype(np.int64).sum() * 2 + n * 8192 + 4096)
        res = np.zeros(n, H2_REQUEST_RESULT_DT); out = np.empty(out_cap, np.uint8)
        _check(lib.b2_h2_pack_requests(self._h, data.ctypes.data, data.nbytes, reqs.ctypes.data, n, out.ctypes.data, out_cap, res.ctypes.data))
        return res, [out[r["out_off"]:r["out_off"] + r["out_len"]].tobytes() for r in res]

    def h2_conn_peer_update(self, conn, header_table_size=None, max_frame_size=None, stream_window_size=None, conn_window_add=None):
        """The peer's SETTINGS / connection WINDOW_UPDATE, parsed by the host, mirrored into the device's connection state."""
        u = np.zeros(1, H2_PEER_UPDATE_DT)
        vals = (header_table_size, max_frame_size, stream_window_size, conn_window_add)
        u[0] = (sum(1 << i for i, v in enumerate(vals) if v is not None), *(0 if v is None else v for v in vals))
        _check(lib.b2_h2_conn_peer_update(self._h, conn, u.ctypes.data))

    def h2_conn_set_next_stream_id(self, conn, next_id):
        _check(lib.b2_h2_conn_set_next_stream_id(self._h, conn, next_id))

    def pack_requests(self, data, reqs, out_cap=None):
        """reqs: REQUEST_DT array (offsets into data).  Returns the packed frame of every request (b"" = rejected)."""
        data = np.ascontiguousarray(data, dtype=np.uint8); reqs = np.ascontiguousarray(reqs, dtype=REQUEST_DT)
        n = len(reqs)
        out_cap = out_cap or int((reqs["payload_len"].astype(np.int64) * 7 // 6 + reqs["attachment_len"] + 640).sum() + 4096)
        out = np.empty(out_cap, np.uint8); offs = np.zeros(n, np.uint32); lens = np.zeros(n, np.uint32)
        _check(lib.b2_pack_requests(self._h, data.ctypes.data, data.nbytes, reqs.ctypes.data, n, out.ctypes.data, out_cap, offs.ctypes.data, lens.ctypes.data))
        return [out[offs[i]:offs[i] + lens[i]].tobytes() for i in range(n)]

    def pack_responses(self, data, replies, out_cap=None):
        """replies: REPLY_DT array (offsets into data).  Returns the frame of every reply (b"" = not packable)."""
        data = np.ascontiguousarray(data, dtype=np.uint8); replies = np.ascontiguousarray(replies, dtype=REPLY_DT)
        n = len(replies)
        out_cap = out_cap or int((replies["body_len"].astype(np.int64) * 7 // 6 + replies["attachment_len"] + replies["error_text_len"] + 1024).sum() + data.nbytes + 4096)
        out = np.empty(out_cap, np.uint8); offs = np.zeros(n, np.uint32); lens = np.zeros(n, np.uint32)
        _check(lib.b2_pack_responses(self._h, data.ctypes.data, data.nbytes, replies.ctypes.data, n, out.ctypes.data, out_cap, offs.ctypes.data, lens.ctypes.data))
        return [out[offs[i]:offs[i] + lens[i]].tobytes() for i in range(n)]

    def counters(self):
        out = (C.c_int64 * 8)()
        _check(lib.b2_counters_read(self._h, out))
        return list(out)

    def counters_device_ptr(self):
        return lib.b2_counters_device_ptr(self._h)
