"""ctypes wrapper of the CPU oracle of b2_h2_decompress_requests (oracle/liboracle_h2gzip.so, built by build()) — tests only."""
import ctypes as C
import os

import numpy as np

from _oracle import H2_MSG_DT

HERE = os.path.dirname(os.path.abspath(__file__))
lib = C.CDLL(os.path.join(os.path.dirname(HERE), "oracle", "liboracle_h2gzip.so"))

H2_UNZ_RESULT_DT = np.dtype([("status", "<u4"), ("out_off", "<u4"), ("out_len", "<u4"), ("reserved", "<u4")])   # == b2_h2_unz_result
H2_UNZ_NONE, H2_UNZ_OK, H2_UNZ_NO_ENCODING, H2_UNZ_NOT_GZIP, H2_UNZ_FAILED, H2_UNZ_HOST, H2_UNZ_NO_ROOM = range(7)
lib.orc_h2_decompress.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]


def h2_decompress(msgs, blob, data=b"", out_cap=4 << 20):
    """orc_h2_decompress over H2_MSG_DT records (header records and bodies in blob; B2_H2_FLAG_BODY_IN_INPUT bodies in data).
    Returns (H2_UNZ_RESULT_DT per message, out bytes up to the end of the last inflated message)."""
    msgs = np.ascontiguousarray(msgs, dtype=H2_MSG_DT)
    blob = np.ascontiguousarray(np.frombuffer(bytes(blob), np.uint8) if not isinstance(blob, np.ndarray) else blob, dtype=np.uint8)
    res = np.zeros(len(msgs), H2_UNZ_RESULT_DT); out = np.zeros(max(out_cap, 1), np.uint8)
    assert lib.orc_h2_decompress(msgs.ctypes.data, len(msgs), bytes(data), blob.ctypes.data, out.ctypes.data, out_cap, res.ctypes.data) == 0
    ok = res["status"] == H2_UNZ_OK
    end = int((res["out_off"][ok].astype(np.int64) + res["out_len"][ok]).max()) if ok.any() else 0
    return res, out[:end].tobytes()
