"""oracle orc_pack_response (SendRpcResponse for host-produced replies, baidu_rpc_protocol.cpp:273-460) against frames serialized by
python-protobuf from the reference's .proto files, the reference's snappy and crc32c (tests/golden/gen_response_vectors.py)."""
import json
import os

import _oracle as O
from _replies import ReplyBatch

HERE = os.path.dirname(os.path.abspath(__file__))


def load_vectors():
    vec = json.load(open(os.path.join(HERE, "golden", "response_vectors.json")))
    b = ReplyBatch()
    for v in vec:
        b.add(error_code=v["error_code"], error_text=v["error_text"].encode(), body=bytes.fromhex(v["body"]), attachment=bytes.fromhex(v["attachment"]),
              compress_type=v["compress_type"], checksum_type=v["checksum_type"], content_type=v["content_type"], correlation_id=v["correlation_id"],
              request_checksum=bytes.fromhex(v["request_checksum"]), stream=v["stream"],
              user_fields=[(v["user_field"][0].encode(), v["user_field"][1].encode())] if v["user_field"] else ())
    return vec, b.arrays()


def test_oracle_reply_frames_equal_python_protobuf():
    vec, (data, recs) = load_vectors()
    kinds = set()
    for v, r in zip(vec, recs):
        assert O.pack_response(r, data).hex() == v["frame"], v
        kinds.add((v["error_code"] != 0, v["compress_type"], v["checksum_type"], v["stream"] is not None, v["user_field"] is not None))
    assert len(kinds) >= 24
    # gzip / zlib replies are not packed
    b = ReplyBatch(); b.add(body=b"x" * 10, compress_type=2); b.add(body=b"x" * 10, compress_type=3); b.add(error_code=1003, error_text=b"e", compress_type=2)
    d, rr = b.arrays()
    assert O.pack_response(rr[0], d) == b"" and O.pack_response(rr[1], d) == b"" and O.pack_response(rr[2], d) != b""
