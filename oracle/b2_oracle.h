/*
 * b2_oracle.h — CPU ORACLE (test infrastructure, NOT product code).
 *
 * A plain-C restatement of apache/brpc's message-processing hot path, written
 * function by function from the reference sources (each function cites the
 * file:line it follows).  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load this library; the product
 * (brpc_b200/libb2rpc.so) never links, imports or calls it.
 *
 * Parity pinning: CRC-32C is pinned by the RFC 3720 vectors of
 * test/crc32c_unittest.cc:18-71 and against the reference's own crc32c.cc
 * compiled into oracle/_ref; the protobuf wire codec (libprotobuf is a
 * third-party dependency absent from /root/reference, pinned 27.3 in
 * MODULE.bazel:11) is pinned by tests/golden/ (json) generated with
 * python-protobuf from the reference's .proto files (tests/golden/gen_golden.py);
 * snappy by the vendored snappy's compressed bytes and decoder verdicts
 * (tests/golden/snappy_vectors.json, snappy_ref_results.json).
 * The reference's tests hold NO golden baidu_std wire bytes (SURVEY §8c), so
 * frame-level parity is pinned by those fixtures, not by reference test vectors.
 */
#ifndef B2_ORACLE_H_
#define B2_ORACLE_H_
#include <stddef.h>
#include <stdint.h>
#include "../include/b2rpc.h"   /* ABI structs only (b2_run, b2_msg_desc, ...) */

#ifdef __cplusplus
extern "C" {
#endif

typedef struct orc_span { uint32_t off; uint32_t len; } orc_span; /* relative to meta start */

/* Decoded brpc.policy.RpcMeta (policy/baidu_rpc_meta.proto:26-55). */
typedef struct orc_rpc_meta {
    uint32_t has;                 /* B2_HAS_* */
    /* RpcRequestMeta */
    int      has_service_name, has_method_name;
    orc_span service_name, method_name, request_id;
    int64_t  log_id, trace_id, span_id, parent_span_id;
    int      has_span_id, has_parent_span_id;
    int32_t  timeout_ms;
    /* RpcResponseMeta */
    int      has_error_code, has_error_text;
    int32_t  error_code;
    orc_span error_text;
    int32_t  compress_type;
    int64_t  correlation_id;
    int32_t  attachment_size;
    int      chunk_has_stream_id, chunk_has_chunk_id;
    orc_span authentication_data;
    int      ss_has_stream_id;
    int64_t  ss_stream_id;
    int      ss_need_feedback, ss_writable;
    uint32_t ss_n_extra;
    uint32_t n_user_fields;       /* map entries seen on the wire */
    int32_t  content_type;
    int32_t  checksum_type;
    orc_span checksum_value;
} orc_rpc_meta;

/* Decoded brpc.StreamFrameMeta (streaming_rpc_meta.proto:39-49). */
typedef struct orc_stream_meta {
    uint32_t has;                 /* B2_SHAS_* | B2_SVAL_HAS_CONTINUATION */
    int64_t  stream_id, source_stream_id, consumed_size;
    int32_t  frame_type;
    int      feedback_has_consumed_size;
} orc_stream_meta;

typedef struct orc_config {
    uint64_t max_body_size;       /* FLAGS_max_body_size, protocol.cpp:52 */
    const char* server_identity;  /* "ip:port" of Controller::AppendServerIdentiy, or NULL */
    const b2_method* methods; uint32_t n_methods;
    int stream_handler;           /* B2_STREAM_* */
    uint32_t protocols;           /* handlers of the messenger, bit = ProtocolType; 0 = baidu_std | streaming_rpc */
} orc_config;

/* ---- leaf codecs ---------------------------------------------------------- */
uint32_t orc_crc32c_extend(uint32_t init_crc, const void* data, size_t n); /* crc32c.cc:379-454 */
uint32_t orc_crc32c_mask(uint32_t crc);                                      /* crc32c.h:38-41 */
uint32_t orc_crc32c_unmask(uint32_t masked);                                 /* crc32c.h:44-47 */
size_t orc_snappy_max_compressed_length(size_t n);                            /* snappy.cc:55-77 */
size_t orc_snappy_compress(const uint8_t* in, size_t n, uint8_t* out);        /* RawCompress, snappy.cc:875-956 */
int orc_snappy_uncompressed_length(const uint8_t* in, size_t n, size_t* ulen); /* GetUncompressedLength */
int orc_snappy_uncompress(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* got);  /* RawUncompress, cap >= length */

/* ---- protobuf wire decode of the path's messages --------------------------
 * return 1 = ParsePbFromIOBuf succeeded (protocol.cpp:236-239), 0 = failed. */
int orc_parse_rpc_meta(const uint8_t* p, size_t n, orc_rpc_meta* out);
int orc_parse_stream_meta(const uint8_t* p, size_t n, orc_stream_meta* out);
/* EchoRequest (example/echo_c++/echo.proto:23-25): span of `message` rel. to p */
int orc_parse_echo_request(const uint8_t* p, size_t n, orc_span* message);

/* ---- encoders (client mirror; used by tests to build traffic) -------------
 * PackRpcRequest (baidu_rpc_protocol.cpp:1045-1133) for an EchoRequest;
 * returns frame length written to out (cap must be large enough). */
typedef struct orc_request_spec {
    const char* service_name; const char* method_name;
    int has_log_id; int64_t log_id;
    int64_t correlation_id;
    int32_t compress_type, checksum_type, content_type;
    const uint8_t* message; uint32_t message_len;
    const uint8_t* attachment; uint32_t attachment_len;
    int has_trace; int64_t trace_id, span_id, parent_span_id;
    const char* request_id;       /* NULL = unset */
    int32_t timeout_ms;           /* 0 = unset */
} orc_request_spec;
size_t orc_pack_echo_request(const orc_request_spec* s, uint8_t* out, size_t cap);
/* PackStreamMessage (streaming_rpc_protocol.cpp:42-58), DATA frame */
size_t orc_pack_stream_frame(int64_t stream_id, int64_t source_stream_id, int frame_type,
                             int has_continuation, int cont_value,
                             const uint8_t* data, uint32_t data_len, uint8_t* out, size_t cap);

/* ---- the whole path over one batch ----------------------------------------
 * For every run: the ProcessNewMessage cut loop, ProcessRpcRequest, the echo
 * service, SendRpcResponse.  Responses are packed back to back (no padding) in
 * message order into resp; msgs[i].resp_off/resp_len index it.
 * Returns 0, or -1 when a capacity is exceeded. */
int orc_process_batch(const orc_config* cfg, const uint8_t* bytes, uint32_t nbytes,
                      const b2_run* runs, uint32_t n_runs,
                      b2_run_status* run_status,
                      b2_msg_desc* msgs, uint32_t msg_cap, uint32_t* n_msgs,
                      uint8_t* resp, uint32_t resp_cap, uint32_t* resp_bytes);

#ifdef __cplusplus
}
#endif
#endif

/* ---- HPACK (h2 header compression), a15 ------------------------------------------------------
 * Restates HPacker::Decode (src/brpc/details/hpack.cpp:765-843), DecodeWithKnownPrefix (:733-763),
 * DecodeInteger (:531-565), DecodeString + HuffmanDecoder (:606-635, :403-473) and the decoder's
 * IndexTable (:72-229).  One orc_hpack holds a connection's dynamic table. */
#ifdef __cplusplus
extern "C" {
#endif
typedef struct orc_hpack orc_hpack;
orc_hpack* orc_hpack_new(uint32_t max_table_size);
void orc_hpack_free(orc_hpack*);
/* Decode a whole header block the way H2StreamContext::ConsumeHeaders loops HPacker::Decode
 * (policy/http2_rpc_protocol.cpp:1221-1232).  Output records: u16 name_len, u16 value_len, name, value.
 * Returns 0 = block consumed, 1 = ran out of bytes inside a field (rc == 0), -1 = error. */
int orc_hpack_decode_block(orc_hpack* h, const uint8_t* in, uint32_t n, uint8_t* out, uint32_t out_cap,
                           uint32_t* out_len, uint32_t* n_headers);
/* H2Context::ConsumeFrameHead (policy/http2_rpc_protocol.cpp:438-465) chained over a byte run:
 * fills frames[i] = {type, flags, stream_id, payload_off, payload_len}; returns the count, sets
 * *consumed and *err (B2_PARSE_ERROR_NOT_ENOUGH_DATA normally, ABSOLUTELY_WRONG on a bad head). */
typedef struct orc_h2_frame { uint8_t type, flags; uint16_t pad; uint32_t stream_id, payload_off, payload_len; } orc_h2_frame;
/* HPacker::Decode, one field (name/value buffers of 64 KiB).  >0 field bytes, 0 out of data, -1 error; *adv = iterator advance */
int orc_hpack_field(orc_hpack* h, const uint8_t* p, uint32_t n, uint8_t* name, uint32_t* nl, uint8_t* value, uint32_t* vl, uint32_t* adv);
/* The server side of ParseH2Message (policy/http2_rpc_protocol.cpp:1103-1138) over one connection's read buffer:
 * H2Context::Consume (:467-543) until it stops, with the reference's unbounded stream map.  Completed requests are
 * appended to msgs (b2_h2_msg, offsets into blob), the WriteAck()ed bytes to ctrl.  Returns the ParseError that ended
 * the loop (B2_PARSE_ERROR_*), *consumed = bytes popped from the buffer. */
typedef struct orc_h2_conn orc_h2_conn;
orc_h2_conn* orc_h2_conn_new(void);
void orc_h2_conn_free(orc_h2_conn*);
uint32_t orc_h2_consume(orc_h2_conn* c, const orc_config* cfg, const uint8_t* in, uint32_t n, uint32_t* consumed,
                        b2_h2_msg* msgs, uint32_t msg_cap, uint32_t* n_msgs,
                        uint8_t* ctrl, uint32_t ctrl_cap, uint32_t* ctrl_len,
                        uint8_t* blob, uint32_t blob_cap, uint32_t* blob_len,
                        uint32_t* remote_max_frame_size, uint32_t* remote_stream_window_size);
/* one response through H2UnsentResponse::AppendAndDestroySelf + PackH2Message on this connection; returns the byte count
 * (out must hold body_len + 9 * (body_len / 16384 + 8) + 1 KiB) */
uint32_t orc_h2_pack_response(orc_h2_conn* c, const b2_h2_response* r, const uint8_t* bytes, uint8_t* out);
/* client side: H2UnsentRequest::New + AppendAndDestroySelf (http2_rpc_protocol.cpp:1382-1592); returns B2_H2_REQ_* */
int32_t orc_h2_pack_request(orc_h2_conn* c, const b2_h2_request* r, const uint8_t* bytes, uint8_t* out, uint32_t* out_len, uint32_t* stream_id);
void orc_h2_conn_set_next_stream_id(orc_h2_conn* c, uint32_t id);
int orc_h2_conn_peer_update(orc_h2_conn* c, const b2_h2_peer_update* u);
uint32_t orc_h2_scan(const uint8_t* in, uint32_t n, uint32_t max_frame_size, orc_h2_frame* frames, uint32_t cap,
                     uint32_t* consumed, uint32_t* err);
/* SendRpcResponse (baidu_rpc_protocol.cpp:273-460) for a reply the host produced: the checker of b2_pack_responses.
 * Frame length; 0 = not packable (gzip / zlib reply); (size_t)-1 = out too small. */
size_t orc_pack_response(const b2_reply* r, const uint8_t* bytes, uint8_t* out, size_t cap);

/* What GzipInputStream(format = B2_COMPRESS_TYPE_GZIP | B2_COMPRESS_TYPE_ZLIB) over `in` (one block) yields before it reports
 * end-of-stream (b2_oracle_gzip.c).  *out is malloc'ed; release with orc_free.  0, or -1 when out of memory. */
int orc_gzip_input_stream(const uint8_t* in, size_t n, int format, uint8_t** out, size_t* out_len);
void orc_free(void* p);
/* the device's sizing pass over the same stream (no data checks): bound of the bytes handed over, limit + 1 when beyond `limit` */
size_t orc_gzip_sizing_bound(const uint8_t* in, size_t n, int format, size_t limit);
#define ORC_GZ_MAX_IN  (1u << 20)   /* b2_inflate.cuh kGzMaxIn / kGzMaxOut: larger bodies are left to the host (B2_MSG_UNSUPPORTED) */
#define ORC_GZ_MAX_OUT (1u << 20)

#ifdef __cplusplus
}
#endif
