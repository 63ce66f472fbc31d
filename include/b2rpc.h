/*
 * b2rpc.h — C ABI of the B200-native brpc message-processing hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  Every entry point names the
 * reference interface it replaces (paths relative to the apache/brpc tree).
 * Plain pointers and sizes only; no C++ / torch types cross this boundary.
 * All compute runs in hand-written sm_100a CUDA kernels; there is no CPU
 * fallback: every call fails with B2_E_NO_DEVICE when no CUDA device exists.
 *
 * Model.  The host messenger gathers, for each readable Socket, the bytes
 * that are pending in its read buffer (reference: Socket::_read_buf filled by
 * Socket::DoRead, src/brpc/socket.cpp:2042-2122) into one *batch*: a flat
 * byte buffer plus one b2_run per socket.  One call cuts every run into
 * messages exactly like InputMessenger::ProcessNewMessage
 * (src/brpc/input_messenger.cpp:206-322) would, decodes the RpcMeta /
 * StreamFrameMeta of each message, runs the registered device handler (echo)
 * and packs the response frames (SendRpcResponse,
 * src/brpc/policy/baidu_rpc_protocol.cpp:273-460).
 * Further down: how bytes cross PCIe (b2_set_modes: kernels pull the pinned read blocks in place, replies by reference or as the
 * writev gather list), the latency path (b2_ring_*: a persistent kernel behind a pinned submit ring), the handler set of the messenger
 * (b2_set_protocols: hulu_pbrpc / sofa_pbrpc / nshead framing; rpc_dump files as a source), leaf codecs with the reference's signatures
 * (CRC32C, snappy), the client mirror (b2_pack_requests), replies the host produced (b2_pack_responses = SendRpcResponse), and the
 * h2/gRPC server path (b2_h2_process_batch = ParseH2Message, b2_h2_pack_responses = H2UnsentResponse + PackH2Message) whose
 * per-connection state lives on the device between calls, and the sending half of h2 client connections (b2_h2_pack_requests =
 * H2UnsentRequest::New + AppendAndDestroySelf; b2_h2_conn_peer_update mirrors the peer's SETTINGS / WINDOW_UPDATE).
 */
#ifndef B2RPC_H_
#define B2RPC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes (never exceptions, never errno side channels) ---------- */
#define B2_OK              0
#define B2_E_INVAL        -1   /* bad argument */
#define B2_E_NO_DEVICE    -2   /* CUDA device/driver missing: there is NO CPU path */
#define B2_E_CUDA         -3   /* a CUDA call failed; see b2_last_error() */
#define B2_E_CAPACITY     -4   /* batch exceeds a ctx capacity (bytes / msgs / resp) */
#define B2_E_NOMEM        -5

/* ---- ParseError, identical values to src/brpc/parse_result.h:25-32 ------- */
#define B2_PARSE_OK                    0
#define B2_PARSE_ERROR_TRY_OTHERS      1
#define B2_PARSE_ERROR_NOT_ENOUGH_DATA 2
#define B2_PARSE_ERROR_TOO_BIG_DATA    3
#define B2_PARSE_ERROR_NO_RESOURCE     4
#define B2_PARSE_ERROR_ABSOLUTELY_WRONG 5

/* ---- ProtocolType subset, values of src/brpc/options.proto:38-67 --------- */
#define B2_PROTOCOL_UNKNOWN       0
#define B2_PROTOCOL_BAIDU_STD     1
#define B2_PROTOCOL_STREAMING_RPC 2
#define B2_PROTOCOL_HULU_PBRPC    3   /* framing only: b2_set_protocols */
#define B2_PROTOCOL_SOFA_PBRPC    4
#define B2_PROTOCOL_NSHEAD        12

/* ---- CompressType / ChecksumType / ContentType, options.proto:69-88 ------ */
#define B2_COMPRESS_TYPE_NONE   0
#define B2_COMPRESS_TYPE_SNAPPY 1
#define B2_COMPRESS_TYPE_GZIP   2
#define B2_COMPRESS_TYPE_ZLIB   3
#define B2_CHECKSUM_TYPE_NONE   0
#define B2_CHECKSUM_TYPE_CRC32C 1
#define B2_CONTENT_TYPE_PB      0

/* ---- brpc error codes used in replies, src/brpc/errno.proto:25-49 -------- */
#define B2_ENOSERVICE 1001
#define B2_ENOMETHOD  1002
#define B2_EREQUEST   1003
#define B2_EINTERNAL  2001
#define B2_ERESPONSE  2002

/* ---- per-message disposition (b2_msg_desc.status) ------------------------ */
#define B2_MSG_ECHOED        0  /* device handler ran, OK response packed            */
#define B2_MSG_ERROR_REPLIED 1  /* error response packed on device (error_code != 0) */
#define B2_MSG_HOST          2  /* valid request of a host-handled method; no reply  */
#define B2_MSG_BAD_META      3  /* RpcMeta failed to parse: reference closes socket
                                   with EREQUEST (baidu_rpc_protocol.cpp:577-582)   */
#define B2_MSG_STREAM_FRAME  4  /* streaming_rpc frame, meta decoded, host routes it */
#define B2_MSG_BAD_STREAM_META 5 /* StreamFrameMeta failed to parse: frame dropped
                                   (streaming_rpc_protocol.cpp:97-100)              */
#define B2_MSG_UNSUPPORTED   6  /* left to the host untouched: a non-pb content type (json ...), a reply the method wants gzip / zlib
                                   COMPRESSED, or a gzip / zlib body beyond 1 MiB (compressed or inflated; one thread walks a DEFLATE stream) */
#define B2_MSG_RESPONSE      7  /* client-side socket: a response was processed (ProcessRpcResponse,
                                   baidu_rpc_protocol.cpp:911-1013).  error_code = what Controller::SetFailed
                                   would get (0 = OK); resp_off/resp_len = the EchoResponse.message bytes,
                                   located in the BATCH buffer */
#define B2_MSG_RESPONSE_UNZ  8  /* same, the response was snappy / gzip / zlib compressed: message bytes are in the resp region */
#define B2_MSG_REPLAY       10  /* a record of an rpc_dump file (B2_RUN_RPC_DUMP) re-packed as a baidu_std request frame: resp_off/resp_len;
                                   compress_type / attachment_size = the sample's; protocol = the sample's protocol_type (only baidu_std
                                   samples are re-packed, others are B2_MSG_UNSUPPORTED) */
#define B2_MSG_FRAMED        9  /* a message of another length-prefixed protocol (hulu_pbrpc, sofa_pbrpc, nshead): cut by the
                                   device, processed by the host; protocol / frame_off / meta_size / body_size are set, body_size
                                   counts the bytes behind the 12- (hulu), 24- (sofa) or 36-byte (nshead) header */

/* ---- has_bits of b2_msg_desc --------------------------------------------- */
#define B2_HAS_REQUEST          (1u << 0)
#define B2_HAS_RESPONSE         (1u << 1)
#define B2_HAS_COMPRESS_TYPE    (1u << 2)
#define B2_HAS_CORRELATION_ID   (1u << 3)
#define B2_HAS_ATTACHMENT_SIZE  (1u << 4)
#define B2_HAS_CHUNK_INFO       (1u << 5)
#define B2_HAS_AUTH_DATA        (1u << 6)
#define B2_HAS_STREAM_SETTINGS  (1u << 7)
#define B2_HAS_USER_FIELDS      (1u << 8)
#define B2_HAS_CONTENT_TYPE     (1u << 9)
#define B2_HAS_CHECKSUM_TYPE    (1u << 10)
#define B2_HAS_CHECKSUM_VALUE   (1u << 11)
#define B2_HAS_LOG_ID           (1u << 12)
#define B2_HAS_TRACE_ID         (1u << 13)
#define B2_HAS_REQUEST_ID       (1u << 14)
#define B2_HAS_TIMEOUT_MS       (1u << 15)
/* streaming_rpc frames reuse bits 0..4: */
#define B2_SHAS_STREAM_ID        (1u << 0)
#define B2_SHAS_SOURCE_STREAM_ID (1u << 1)
#define B2_SHAS_FRAME_TYPE       (1u << 2)
#define B2_SHAS_HAS_CONTINUATION (1u << 3)
#define B2_SHAS_FEEDBACK         (1u << 4)
#define B2_SVAL_HAS_CONTINUATION (1u << 8)  /* value of has_continuation */

/*
 * One socket's pending bytes inside the batch buffer.
 * Reference: Socket::_read_buf + Socket::preferred_index()
 * (src/brpc/socket.h:865-883).  `offset` must be a multiple of 16.
 */
typedef struct b2_run {
    uint64_t socket_id;        /* opaque (SocketId); echoed back, never interpreted */
    uint32_t offset;           /* byte offset of the run inside the batch buffer */
    uint32_t length;           /* pending bytes of this socket */
    int32_t  preferred_proto;  /* Socket::preferred_index(): B2_PROTOCOL_* or -1 */
    uint32_t flags;            /* B2_RUN_* */
} b2_run;                      /* 24 bytes */
#define B2_RUN_RPC_DUMP 4u     /* the run is not a socket but an rpc_dump FILE (src/brpc/rpc_dump.cpp:237-258: records "PRPC" BE32(meta+request) BE32(meta)
                                  RpcDumpMeta request): records are cut like SampleIterator::Pop (:322-361) and every baidu_std sample is turned into the
                                  request frame rpc_replay would send (PackRpcRequest's replay branch, baidu_rpc_protocol.cpp:1067-1075): status
                                  B2_MSG_REPLAY, the frame in the resp region, correlation_id = socket_id + index of the record in the run */
#define B2_RUN_CLIENT 1u       /* Socket::CreatedByConnect(): client-side protocol rules of CutInputMessage
                                  (input_messenger.cpp:122-138) and ProcessRpcResponse instead of ProcessRpcRequest */

/*
 * Result of the cut loop for one run == what InputMessenger::ProcessNewMessage
 * leaves behind on the Socket.
 */
typedef struct b2_run_status {
    uint32_t consumed;         /* bytes cut off the front of the run (pop_front) */
    uint32_t parse_error;      /* B2_PARSE_ERROR_* that ended the loop; anything
                                  other than NOT_ENOUGH_DATA closes the socket
                                  (input_messenger.cpp:227-239) */
    uint32_t n_msgs;           /* messages cut (Socket::AddInputMessages) */
    uint32_t first_msg;        /* index of this run's first b2_msg_desc */
    int32_t  preferred_proto;  /* Socket::preferred_index() after the loop */
    uint32_t n_unanswered;     /* B2_RESP_IOVEC only (else 0): messages of this run that are NOT a device-written reply
                                  (B2_MSG_HOST, stream frames, framed-only protocols, unsupported codecs, bad metas ...), i.e.
                                  the ones the host must pick out of msgs[].  (The _avg_msg_size read-size hint,
                                  input_messenger.cpp:242-261, stays on the host: it is consumed / n_msgs smoothed.) */
    uint32_t resp_off;         /* first response byte of this run in the resp region */
    uint32_t resp_bytes;       /* span (incl. alignment padding) of this run's responses */
} b2_run_status;               /* 32 bytes */

/*
 * One cut message == MostCommonMessage (policy/most_common_message.h:33-49)
 * + the decoded RpcMeta (policy/baidu_rpc_meta.proto:26-55)
 * + where its response frame was packed.  Exactly 64 bytes, written once by
 * the device.  For B2_PROTOCOL_STREAMING_RPC frames: correlation_id =
 * StreamFrameMeta.stream_id, log_id = source_stream_id, compress_type =
 * frame_type, attachment_size = low 32 bits of feedback.consumed_size,
 * checksum_type = high 32 bits of it.
 */
typedef struct b2_msg_desc {
    uint32_t run_idx;          /* index of the b2_run this message was cut from */
    uint32_t frame_off;        /* offset of the 12-byte header in the batch buffer */
    uint32_t body_size;        /* header: meta + payload (+attachment) bytes */
    uint32_t meta_size;        /* header: RpcMeta bytes */
    int64_t  correlation_id;
    int64_t  log_id;
    int32_t  attachment_size;
    int32_t  compress_type;
    int32_t  checksum_type;
    int32_t  error_code;       /* brpc error code carried by the reply (0 = OK) */
    uint16_t has_bits;         /* B2_HAS_* */
    uint8_t  protocol;         /* B2_PROTOCOL_* */
    uint8_t  content_type;
    int16_t  method_idx;       /* registered method index, -1 = not found */
    uint16_t status;           /* B2_MSG_* */
    uint32_t resp_off;         /* offset of the reply frame in the resp region */
    uint32_t resp_len;         /* bytes of the reply frame (0 = none) */
} b2_msg_desc;                 /* 64 bytes */

/* device handler kinds for b2_register_method */
#define B2_HANDLER_HOST 0      /* descriptor only: user code runs on the host */
#define B2_HANDLER_ECHO 1      /* example::EchoService::Echo, example/echo_c++/server.cpp:44-84 */

typedef struct b2_method {
    const char* service_full_name;  /* "example.EchoService" */
    const char* service_name;       /* "EchoService" (jprotobuf short name,
                                       baidu_rpc_protocol.cpp:738-748) */
    const char* method_name;        /* "Echo" */
    const char* request_type_name;  /* "example.EchoRequest" (used in EREQUEST text) */
    int32_t handler;                /* B2_HANDLER_* */
    int32_t echo_attachment;        /* -echo_attachment (server.cpp:31) */
    int32_t response_checksum_type; /* -enable_checksum -> CRC32C (server.cpp:80-82) */
    int32_t response_compress_type; /* cntl->set_response_compress_type() */
} b2_method;

typedef struct b2_options {
    int32_t  device;           /* CUDA ordinal */
    uint32_t max_batch_bytes;  /* capacity of the device batch buffer */
    uint32_t max_msgs;         /* capacity of the descriptor array */
    uint32_t max_runs;
    uint32_t max_resp_bytes;   /* capacity of the response region (0 = derive) */
    uint32_t tile_bytes;       /* speculative scan tile, power of two (0 = default) */
    uint64_t max_body_size;    /* FLAGS_max_body_size (protocol.cpp:52), 0 = 64 MiB */
} b2_options;

/* B2_RESP_BY_REF: where reply i's payload lives.  Reply i = resp[msgs[i].resp_off, +prefix_len) followed by
 * bytes[src_off, +src_len) of the REQUEST batch — exactly how SendRpcResponse builds res_buf: header + meta, then
 * res_buf.append(res_body.movable()) / append(attachment) by reference (baidu_rpc_protocol.cpp:383-389).
 * msgs[i].resp_len = prefix_len + src_len.  src_len == 0: the whole reply is in resp (error replies, checksummed or
 * compressed replies, client-side results). */
typedef struct b2_resp_ref { uint32_t prefix_len, src_off, src_len, reserved; } b2_resp_ref;   /* 16 bytes */

/* B2_RESP_IOVEC: the same replies as ready-made `struct iovec` pairs (layout of <sys/uio.h>) with HOST addresses — what
 * IOBuf::cut_multiple_into_file_descriptor (src/butil/iobuf.cpp:954-992) assembles from the block references of the queued
 * replies before its writev, written by the GPU instead: iov[2*i] = reply i's bytes in the pinned resp block (the prefix, or the
 * whole reply), iov[2*i + 1] = its payload inside the caller's request bytes (length 0 when there is none).  A message the device
 * did not answer has two zero-length entries, so a run's replies are writev(fd, iov + 2*first_msg, 2*n_msgs) as they stand, and
 * b2_run_status.n_unanswered says whether the host has to look at that run's descriptors at all. */
typedef struct b2_iovec { void* iov_base; size_t iov_len; } b2_iovec;

/* Pointers into ctx-owned PINNED host memory, valid until the next batch call. */
typedef struct b2_batch_result {
    const b2_run_status* runs;     uint32_t n_runs;
    const b2_msg_desc*   msgs;     uint32_t n_msgs;
    const uint8_t*       resp;     uint32_t resp_bytes;   /* span of the resp region used */
    float kernel_ms;               /* device time of the kernels (CUDA events) */
    uint32_t n_launches;           /* kernels launched for this batch */
    const b2_resp_ref*   refs;     /* [n_msgs] in B2_RESP_BY_REF mode, else NULL */
    const b2_iovec*      iov;      /* [2 * n_msgs] in B2_RESP_IOVEC mode (refs is NULL then), else NULL */
} b2_batch_result;

typedef struct b2_ctx b2_ctx;

/* ---- lifecycle ----------------------------------------------------------- */
int  b2_ctx_create(const b2_options* opt, b2_ctx** out);
void b2_ctx_destroy(b2_ctx* ctx);
const char* b2_last_error(void);        /* thread-local text of the last failure */
const char* b2_version(void);

/* Replaces Server::AddService's method map used by ProcessRpcRequest
 * (FindMethodPropertyByFullName, baidu_rpc_protocol.cpp:749-756).
 * Returns the method index (>= 0) or a negative B2_E_*. */
int  b2_register_method(b2_ctx* ctx, const b2_method* m);

/* Which Protocol::parse handlers the messenger holds (InputMessenger::AddHandler, one bit per ProtocolType, probed in index order
 * exactly like CutInputMessage): default (1 << B2_PROTOCOL_BAIDU_STD) | (1 << B2_PROTOCOL_STREAMING_RPC).  The other length-prefixed
 * protocols that share MostCommonMessage can be added — ParseHuluMessage (policy/hulu_pbrpc_protocol.cpp:178-223), ParseSofaMessage
 * (policy/sofa_pbrpc_protocol.cpp:165-205), ParseNsheadMessage (policy/nshead_protocol.cpp:154-182): their messages are cut in the
 * same loop (preferred-index switching included) and surface as B2_MSG_FRAMED descriptors.  b2_run.preferred_proto may name any
 * enabled handler. */
int  b2_set_protocols(b2_ctx* ctx, uint32_t protocol_mask);

/* What the device does with streaming_rpc DATA frames beyond cutting them and decoding StreamFrameMeta:
 * B2_STREAM_DESC_ONLY (default) or B2_STREAM_SNAPPY_UNCOMPRESS — the frame payload is a snappy stream
 * (policy::SnappyDecompress(IOBuf, IOBuf), src/brpc/policy/snappy_compress.cpp:77-82, as an application of
 * example/streaming_echo_c++ would call on each received message) and is decompressed into the resp
 * region: resp_off/resp_len = the plain bytes, error_code = B2_EREQUEST when the stream is malformed. */
#define B2_STREAM_DESC_ONLY         0
#define B2_STREAM_SNAPPY_UNCOMPRESS 1
int  b2_set_stream_handler(b2_ctx* ctx, int kind);

/* "ip:port" that Controller::AppendServerIdentiy (src/brpc/controller.cpp:407-428)
 * prepends to every error text as "[ip:port]"; NULL/"" = no server identity. */
int  b2_set_server_identity(b2_ctx* ctx, const char* ip_port);

/* ---- block pool: assignable to butil::iobuf::blockmem_allocate/deallocate
 * (src/butil/iobuf.cpp:168-169), same role as rdma::block_pool
 * (src/brpc/rdma/rdma_helper.cpp:579-582, rdma/block_pool.h:74-105).  Pinned AND mapped memory, pooled: blocks
 * <= 8 KiB come from 4 MiB slabs, larger ones are cached per power-of-two class; cudaHostAlloc runs per slab, never
 * per block.  Thread-safe. ------ */
void* b2_block_alloc(size_t size);
void  b2_block_free(void* p);
uint64_t b2_block_pool_host_allocs(void);   /* cudaHostAlloc calls so far (pool diagnostics) */

/* ---- how bytes cross PCIe (both default to COPY) ---------------------------------------------------------
 * input:  B2_INPUT_COPY  cudaMemcpyAsync of the batch bytes into HBM, kernels read HBM.
 *         B2_INPUT_PULL  `bytes` of every batch call MUST be memory from b2_block_alloc (pinned + mapped; the socket
 *                        read blocks themselves, like the RDMA transport's registered blocks): the kernels read it IN
 *                        PLACE over PCIe, so only what the parse touches crosses the link — frame headers, RpcMeta, the
 *                        first body bytes, the speculative scan windows; bodies only when a checksum / codec needs them.
 * resp:   B2_RESP_COPY   every reply frame is materialised in the resp region and copied back.
 *         B2_RESP_BY_REF an OK echo reply is {prefix in resp, payload = a span of the request bytes} (b2_resp_ref), what
 *                        SendRpcResponse does with IOBuf references; only descriptors, refs and <= 64-byte prefixes
 *                        come back.  Everything else (errors, CRC'd / compressed replies) is still materialised.
 *         B2_RESP_IOVEC  BY_REF with the references already turned into the iovec list of the write (b2_iovec): the host
 *                        side does no per-message work for device-answered traffic. */
#define B2_INPUT_COPY 0
#define B2_INPUT_PULL 1
#define B2_RESP_COPY   0
#define B2_RESP_BY_REF 1
#define B2_RESP_IOVEC  2   /* BY_REF, and the device also writes the gather list: b2_batch_result.iov (below) */
int  b2_set_modes(b2_ctx* ctx, int input_mode, int resp_mode);

/* ---- the hot path, host-facing (H2D + kernels + D2H inside) ---------------
 * Replaces, for every run: InputMessenger::ProcessNewMessage
 * (input_messenger.cpp:206-322) -> CutInputMessage (:84-179) ->
 * ParseRpcMessage / ParseStreamingMessage -> ProcessRpcRequest
 * (baidu_rpc_protocol.cpp:568-866) -> SendRpcResponse (:273-460).
 * `bytes` may be any host memory (pinned memory from b2_block_alloc avoids a
 * staging copy). */
int  b2_process_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes,
                      const b2_run* runs, uint32_t n_runs, b2_batch_result* out);

/* b2_process_batch split in two so that several batches (one ctx each) can be in flight on
 * one GPU: submit enqueues H2D + kernels on the ctx's stream and returns; collect waits and
 * brings descriptors + responses back.  With >= 3 contexts the H2D copy of one batch, the
 * kernels of another and the D2H copy of a third overlap (full-duplex PCIe). */
int  b2_batch_submit(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs);
int  b2_batch_collect(b2_ctx* ctx, b2_batch_result* out);

/* ---- the latency path: a PERSISTENT kernel per context fed through a submit ring (north star: "a persistent per-GPU kernel
 * pulls batches of raw socket bytes staged into pinned host IOBuf blocks") -----------------------------------------------
 * For batches of up to 128 KiB / 512 runs / 1024 messages — what a set of synchronous clients keeps in flight — there is no
 * kernel launch, no cudaMemcpy and no stream synchronisation per batch: b2_ring_submit fills a slot of a ring that lives in
 * pinned + mapped host memory and rings its doorbell with a plain store; the resident kernel (one CTA, started by
 * b2_ring_start or by the first submission) polls the doorbell over PCIe, pulls runs and bytes (in place when `bytes` is
 * b2_block_alloc memory, else from the slot's staging copy), runs the same cut / decode / echo / pack code as
 * b2_process_batch and writes descriptors + replies straight into the slot's pinned output block; b2_ring_wait spins on the
 * slot's completion word.  Same role as the RDMA transport's always-polling completion loop (RdmaEndpoint::PollCq,
 * src/brpc/rdma/rdma_endpoint.cpp:1470-1591).  Up to 8 tickets may be in flight; a result stays valid until 8 further
 * submissions.  The kernel retires after 20 ms without work (B2_RING_IDLE_MS) so that it never blocks device-wide
 * synchronisation for long, and comes back with the next submission.  A batch whose results do not fit the compact block is
 * served by the big pipeline inside b2_ring_wait (needs every other ticket collected).  Not to be mixed with concurrent
 * batch calls on the same context. */
int  b2_ring_start(b2_ctx* ctx);
int  b2_ring_stop(b2_ctx* ctx);
int  b2_ring_submit(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs, uint32_t* ticket);
int  b2_ring_wait(b2_ctx* ctx, uint32_t ticket, b2_batch_result* out);
uint64_t b2_ring_launches(b2_ctx* ctx);   /* how many times the resident kernel was (re)started: the launches of the ring path */
/* Device-side phases of a collected ticket (diagnostics), nanoseconds since the resident kernel saw the doorbell:
 * [0] slot header read, [1] runs + bytes pulled into HBM, [2] cut / decode / echo / pack done, [3] results pushed to the host. */
int  b2_ring_phase_ns(b2_ctx* ctx, uint32_t ticket, uint64_t out[4]);
/* Measurement helper: us_out[i] = wall-clock microseconds of the i-th of `iters` back-to-back single-batch calls —
 * b2_process_batch (use_ring 0) or b2_ring_submit + b2_ring_wait (use_ring 1) — timed inside the library. */
int  b2_latency_probe(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs,
                      uint32_t iters, int use_ring, float* us_out);

/* ---- the same path split in three, for measurement with inputs resident in
 * HBM (bench.py `value`): upload once, execute many times, download. -------- */
int  b2_batch_upload(b2_ctx* ctx, const void* bytes, uint32_t nbytes,
                     const b2_run* runs, uint32_t n_runs);
int  b2_batch_execute(b2_ctx* ctx, float* kernel_ms, uint32_t* n_launches);
int  b2_batch_download(b2_ctx* ctx, b2_batch_result* out);
/* `steps` back-to-back passes of the whole kernel pipeline over the resident batch,
 * one CUDA-event pair around all of them on the launching stream. */
int  b2_batch_execute_many(b2_ctx* ctx, uint32_t steps, float* total_ms, uint32_t* n_launches);

/* Asynchronous form for pipelining several resident batches (one ctx each) on one GPU:
 * b2_batch_launch enqueues one pass on the ctx's stream and returns; b2_batch_wait blocks
 * until it is done.  b2_elapsed_ms(a, b) = device time from a's FIRST launch since its last
 * wait to b's LAST launch end (CUDA events; a and b may be the same ctx). */
int  b2_batch_launch(b2_ctx* ctx);
int  b2_batch_wait(b2_ctx* ctx);
int  b2_elapsed_ms(b2_ctx* a, b2_ctx* b, float* ms);

/* What the last upload / launch decided: out[0] tile bytes, [1] tiles, [2] frame offsets kept per tile, [3] 1 = the fused
 * decode+pack kernel served the batch (0 = the slot-scan pipeline). */
int  b2_batch_info(b2_ctx* ctx, uint32_t out[4]);

/* PCI bus id ("0000:1b:00.0") of a device, for a host side that wants to run its polling threads and first-touch its pinned blocks on
 * the CPUs next to the GPU (/sys/bus/pci/devices/<id>/local_cpulist): zero-copy reads that cross the socket interconnect lose most of
 * their rate.  No ctx needed.  (brpc pins nothing itself; its RDMA endpoint leaves NUMA placement to the deployment as well.) */
int  b2_device_pci_bus_id(int device, char* out, int cap);

/* Device time of each stage of the last execute (or b2_h2_decompress_requests), in launch order.  Writes up to
 * `cap` entries of (name, ms); returns the number of stages. */
int  b2_stage_times(b2_ctx* ctx, const char** names, float* ms, int cap);

/* ---- leaf codecs on device-resident or host buffers ----------------------
 * b2_crc32c_batch: one CRC-32C per (offset,length) slice == butil::crc32c::Value
 * (src/butil/crc32c.h:30-33) on each slice; out[i] is the UNMASKED crc. */
int  b2_crc32c_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes,
                     const uint32_t* offs, const uint32_t* lens, uint32_t n,
                     uint32_t* out);

/* b2_snappy_uncompress_batch: butil::snappy::Uncompress (src/butil/third_party/snappy/snappy.cc:1526-1552)
 * on each (offset,length) slice of raw-format snappy.  Output i is written to out + out_offs[i]
 * (out_offs is filled by the call, 16-byte aligned, in slice order) and out_lens[i] is its length,
 * or -1 when the reference would return false (malformed stream / length mismatch). */
int  b2_snappy_uncompress_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes,
                                const uint32_t* offs, const uint32_t* lens, uint32_t n,
                                void* out, uint32_t out_cap, uint32_t* out_offs, int32_t* out_lens);

/* b2_snappy_compress_batch: butil::snappy::Compress (snappy.cc:875-956), BIT-EXACT with the vendored
 * 1.1.3 encoder, on each (offset,length) slice.  Output i goes to out + out_offs[i] (filled by the
 * call: slots of MaxCompressedLength, 16-byte aligned), out_lens[i] = compressed size. */
int  b2_snappy_compress_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes,
                              const uint32_t* offs, const uint32_t* lens, uint32_t n,
                              void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens);

/* ---- the same leaves with the REFERENCE's own signatures, for direct substitution at seam 4 (the bodies of the
 * CompressHandler / ChecksumHandler registered in src/brpc/global.cpp:400-418, or any direct caller):
 *   b2_crc32c_extend                  == butil::crc32c::Extend          (src/butil/crc32c.h:24)
 *   b2_snappy_max_compressed_length   == butil::snappy::MaxCompressedLength   (third_party/snappy/snappy.h:112)
 *   b2_snappy_raw_compress            == butil::snappy::RawCompress     (snappy.h:125)   bit-exact output
 *   b2_snappy_get_uncompressed_length == butil::snappy::GetUncompressedLength (snappy.h:141), returns 1/0 for true/false
 *   b2_snappy_raw_uncompress          == butil::snappy::RawUncompress   (snappy.h:135), returns 1/0
 * They run on a process-wide default context (device $B2_DEVICE, default 0), one buffer per call: correct, not fast — the
 * batch forms above are the throughput path. */
uint32_t b2_crc32c_extend(uint32_t init_crc, const char* data, size_t n);
size_t   b2_snappy_max_compressed_length(size_t source_bytes);
void     b2_snappy_raw_compress(const char* input, size_t input_length, char* compressed, size_t* compressed_length);
int      b2_snappy_get_uncompressed_length(const char* compressed, size_t compressed_length, size_t* result);
int      b2_snappy_raw_uncompress(const char* compressed, size_t compressed_length, char* uncompressed);

/* ---- client mirror (SURVEY §8a a13 / a14): PackRpcRequest (src/brpc/policy/baidu_rpc_protocol.cpp:1045-1133) with
 * SerializeRpcRequest (:1015-1043: EchoRequest{message}, COMPRESS_TYPE_NONE / SNAPPY, CRC32C over the serialized body)
 * and PackStreamMessage (policy/streaming_rpc_protocol.cpp:42-58), one warp per frame.  RpcRequestMeta carries the
 * registered method's service_full_name / method_name (-baidu_protocol_use_fullname=true), log_id and timeout_ms when
 * flagged; RpcMeta always carries compress_type, correlation_id, content_type(0), checksum_type and checksum_value (what
 * PackRpcRequest sets unconditionally) and attachment_size when there is an attachment.  Tracing fields and request_id
 * are not covered.  Frame i lands at out + out_offs[i] (filled by the call), out_lens[i] long (0 = could not be packed). */
#define B2_REQ_BAIDU_STD     0
#define B2_REQ_STREAM_FRAME  1
#define B2_REQ_HAS_LOG_ID            1u   /* baidu_std */
#define B2_REQ_HAS_TIMEOUT           2u   /* baidu_std: timeout_ms > 0 is written */
#define B2_REQ_HAS_SOURCE_STREAM_ID  1u   /* stream frame */
#define B2_REQ_HAS_CONTINUATION      2u   /* stream frame: has_continuation is present ... */
#define B2_REQ_CONTINUATION_VALUE    4u   /* ... with this value */
typedef struct b2_request {
    uint32_t kind, flags;
    int32_t  method_idx;             /* baidu_std: registered method */
    int32_t  timeout_ms;             /* baidu_std */
    int64_t  correlation_id;         /* stream frame: stream_id */
    int64_t  log_id;                 /* stream frame: source_stream_id */
    int32_t  compress_type, checksum_type;   /* baidu_std */
    int32_t  frame_type;             /* stream frame: brpc::FrameType */
    uint32_t payload_off, payload_len;        /* EchoRequest.message / the stream data */
    uint32_t attachment_off, attachment_len;  /* baidu_std */
    uint32_t reserved;
} b2_request;                        /* 64 bytes */
int  b2_pack_requests(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_request* reqs, uint32_t n,
                      void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens);

/* ---- replies the HOST produced (B2_HANDLER_HOST methods, any service above the transport): SendRpcResponse
 * (src/brpc/policy/baidu_rpc_protocol.cpp:273-460) as a batch, one warp per reply.  `bytes` holds what the host has: the response
 * message as its Serializer wrote it (UNcompressed), the attachment, the error text, the request's checksum bytes, user fields.
 *   - body: SerializeResponse (:218-246) -> SerializeRpcMessage (:148-216): COMPRESS_TYPE_NONE copies it, SNAPPY compresses it here
 *     (bit-exact with the vendored snappy); response_checksum_type CRC32C is computed here over the (compressed) body
 *     (Crc32cCompute, policy/crc32c_checksum.cpp:28-42).  gzip / zlib replies are not packed (out_lens[i] = 0): bit-exact deflate
 *     output is zlib-version specific.
 *   - error_code != 0 (cntl->Failed()): no body, no attachment, nothing compressed or checksummed (:316-330); -1 becomes
 *     EINTERNAL (:333-337); error_text is written only when non-empty (:343-347).
 *   - RpcMeta (:339-380): response{error_code,[error_text]}, compress_type, correlation_id, [attachment_size], [stream_settings
 *     {stream_id, need_feedback, writable, extra_stream_ids}] (Stream::FillSettings, stream.cpp:678-682), [user_fields], content_type,
 *     checksum_type, checksum_value.  checksum_value = the CRC when one was computed, else the bytes at checksum_value_off — the
 *     REQUEST's checksum_value, which the Controller still holds (:608 + :349).  user_fields are written in the order given (a
 *     protobuf map has no defined wire order; with one entry there is nothing to order).
 * Reply i lands at out + out_offs[i] (filled by the call), out_lens[i] long (0 = could not be packed). */
#define B2_RSP_HAS_STREAM         1u
#define B2_RSP_STREAM_NEED_FEEDBACK 2u
#define B2_RSP_STREAM_WRITABLE    4u
typedef struct b2_reply {
    uint32_t flags;
    int32_t  error_code;
    int64_t  correlation_id;
    int32_t  compress_type, checksum_type, content_type;
    uint32_t error_text_off, error_text_len;
    uint32_t body_off, body_len;
    uint32_t attachment_off, attachment_len;
    uint32_t checksum_value_off, checksum_value_len;
    uint32_t extra_streams_off, n_extra_streams;   /* int64 little-endian each, 8-byte aligned offset */
    uint32_t user_fields_off, n_user_fields;       /* records: u32 key_len, u32 value_len, key bytes, value bytes (unaligned, back to back) */
    uint32_t reserved;
    int64_t  stream_id;
} b2_reply;                          /* 88 bytes */
int  b2_pack_responses(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_reply* replies, uint32_t n,
                       void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens);

/* ---- h2 / gRPC (SURVEY §8a a15): leaf calls first, then the whole server-side parser and the reply framing -----
 * b2_h2_scan_batch: H2Context::ConsumeFrameHead (src/brpc/policy/http2_rpc_protocol.cpp:438-465)
 * chained over every connection run.  runs[i].flags & B2_RUN_H2_PREFACE: the run starts a server-side
 * connection, the 24-byte client preface (:119-120, :469-479) is checked and skipped first.
 * frames of run i land at frames[i * cap_per_run ...]; err[i] is a B2_PARSE_ERROR_*. */
#define B2_RUN_H2_PREFACE 2u
typedef struct b2_h2_frame { uint8_t type, flags; uint16_t pad; uint32_t stream_id, payload_off, payload_len; } b2_h2_frame;
int  b2_h2_scan_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs,
                      uint32_t max_frame_size, b2_h2_frame* frames, uint32_t cap_per_run,
                      uint32_t* n_frames, uint32_t* consumed, uint32_t* err);
/* b2_hpack_decode_batch: HPacker::Decode (src/brpc/details/hpack.cpp:765-843) looped over header
 * blocks like H2StreamContext::ConsumeHeaders (http2_rpc_protocol.cpp:1221-1232).  Blocks of one
 * connection must be adjacent and in wire order; every connection (0 .. B2_HPACK_MAX_CONNS-1) owns a
 * dynamic table that persists across calls (b2_hpack_reset starts a new connection).  Block i's
 * records (u16 name_len, u16 value_len, name, value) land at out + i * per_block_cap.
 * status[i]: 0 consumed, 1 ran out of bytes inside a field, -1 malformed, -2 per_block_cap exceeded. */
#define B2_HPACK_MAX_CONNS 4096
typedef struct b2_hpack_block { uint32_t conn, offset, length, reserved; } b2_hpack_block;
int  b2_hpack_reset(b2_ctx* ctx, uint32_t conn, uint32_t max_table_size);
int  b2_hpack_decode_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_hpack_block* blocks, uint32_t n_blocks,
                           void* out, uint32_t per_block_cap, uint32_t* out_lens, int32_t* status, uint32_t* n_headers);

/* b2_h2_process_batch: the server side of ParseH2Message (src/brpc/policy/http2_rpc_protocol.cpp:1103-1138) =
 * H2Context::Consume (:467-543) looped over every connection run: client preface, frame heads, the frame handlers
 * OnData/OnHeaders/OnContinuation/OnResetStream/OnSettings/OnPing/OnGoAway/OnWindowUpdate (:545-1041) with their
 * flow-control bookkeeping, H2StreamContext::ConsumeHeaders (:1221-1306) over the connection's HPACK table, and — for
 * every stream that reaches OnEndStream — what ProcessHttpRequest reads first: ParseContentType and RemoveGrpcPrefix
 * (policy/http_rpc_protocol.cpp:176-230, :264-277) and the "/service/method" lookup of FindMethodPropertyByURIImpl
 * (:1088-1138, plain service/method form only).
 *   runs[i].socket_id = connection index (0 .. B2_H2_MAX_CONNS-1); state (settings, windows, pending streams, HPACK
 *   table) persists across calls; b2_h2_conn_reset starts a new server-side connection (H2Context ctor + Init).
 *   rs[i].ctrl_off/len  : the bytes the reference WriteAck()s while parsing (SETTINGS + WINDOW_UPDATE after the
 *                         preface, SETTINGS acks, PING acks, RST_STREAM, GOAWAY, WINDOW_UPDATEs), in order, inside out.
 *   msgs                : one per completed request, in parse order per run; header records (u16 name_len,
 *                         u16 value_len, name, value — every decoded field in order) and the concatenated DATA
 *                         payloads live in out.
 * Device capacities (the reference has none; they are run-time choices, b2_h2_configure): `max_pending` concurrent unfinished
 * streams per connection and `stream_bytes` (4 KiB of header records + the body) per unfinished stream whose body spans
 * several DATA frames (a body carried by one DATA frame is referenced in the input and needs none); beyond them the run ends
 * with B2_PARSE_ERROR_NO_RESOURCE (the host takes the connection over or closes it, input_messenger.cpp:227-239).
 * Defaults: B2_H2_MAX_CONNS connections x B2_H2_MAX_PENDING streams x B2_H2_STREAM_BYTES.  gRPC clients keep up to 100
 * calls in flight per connection (the server side of brpc advertises no SETTINGS_MAX_CONCURRENT_STREAMS): size
 * max_pending for that, e.g. b2_h2_configure(ctx, 256, 128, 69632) = 2.2 GB of the 180 GB HBM. */
#define B2_H2_MAX_CONNS 1024
#define B2_H2_MAX_PENDING 8
#define B2_H2_STREAM_BYTES 69632
/* Must precede the first h2 call on the context (the pool is allocated then).  stream_bytes: multiple of 16, > 4 KiB. */
int  b2_h2_configure(b2_ctx* ctx, uint32_t max_conns, uint32_t max_pending, uint32_t stream_bytes);
#define B2_H2_HEADER_BYTES 4096
#define B2_H2_FLAG_GRPC            1u   /* content-type is application/grpc[+...] (is_grpc_ct) */
#define B2_H2_FLAG_GRPC_PREFIX_OK  2u   /* RemoveGrpcPrefix succeeded: msg_off/msg_len are valid */
#define B2_H2_FLAG_GRPC_COMPRESSED 4u   /* compressed flag of the 5-byte prefix */
#define B2_H2_FLAG_HAS_PATH        8u
#define B2_H2_FLAG_BODY_IN_INPUT  16u   /* body_off/msg_off index the INPUT bytes (a single DATA frame carried the whole body): zero copy */
#define B2_H2_NO_METHOD 255u            /* no :method header (HttpHeader defaults to GET) */
typedef struct b2_h2_run_status {
    uint32_t consumed, parse_error, n_msgs, first_msg;
    uint32_t ctrl_off, ctrl_len;
    uint32_t remote_max_frame_size, remote_stream_window_size;   /* what PackH2Message needs next */
} b2_h2_run_status;                                              /* 32 bytes */
typedef struct b2_h2_msg {
    uint32_t run_idx, stream_id;
    uint32_t headers_off, headers_len, n_headers;
    uint32_t body_off, body_len;
    uint32_t http_method;        /* brpc::HttpMethod of the last :method, B2_H2_NO_METHOD if none */
    uint32_t content_type;       /* brpc::HttpContentType of the last content-type header (0 = others / none) */
    uint32_t flags;              /* B2_H2_FLAG_* */
    int32_t  method_idx;         /* registered method named by :path, -1 if none */
    uint32_t msg_off, msg_len;   /* gRPC message (body without the 5-byte prefix) */
    uint32_t path_off, path_len; /* the path part of :path inside out */
    uint32_t reserved;
} b2_h2_msg;                     /* 64 bytes */
int  b2_h2_conn_reset(b2_ctx* ctx, uint32_t conn);
int  b2_h2_process_batch(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs,
                         b2_h2_run_status* rs, b2_h2_msg* msgs, uint32_t msg_cap, uint32_t* n_msgs,
                         void* out, uint32_t out_cap);

/* b2_h2_pack_responses: H2UnsentResponse::AppendAndDestroySelf (src/brpc/policy/http2_rpc_protocol.cpp:1688-1750) +
 * PackH2Message (:1310-1380) + AddGrpcPrefix (policy/http_rpc_protocol.cpp:254-262) for a list of responses:
 * connection flow control (MinusWindowSize, else RST_STREAM(FLOW_CONTROL_ERROR)), HPacker::Encode (details/hpack.cpp:696-726)
 * of ":status" and "content-type" — and of the "grpc-status" / "grpc-message" trailers of a gRPC response — against
 * the connection's ENCODER table (indexed if present, else literal with incremental indexing and a name index when one
 * exists, no Huffman: the reference's defaults; never-indexed when the peer announced header_table_size 0), HEADERS
 * (+CONTINUATION), DATA frames split at the peer's max_frame_size, trailers, and the deferred connection WINDOW_UPDATE.
 * Responses of one connection must be adjacent and in write order; the state is the connection's (b2_h2_process_batch).
 * Response i's bytes land at out + out_offs[i] (filled by the call), out_lens[i] long.  User-defined response headers
 * are not covered.  bytes may be NULL (nbytes 0) when every field uses a zero-copy source. */
#define B2_H2_RESP_GRPC 1u
/* zero-copy sources: the buffers of the LAST b2_h2_process_batch on this context are still on the device */
#define B2_H2_RESP_BODY_IN_INPUT 2u   /* body_off indexes that call's input bytes (e.g. an echoed B2_H2_FLAG_BODY_IN_INPUT message) */
#define B2_H2_RESP_BODY_IN_OUT   4u   /* body_off indexes that call's out buffer */
#define B2_H2_RESP_CT_IN_OUT     8u   /* content_type_off indexes that call's out buffer (the request's own content-type value) */
#define B2_H2_RESP_BODY_IN_UNZ  16u   /* body_off indexes the last b2_h2_decompress_requests output (zero copy) */
typedef struct b2_h2_response {
    uint32_t conn, stream_id;
    int32_t  status_code;                            /* :status */
    uint32_t flags;                                  /* B2_H2_RESP_GRPC */
    uint32_t content_type_off, content_type_len;     /* inside bytes; length 0 = no content-type header */
    uint32_t body_off, body_len;                     /* the body; for gRPC the serialized message (the prefix is added here) */
    int32_t  grpc_status;
    uint32_t grpc_message_off, grpc_message_len;     /* already percent-encoded; length 0 = none */
    uint32_t reserved;
} b2_h2_response;                                    /* 48 bytes */
int  b2_h2_pack_responses(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_h2_response* resps, uint32_t n,
                          void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens);

/* b2_h2_decompress_requests: the GzipDecompress step of ProcessHttpRequest (src/brpc/policy/http_rpc_protocol.cpp:1646-1683) for
 * messages of the LAST b2_h2_process_batch on this context (their header records and bodies are still on the device).
 *   - gRPC (B2_H2_FLAG_GRPC): only a message whose prefix is valid (B2_H2_FLAG_GRPC_PREFIX_OK) and has the compressed flag is looked
 *     at; its encoding is the "grpc-encoding" header, and a missing header is the reference's EREQUEST "Fail to find header
 *     `grpc-encoding' in compressed gRPC request".  The message (msg_off/msg_len) is inflated.
 *   - otherwise a non-empty body's encoding is the "content-encoding" header, and the whole body is inflated.
 *   - headers are looked up the way HttpHeader keeps them (http_header.cpp:100-116): names case-insensitively, a repeated header
 *     folded with "," onto a non-empty value (an empty value is overwritten).  Only the exact value "gzip" is inflated
 *     (policy::GzipDecompress, gzip_compress.cpp:138-176,187-190); any other value leaves the bytes to the parser as they are.
 * Messages are taken in the order given and the caller passes the ones it would parse (method_idx is not looked at).  Inflated
 * messages are laid out back to back in `out` in message order; a message that does not fit into out_cap after the earlier ones
 * is B2_H2_UNZ_NO_ROOM.  Only the bytes up to the end of the last inflated message are written.  The output also stays on the
 * device for b2_h2_pack_responses (B2_H2_RESP_BODY_IN_UNZ) as long as the batch does (the rule of B2_H2_RESP_BODY_IN_INPUT).
 * Replies are not compressed (brpc compresses one only when the service sets response_compress_type, :971-994).
 * out_cap <= max_resp_bytes.  B2_E_INVAL: no h2 batch is live, or a message's ranges lie outside that batch's buffers. */
#define B2_H2_UNZ_NONE        0   /* nothing to inflate (not compressed / not gzip-encoded body): the message is msg_off/msg_len, or the body */
#define B2_H2_UNZ_OK          1   /* inflated: out[out_off, +out_len) */
#define B2_H2_UNZ_NO_ENCODING 2   /* compressed gRPC message, no grpc-encoding header -> EREQUEST (text above) */
#define B2_H2_UNZ_NOT_GZIP    3   /* compressed / encoded, but the (folded) value is not "gzip": parsed as it is */
#define B2_H2_UNZ_FAILED      4   /* GzipDecompress returned false -> EREQUEST "Fail to un-gzip request body" (a body in one block
                                     never yields it: DESIGN §5) */
#define B2_H2_UNZ_HOST        5   /* input or output beyond 1 MiB: left to the host, like B2_MSG_UNSUPPORTED */
#define B2_H2_UNZ_NO_ROOM     6   /* out_cap used up by earlier messages of this call */
typedef struct b2_h2_unz_result { uint32_t status, out_off, out_len, reserved; } b2_h2_unz_result;   /* 16 bytes */
int  b2_h2_decompress_requests(b2_ctx* ctx, const b2_h2_msg* msgs, uint32_t n, void* out, uint32_t out_cap, b2_h2_unz_result* res);

/* b2_h2_pack_requests — the CLIENT side of the same connection state: H2UnsentRequest::New (src/brpc/policy/http2_rpc_protocol.cpp:
 * 1382-1453: the header list) + H2UnsentRequest::AppendAndDestroySelf (:1496-1592) + PackH2Message (:1310-1380), what PackH2Request
 * (:1784-1800) queues for a call on an "h2" / "h2:grpc" channel.  Per request, in the reference's order:
 *   - the first request of a connection (b2_h2_conn_reset, nothing packed yet) is preceded by the 24-byte client preface and
 *     SerializeH2SettingsFrameAndWU of the default client settings (:253-265, flags :34-43: ENABLE_PUSH 0, INITIAL_WINDOW_SIZE 256 KiB,
 *     connection WINDOW_UPDATE 1 MiB - 65535) — written even when the request itself is then refused, as `out` has them there;
 *   - AllocateClientStreamId (http2_rpc_protocol.h:399-412): 1, 3, 5, ...; past 0x7fffffff -> B2_H2_REQ_RUNOUT (EH2RUNOUTSTREAMS);
 *   - a non-empty body is charged to the flow-control windows (H2StreamContext::ConsumeWindowSize :1199-1219): the peer's initial stream
 *     window, then MinusWindowSize on the connection window; not enough -> B2_H2_REQ_ELIMIT, the stream id stays consumed;
 *   - HPacker::Encode (details/hpack.cpp:696-726) against the connection's encoder table of ":method" (POST, or GET with
 *     B2_H2_REQ_GET), ":scheme" (http / https), ":path", ":authority", "content-type" when non-empty, "accept: * / *" and
 *     "user-agent: brpc/1.0 curl/7.0" when the flags say the call set neither (need_accept / need_user_agent), then the call's own
 *     headers in the order the caller lists them (the reference iterates its HttpHeader map: for gRPC "te: trailers",
 *     "grpc-accept-encoding", "grpc-timeout" of policy/http_rpc_protocol.cpp:660-704); never-indexed when the peer announced
 *     header_table_size 0;
 *   - HEADERS (+CONTINUATION) and the body as DATA frames split at the peer's max_frame_size, END_STREAM on the last frame, the
 *     deferred connection WINDOW_UPDATE; B2_H2_REQ_GRPC prepends AddGrpcPrefix's 5 bytes (policy/http_rpc_protocol.cpp:254-262).
 * `extra` headers: records {u16 name_len, u16 value_len (little endian), name, value} back to back at extra_off, extra_len bytes.
 * The pending-stream count against max_concurrent_streams (:1529) and GOAWAY (TryToInsertStream :425-436) belong to the
 * caller's correlation map, not to this call.  NOT built: the receiving half of a client connection (ParseH2Message on a socket
 * created by connect -> H2StreamContext::OnEndStream :823-846 -> ProcessHttpResponse) — the host's H2Context keeps parsing the
 * server's frames and mirrors what they change into the device's connection with b2_h2_conn_peer_update.  Requests of one
 * connection must be adjacent and in write order. */
#define B2_H2_REQ_GRPC       1u
#define B2_H2_REQ_GET        2u     /* :method GET instead of POST */
#define B2_H2_REQ_HTTPS      4u     /* :scheme https */
#define B2_H2_REQ_ACCEPT     8u     /* need_accept: append accept: * / * */
#define B2_H2_REQ_USER_AGENT 16u    /* need_user_agent: append user-agent: brpc/1.0 curl/7.0 */
#define B2_H2_REQ_OK     0
#define B2_H2_REQ_ELIMIT 1          /* brpc ELIMIT: remote_window_left is not enough */
#define B2_H2_REQ_RUNOUT 2          /* brpc EH2RUNOUTSTREAMS */
typedef struct b2_h2_request {
    uint32_t conn, flags;
    uint32_t path_off, path_len;                     /* inside bytes: URI::GenerateH2Path's result */
    uint32_t authority_off, authority_len;
    uint32_t content_type_off, content_type_len;     /* length 0 = no content-type header */
    uint32_t body_off, body_len;                     /* the attachment; for gRPC the serialized message */
    uint32_t extra_off, extra_len;
} b2_h2_request;                                     /* 48 bytes */
typedef struct b2_h2_request_result { int32_t status; uint32_t stream_id, out_off, out_len; } b2_h2_request_result;   /* 16 bytes */
int  b2_h2_pack_requests(b2_ctx* ctx, const void* bytes, uint32_t nbytes, const b2_h2_request* reqs, uint32_t n,
                         void* out, uint32_t out_cap, b2_h2_request_result* results);
/* What the peer's frames change in the state b2_h2_pack_requests / b2_h2_pack_responses read, for a connection whose frames the HOST
 * parses: H2Context::OnSettings (:848-915: _remote_settings; the first SETTINGS also takes MAX_WINDOW_SIZE - 65535 off the connection
 * window — pass it as a negative conn_window_add) and OnWindowUpdate on stream 0 (:1006-1041: AddWindowSize, B2_E_INVAL when the
 * window would pass 2^31 - 1 — FLOW_CONTROL_ERROR there).  Fields are applied when their bit is set in `set`. */
#define B2_H2_PEER_HEADER_TABLE_SIZE 1u
#define B2_H2_PEER_MAX_FRAME_SIZE    2u
#define B2_H2_PEER_STREAM_WINDOW     4u
#define B2_H2_PEER_CONN_WINDOW_ADD   8u
typedef struct b2_h2_peer_update {
    uint32_t set, header_table_size, max_frame_size, stream_window_size;
    int64_t  conn_window_add;
} b2_h2_peer_update;                                 /* 24 bytes */
int  b2_h2_conn_peer_update(b2_ctx* ctx, uint32_t conn, const b2_h2_peer_update* u);
/* the reference's own unit-test hook (:348-352: its tests start 10 000 ids before the end of the id space): the next client stream id */
int  b2_h2_conn_set_next_stream_id(b2_ctx* ctx, uint32_t conn, uint32_t next_id);

/* ---- counters (bvar::Adder-like, SURVEY §8e): per-GPU totals accumulated by
 * the kernels: [0] in_bytes [1] in_msgs [2] out_bytes [3] out_msgs [4] errors
 * [5] batches [6..7] reserved.  The cross-GPU reduce is an NCCL all-reduce on
 * this int64[8] done by the caller's communicator. -------------------------- */
#define B2_N_COUNTERS 8
int  b2_counters_read(b2_ctx* ctx, int64_t out[B2_N_COUNTERS]);
/* device pointer of the int64[8] (for ncclAllReduce / torch.distributed) */
void* b2_counters_device_ptr(b2_ctx* ctx);
/* bvar's cross-shard sum (an Adder combined over agents, src/bvar/reducer.h:227-233,335) across GPUs: ncclAllReduce(sum, int64 x 8) of the
 * counters IN PLACE on `nccl_comm` (an ncclComm_t of the caller: one rank per GPU) and the ctx's stream; the call returns when the sum is
 * there.  The library does not link NCCL: the entry point is looked up in the running process (torch / the transport loaded it), and the
 * call fails with B2_E_INVAL when it is not there.  Every rank of the communicator must call it. */
int  b2_counters_allreduce(b2_ctx* ctx, void* nccl_comm);

#ifdef __cplusplus
}
#endif
#endif  /* B2RPC_H_ */
