// b2_h2.cuh — h2 frame-head scan and HPACK decode on the device (SURVEY §2.3 K8, §8a a15).
//   h2 frame heads  <- H2Context::ConsumeFrameHead   src/brpc/policy/http2_rpc_protocol.cpp:438-465
//   HPACK decode    <- HPacker::Decode               src/brpc/details/hpack.cpp:765-843 (+ :531-635, :403-473, :72-229)
// Both are per-connection serial state machines (frame chain; dynamic table), so the unit of
// parallelism is the connection: one thread per connection, thousands of connections per batch.
// Further down: the whole server side of ParseH2Message (k_h2_consume: stream state machine, SETTINGS / WINDOW_UPDATE /
// GOAWAY side effects as the bytes to write back) and the reply framing with HPACK encoding (k_h2_pack).
#pragma once
#include <cuda_runtime.h>
#include "b2_core.cuh"
#include "b2_hpack_tables.cuh"
#include "b2_inflate.cuh"

namespace b2 {

struct HpackState {                     // one connection's decoder table (IndexTable, hpack.cpp:72-229)
    uint32_t max_size, size, count, head, byte_head, pad[3];
    struct { uint16_t off, nl, vl, pad; } meta[128];   // ring, newest at `head`
    uint8_t bytes[4096];                // ring of name||value bytes, FIFO like the entries
};

#if defined(__CUDACC__)
__device__ __forceinline__ void hp_pop(HpackState& h) {
    const uint32_t i = (h.head + h.count - 1) & 127u;
    h.size -= (uint32_t)h.meta[i].nl + h.meta[i].vl + 32u;
    h.count--;
}
// AddHeader (hpack.cpp:150-177); entry bytes are read from `src` (name then value, contiguous)
__device__ __forceinline__ int hp_add(HpackState& h, const uint8_t* src, uint32_t nl, uint32_t vl) {
    const uint32_t es = nl + vl + 32u;
    if (nl == 0) return -1;                             // reference CHECK-aborts on an empty name
    while (h.count && h.size + es > h.max_size) hp_pop(h);
    if (es > h.max_size) return 0;
    if (h.count >= 128) return -1;
    h.head = (h.head + 127u) & 127u;
    h.meta[h.head].off = (uint16_t)h.byte_head; h.meta[h.head].nl = (uint16_t)nl; h.meta[h.head].vl = (uint16_t)vl;
    for (uint32_t i = 0; i < nl + vl; i++) h.bytes[(h.byte_head + i) & 4095u] = src[i];
    h.byte_head = (h.byte_head + nl + vl) & 4095u;
    h.count++; h.size += es;
    return 0;
}
// DecodeInteger (hpack.cpp:531-565): >0 bytes used, 0 not enough data, -1 malformed
__device__ __forceinline__ int hp_int(const uint8_t* p, uint32_t n, uint32_t prefix, uint32_t& value) {
    if (n == 0) return 0;
    unsigned long long tmp = p[0] & ((1u << prefix) - 1);
    if (tmp < ((1u << prefix) - 1)) { value = (uint32_t)tmp; return 1; }
    uint32_t i = 1; int m = 0; uint8_t cur;
    do {
        if (i >= n) return 0;
        cur = p[i++];
        tmp += (unsigned long long)(cur & 0x7f) << m;
        m += 7;
    } while ((cur & 0x80) && tmp < 10ull * 1024 * 1024);
    if (tmp >= 10ull * 1024 * 1024) return -1;
    value = (uint32_t)tmp;
    return (int)i;
}
// DecodeString (:606-635) with the Huffman walk of HuffmanDecoder (:414-468) over the pre-built tree
__device__ __forceinline__ int hp_str(const uint8_t* p, uint32_t n, uint8_t* out, uint32_t cap, uint32_t& olen) {
    if (n == 0) return 0;
    const bool huffman = p[0] & 0x80;
    uint32_t length = 0;
    const int ib = hp_int(p, n, 7, length);
    if (ib <= 0) return -1;
    if (length > n - (uint32_t)ib) return 0;
    const uint8_t* s = p + ib;
    if (!huffman) {
        if (length > cap) return -2;
        for (uint32_t i = 0; i < length; i++) out[i] = s[i];
        olen = length; return ib + (int)length;
    }
    int node = 0; uint32_t depth = 0, o = 0; bool padding = true;
    for (uint32_t i = 0; i < length; i++) {
        const uint32_t byte = s[i];
        for (int b = 7; b >= 0; b--) {
            const uint32_t bit = (byte >> b) & 1u;
            const int nx = kHuffTree[node][bit];
            if (nx == 0) return -1;                          // NULL_NODE
            if (nx < 0) {
                const int sym = -nx - 1;
                if (sym == 256) return -1;                   // EOS inside the string
                if (o >= cap) return -2;
                out[o++] = (uint8_t)sym; node = 0; depth = 0; padding = true;
                continue;
            }
            node = nx; depth++; padding = padding && bit;
        }
    }
    if (!(depth == 0 || (depth <= 7 && padding))) return -1;
    olen = o; return ib + (int)length;
}
// HeaderAt: 1..61 static, 62.. dynamic newest first; copies name (and value) into out
__device__ __forceinline__ bool hp_copy_indexed(const HpackState& h, uint32_t index, bool with_value, uint8_t* out, uint32_t cap,
                                                uint32_t& nl, uint32_t& vl, bool& overflow) {
    overflow = false;
    if (index >= 1 && index <= 61) {
        nl = kHpackStaticName[index - 1][1]; vl = with_value ? kHpackStaticValue[index - 1][1] : 0;
        if (nl + vl > cap) { overflow = true; return false; }
        for (uint32_t i = 0; i < nl; i++) out[i] = kHpackStaticBlob[kHpackStaticName[index - 1][0] + i];
        for (uint32_t i = 0; i < vl; i++) out[nl + i] = kHpackStaticBlob[kHpackStaticValue[index - 1][0] + i];
        return true;
    }
    if (index >= 62 && index - 62 < h.count) {
        const uint32_t e = (h.head + (index - 62)) & 127u;
        nl = h.meta[e].nl; vl = with_value ? h.meta[e].vl : 0;
        if (nl + vl > cap) { overflow = true; return false; }
        const uint32_t off = h.meta[e].off, nb = nl + vl;
        if (off + nb <= 4096u) {                                      // the entry does not wrap the ring: word copies
            uint32_t i = 0;
            for (; i + 4 <= nb; i += 4) { const uint32_t wv = ld32_any(h.bytes + off + i); out[i] = (uint8_t)wv; out[i + 1] = (uint8_t)(wv >> 8); out[i + 2] = (uint8_t)(wv >> 16); out[i + 3] = (uint8_t)(wv >> 24); }
            for (; i < nb; i++) out[i] = h.bytes[off + i];
        } else for (uint32_t i = 0; i < nb; i++) out[i] = h.bytes[(off + i) & 4095u];
        return true;
    }
    return false;
}
// HPacker::Decode (hpack.cpp:765-843): ONE field at p[0..left).  The record bytes (name then value) land in rec.
// rc > 0: a field was produced, `adv` bytes consumed; rc == 0: ran out of bytes inside an indexed field / size update
// (the iterator is then at the end: the bytes are swallowed, as in the reference); -1 malformed; -2 rec too small.
__device__ __forceinline__ int hpack_decode_field(HpackState& h, const uint8_t* p, uint32_t left, uint8_t* rec, uint32_t cap,
                                                  uint32_t& nl, uint32_t& vl, uint32_t& adv) {
    const uint8_t* p0 = p;
    nl = vl = 0; adv = 0;
    // (001x) dynamic table size updates precede the field they travel with
    while (left && (p[0] >> 5) == 1) {
        uint32_t max_size = 0;
        const int ib = hp_int(p, left, 5, max_size);
        if (ib <= 0) return ib;
        if (max_size > 4096) return -1;
        if (max_size > h.max_size) h.max_size = max_size;
        else if (max_size < h.max_size) { h.max_size = max_size; while (h.size > h.max_size) hp_pop(h); }
        p += ib; left -= (uint32_t)ib;
    }
    if (!left) return 0;
    const uint8_t fb = p[0];
    uint32_t index = 0;
    bool ovf = false;
    if (fb & 0x80) {                                     // indexed field
        const int ib = hp_int(p, left, 7, index);
        if (ib <= 0) return ib;
        if (!hp_copy_indexed(h, index, true, rec, cap, nl, vl, ovf)) return ovf ? -2 : -1;
        p += ib;
    } else {
        const bool incremental = (fb >> 6) == 1;
        const int ib = hp_int(p, left, incremental ? 6 : 4, index);
        if (ib <= 0) return -1;
        uint32_t used = (uint32_t)ib;
        if (index != 0) {
            if (!hp_copy_indexed(h, index, false, rec, cap, nl, vl, ovf)) return ovf ? -2 : -1;
        } else {
            const int nb = hp_str(p + used, left - used, rec, cap, nl);
            if (nb <= 0) return nb == -2 ? -2 : -1;
            used += (uint32_t)nb;
            for (uint32_t i = 0; i < nl; i++) if (rec[i] >= 'A' && rec[i] <= 'Z') rec[i] = (uint8_t)(rec[i] + 32);
        }
        const int vb = hp_str(p + used, left - used, rec + nl, cap - nl, vl);
        if (vb <= 0) return vb == -2 ? -2 : -1;
        used += (uint32_t)vb;
        if (incremental && hp_add(h, rec, nl, vl) != 0) return -1;
        p += used;
    }
    adv = (uint32_t)(p - p0);
    return 1;
}
// One header block, the way ConsumeHeaders loops HPacker::Decode.  Records: u16 name_len, u16 value_len, name, value.
// status: 0 consumed, 1 ran out of bytes inside a field, -1 malformed, -2 output capacity exceeded
__device__ __noinline__ int hpack_decode_block(HpackState& h, const uint8_t* in, uint32_t n, uint8_t* out, uint32_t out_cap,
                                               uint32_t& out_len, uint32_t& n_headers) {
    uint32_t pos = 0, o = 0, cnt = 0;
    int status = 0;
    while (pos < n) {
        if (o + 4 > out_cap) { status = -2; break; }
        uint32_t nl = 0, vl = 0, adv = 0;
        const int rc = hpack_decode_field(h, in + pos, n - pos, out + o + 4, out_cap - o - 4, nl, vl, adv);
        if (rc <= 0) { status = rc == 0 ? 1 : rc; break; }
        out[o] = (uint8_t)nl; out[o + 1] = (uint8_t)(nl >> 8); out[o + 2] = (uint8_t)vl; out[o + 3] = (uint8_t)(vl >> 8);
        o += 4 + nl + vl; cnt++;
        pos += adv;
    }
    out_len = o; n_headers = cnt;
    return status;
}

struct H2Frame { uint8_t type, flags; uint16_t pad; uint32_t stream_id, payload_off, payload_len; };   // == b2_h2_frame

// blocks [first[g], first[g+1]) belong to one connection and are decoded in order by one thread
__global__ void k_hpack_decode(const uint8_t* bytes, const uint32_t* blk_conn, const uint32_t* blk_off, const uint32_t* blk_len,
                               const uint32_t* group_first, uint32_t n_groups, HpackState* states, uint8_t* out, uint32_t per_block_cap,
                               uint32_t* out_lens, int32_t* status, uint32_t* n_headers) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    for (uint32_t b = group_first[g]; b < group_first[g + 1]; b++) {
        uint32_t ol = 0, nh = 0;
        const int st = hpack_decode_block(states[blk_conn[b]], bytes + blk_off[b], blk_len[b], out + (size_t)b * per_block_cap, per_block_cap, ol, nh);
        out_lens[b] = ol; status[b] = st; n_headers[b] = nh;
    }
}
__global__ void k_hpack_reset(HpackState* states, uint32_t conn, uint32_t max_size) {
    HpackState& h = states[conn];
    h.max_size = max_size; h.size = 0; h.count = 0; h.head = 0; h.byte_head = 0;
}

// one thread per connection run: the chain of 9-byte frame heads
__global__ void k_h2_scan(const uint8_t* bytes, const b2_run* runs, uint32_t n_runs, uint32_t max_frame_size, H2Frame* frames,
                          uint32_t cap_per_run, uint32_t* n_frames, uint32_t* consumed, uint32_t* err) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint8_t* in = bytes + runs[r].offset; const uint32_t n = runs[r].length;
    uint32_t pos = 0, cnt = 0, e = B2_PARSE_ERROR_NOT_ENOUGH_DATA;
    if (runs[r].flags & 2u) {                               // server side, connection start: the 24-byte client preface
        const char* pre = "PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n";
        const uint32_t k = n < 24 ? n : 24;
        bool match = true;
        for (uint32_t i = 0; i < k; i++) if (in[i] != (uint8_t)pre[i]) { match = false; break; }
        if (!match) { n_frames[r] = 0; consumed[r] = 0; err[r] = B2_PARSE_ERROR_TRY_OTHERS; return; }
        if (n < 24) { n_frames[r] = 0; consumed[r] = 0; err[r] = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return; }
        pos = 24;
    }
    H2Frame* out = frames + (size_t)r * cap_per_run;
    for (;;) {
        if (n - pos < 3) break;
        const uint32_t length = ((uint32_t)in[pos] << 16) | ((uint32_t)in[pos + 1] << 8) | in[pos + 2];
        if (length > max_frame_size) { e = B2_PARSE_ERROR_ABSOLUTELY_WRONG; break; }
        if ((unsigned long long)(n - pos - 3) < 6ull + length) break;
        const uint32_t sid = load_be32(in + pos + 5);
        if (sid & 0x80000000u) { e = B2_PARSE_ERROR_ABSOLUTELY_WRONG; break; }
        if (cnt < cap_per_run) {
            H2Frame f; f.type = in[pos + 3]; f.flags = in[pos + 4]; f.pad = 0; f.stream_id = sid;
            f.payload_off = runs[r].offset + pos + 9; f.payload_len = length;
            out[cnt] = f;
        }
        cnt++; pos += 9 + length;
    }
    n_frames[r] = cnt; consumed[r] = pos; err[r] = e;
}

// ---------------------------------------------------------------------------------------------------------
// The server side of ParseH2Message: one thread per connection run walks H2Context::Consume
// (policy/http2_rpc_protocol.cpp:467-543) frame by frame.  A connection is a serial state machine (HPACK table,
// settings, windows, pending streams), so connections are the unit of parallelism, exactly like the reference
// runs one input bthread per socket.  Every quirk of the reference that shapes the byte stream is kept: handlers
// that fail (or PING acks) leave the rest of their payload unread and the next "frame head" is parsed from there.
constexpr uint32_t kH2HdrBytes = B2_H2_HEADER_BYTES;
constexpr long long kH2MaxWindow = 2147483647ll;                 // H2Settings::MAX_WINDOW_SIZE
// n bytes src -> dst by ONE thread: 16-byte words when the pointers agree mod 16, else 4-byte words assembled from
// aligned loads (a connection is a serial state machine; its bulk copies are the only place worth widening)
__device__ __forceinline__ void thread_copy(uint8_t* dst, const uint8_t* src, uint32_t n) {
    uint32_t i = 0;
    if ((((uintptr_t)dst ^ (uintptr_t)src) & 15u) == 0) {
        while (i < n && ((uintptr_t)(dst + i) & 15u)) { dst[i] = src[i]; i++; }
        for (; i + 64 <= n; i += 64) {
            const uint4 a = *reinterpret_cast<const uint4*>(src + i), b = *reinterpret_cast<const uint4*>(src + i + 16);
            const uint4 c = *reinterpret_cast<const uint4*>(src + i + 32), d = *reinterpret_cast<const uint4*>(src + i + 48);
            *reinterpret_cast<uint4*>(dst + i) = a; *reinterpret_cast<uint4*>(dst + i + 16) = b;
            *reinterpret_cast<uint4*>(dst + i + 32) = c; *reinterpret_cast<uint4*>(dst + i + 48) = d;
        }
        for (; i + 16 <= n; i += 16) *reinterpret_cast<uint4*>(dst + i) = *reinterpret_cast<const uint4*>(src + i);
    } else {
        while (i < n && ((uintptr_t)(dst + i) & 3u)) { dst[i] = src[i]; i++; }
        const uint32_t sh = 8u * (uint32_t)((uintptr_t)(src + i) & 3u);
        if (i + 8 <= n) {
            const uint32_t* q = reinterpret_cast<const uint32_t*>((uintptr_t)(src + i) & ~(uintptr_t)3);
            uint32_t w0 = q[0];
            for (; i + 8 <= n; i += 4) {                         // (+8: the look-ahead word stays inside the source)
                const uint32_t w1 = *++q;
                *reinterpret_cast<uint32_t*>(dst + i) = sh ? __funnelshift_r(w0, w1, sh) : w0;
                w0 = w1;
            }
        }
    }
    for (; i < n; i++) dst[i] = src[i];
}
struct H2Stream {
    int32_t id; uint32_t hdr_len, n_headers, body_len;
    uint32_t stream_ended, body_input_off;                       // body_input_off: the whole body is one DATA payload of THIS batch (0 = it lives in the slot)
    long long remote_window_left, deferred_wu;
};
struct H2Conn {
    uint32_t conn_state; int32_t last_received_stream_id; uint32_t remote_settings_received, n_pending;
    uint32_t r_header_table_size, r_enable_push, r_max_concurrent_streams, r_stream_window_size, r_max_frame_size, r_max_header_list_size;
    uint32_t l_stream_window_size, l_max_frame_size;
    long long remote_window_left, deferred_window_update;
    long long last_sent_stream_id; uint32_t preface_sent, pad0;  // client side: H2Context::_last_sent_stream_id (:331); the preface goes out with the first request
    HpackState enc;                                              // HPacker::_encode_table (responses)
};
// Pending streams live outside H2Conn so that their number and size are run-time choices (b2_h2_configure): connection i
// owns streams[i * pending ...] and slots[(i * pending + k) * stream_bytes ...]: [0, kH2HdrBytes) header records, then the body.
struct H2Pool { H2Stream* streams; uint8_t* slots; uint32_t pending, stream_bytes; };
struct H2Out {                      // this run's slice of the output buffer
    uint8_t* base; uint32_t ctrl_cap, ctrl_len, blob_off, blob_end; bool overflow;
};
__device__ __forceinline__ void h2_conn_init(H2Conn& c, H2Stream* S, uint32_t P) {
    c.conn_state = 0; c.last_received_stream_id = -1; c.remote_settings_received = 0; c.n_pending = 0;
    // _remote_settings: H2Settings() with the windows maximised (H2Context ctor, :323-345)
    c.r_header_table_size = 4096; c.r_enable_push = 0; c.r_max_concurrent_streams = 0xffffffffu;
    c.r_stream_window_size = (uint32_t)kH2MaxWindow; c.r_max_frame_size = 16384; c.r_max_header_list_size = 0xffffffffu;
    c.l_stream_window_size = 256 * 1024; c.l_max_frame_size = 16384;     // H2Settings() defaults, http2.cpp:26-34
    c.remote_window_left = kH2MaxWindow; c.deferred_window_update = 0;
    c.last_sent_stream_id = 1; c.preface_sent = 0; c.pad0 = 0;
    for (uint32_t i = 0; i < P; i++) S[i].id = -1;
    c.enc.max_size = 4096; c.enc.size = 0; c.enc.count = 0; c.enc.head = 0; c.enc.byte_head = 0;   // _hpacker.Init(header_table_size), :367
}
__device__ __forceinline__ void h2_put_head(uint8_t* p, uint32_t payload, uint8_t type, uint8_t flags, uint32_t sid) {   // SerializeFrameHead :123-136
    p[0] = (uint8_t)(payload >> 16); p[1] = (uint8_t)(payload >> 8); p[2] = (uint8_t)payload; p[3] = type; p[4] = flags;
    p[5] = (uint8_t)(sid >> 24); p[6] = (uint8_t)(sid >> 16); p[7] = (uint8_t)(sid >> 8); p[8] = (uint8_t)sid;
}
__device__ __forceinline__ uint8_t* h2_ack_room(H2Out& o, uint32_t n) {                  // WriteAck :144-150
    if (o.ctrl_len + n > o.ctrl_cap) { o.overflow = true; return nullptr; }
    uint8_t* p = o.base + o.ctrl_len; o.ctrl_len += n; return p;
}
__device__ __forceinline__ void h2_write_wu(H2Out& o, uint32_t sid, long long inc) {
    uint8_t* p = h2_ack_room(o, 13); if (!p) return;
    h2_put_head(p, 4, 8, 0, sid); put_be32(p + 9, (uint32_t)inc);
}
// AddWindowSize (:261-281), literally: the sum is stored even when the check fails
__device__ __forceinline__ bool h2_add_window(long long& w, long long diff) {
    const long long before = w; w = before + diff;
    const long long mask = (long long)(int)0x80000000;            // `(1 << 31)` promoted to int64
    if ((((before | diff) >> 31) & 1) == 0) { if ((before + diff) & mask) return false; }
    if ((((before & diff) >> 31) & 1) == 1) { if (((before + diff) & mask) == 0) return false; }
    return true;
}
__device__ __forceinline__ void h2_defer_wu(H2Conn& c, H2Out& o, long long size) {         // H2Context::DeferWindowUpdate :1078-1094
    if (size <= 0) return;
    c.deferred_window_update += size;
    if (c.deferred_window_update >= (long long)(c.l_stream_window_size / 2)) {
        const long long conn_wu = c.deferred_window_update; c.deferred_window_update = 0;
        if (conn_wu > 0) h2_write_wu(o, 0, conn_wu);
    }
}
__device__ __forceinline__ int h2_find(const H2Stream* S, uint32_t P, int32_t id) {
    for (uint32_t i = 0; i < P; i++) if (S[i].id == id) return (int)i;
    return -1;
}
// RemoveStreamAndDeferWU (:378-392); returns the slot (the caller still reads the stream's data) or -1
__device__ __forceinline__ int h2_remove_stream(H2Conn& c, H2Stream* S, uint32_t P, H2Out& o, int32_t id) {
    const int k = h2_find(S, P, id);
    if (k < 0) return -1;
    S[k].id = -1; c.n_pending--;
    const long long d = S[k].deferred_wu; S[k].deferred_wu = 0;
    h2_defer_wu(c, o, d);
    return k;
}
__device__ __forceinline__ bool ci_eq(const uint8_t* a, uint32_t n, const char* lit) {    // strcasecmp(a (c_str of n bytes), lit) == 0
    uint32_t i = 0;
    for (; lit[i]; i++) {
        if (i >= n) return false;
        uint8_t x = a[i]; if (x >= 'a' && x <= 'z') x = (uint8_t)(x - 32);
        if (x != (uint8_t)lit[i]) return false;
    }
    return i == n;
}
__device__ __forceinline__ uint32_t cstr_len(const uint8_t* p, uint32_t n) {           // strnlen: four bytes per step
    uint32_t i = 0;
    for (; i + 4 <= n; i += 4) {
        const uint32_t z = __vcmpeq4(ld32_any(p + i), 0u);
        if (z) return i + ((__ffs(z) - 1) >> 3);
    }
    while (i < n && p[i]) i++;
    return i;
}
__device__ __forceinline__ bool lit_eq(const uint8_t* a, uint32_t n, const char* lit) {   // strcmp(c_str, lit) == 0
    uint32_t i = 0;
    for (; lit[i]; i++) if (i >= n || a[i] != (uint8_t)lit[i]) return false;
    return i == n;
}
__device__ __forceinline__ bool has_prefix(const uint8_t* a, uint32_t n, const char* lit, uint32_t& l) {
    l = 0; while (lit[l]) { if (l >= n || a[l] != (uint8_t)lit[l]) return false; l++; }
    return true;
}
// Str2HttpMethod (http_method.cpp:104-140): case-insensitive exact match of the c_str against the 27 names
__device__ __forceinline__ int h2_http_method(const uint8_t* v, uint32_t vl) {
    const uint32_t n = cstr_len(v, vl);
    const char* const names[27] = { "DELETE", "GET", "HEAD", "POST", "PUT", "CONNECT", "OPTIONS", "TRACE", "COPY", "LOCK", "MKCOL", "MOVE",
        "PROPFIND", "PROPPATCH", "SEARCH", "UNLOCK", "REPORT", "MKACTIVITY", "CHECKOUT", "MERGE", "M-SEARCH", "NOTIFY", "SUBSCRIBE",
        "UNSUBSCRIBE", "PATCH", "PURGE", "MKCALENDAR" };
    for (int m = 0; m < 27; m++) if (ci_eq(v, n, names[m])) return m;
    return -1;
}
// ParseContentType (policy/http_rpc_protocol.cpp:176-230)
__device__ __forceinline__ uint32_t h2_content_type(const uint8_t* ct, uint32_t n, bool& is_grpc) {
    is_grpc = false;
    uint32_t l;
    if (!has_prefix(ct, n, "application/", l)) return 0;
    ct += l; n -= l;
    if (has_prefix(ct, n, "grpc", l)) {
        if (n == 4 || ct[4] == ';') { is_grpc = true; return 2; }
        else if (ct[4] == '+') { ct += 5; n -= 5; is_grpc = true; }
    }
    uint32_t type;
    if (has_prefix(ct, n, "json", l)) type = 1;
    else if (has_prefix(ct, n, "proto-json", l)) type = 4;
    else if (has_prefix(ct, n, "proto-text", l)) type = 3;
    else if (has_prefix(ct, n, "proto", l)) type = 2;
    else if (has_prefix(ct, n, "x-protobuf", l)) type = 2;
    else return 0;
    ct += l; n -= l;
    return (n == 0 || ct[0] == ';') ? type : 0;
}
// one header of ConsumeHeaders (:1232-1287): false = the reference returns -1
__device__ __forceinline__ bool h2_check_header(const uint8_t* name, uint32_t nl, const uint8_t* value, uint32_t vl) {
    const uint32_t n = cstr_len(name, nl);
    if (n == 0 || name[0] != ':') return true;
    const uint8_t c1 = n > 1 ? name[1] : 0;
    const uint8_t* rest = name + 2; const uint32_t rn = n > 2 ? n - 2 : 0;
    switch (c1) {
    case 'a': return lit_eq(rest, rn, "uthority");
    case 'm': return lit_eq(rest, rn, "ethod") && h2_http_method(value, vl) >= 0;
    case 'p': return lit_eq(rest, rn, "ath");
    case 's':
        if (lit_eq(rest, rn, "cheme")) return true;
        if (lit_eq(rest, rn, "tatus")) {                 // strtol(value, &end, 10) must stop at the terminating NUL
            const uint32_t m = cstr_len(value, vl);
            uint32_t i = 0;
            while (i < m && (value[i] == ' ' || (value[i] >= 9 && value[i] <= 13))) i++;
            uint32_t j = i;
            if (j < m && (value[j] == '+' || value[j] == '-')) j++;
            uint32_t d = j; while (d < m && value[d] >= '0' && value[d] <= '9') d++;
            const uint32_t end = d > j ? d : 0;          // no digits: endptr = nptr
            return end == m;
        }
        return false;
    default: return false;
    }
}
struct H2Res { int kind; uint32_t err; int32_t err_stream; int slot; };   // kind 0 ok, 1 ok + message in `slot`, 2 error
__device__ __forceinline__ H2Res h2_ok() { H2Res r; r.kind = 0; r.err = 0; r.err_stream = 0; r.slot = -1; return r; }
__device__ __forceinline__ H2Res h2_err(uint32_t e, int32_t sid = 0) { H2Res r; r.kind = 2; r.err = e; r.err_stream = sid; r.slot = -1; return r; }

// H2StreamContext::ConsumeHeaders over one fragment, records appended to the stream's slot
__device__ __forceinline__ int h2_consume_headers(H2Conn& c, HpackState& hp, H2Stream& st, uint8_t* slot, const uint8_t* frag, uint32_t n, bool& no_room) {
    uint32_t pos = 0;
    while (pos < n) {
        if (st.hdr_len + 4 > kH2HdrBytes) { no_room = true; return -1; }
        uint8_t* rec = slot + st.hdr_len;
        uint32_t nl = 0, vl = 0, adv = 0;
        const int rc = hpack_decode_field(hp, frag + pos, n - pos, rec + 4, kH2HdrBytes - st.hdr_len - 4, nl, vl, adv);
        if (rc == -2) { no_room = true; return -1; }
        if (rc < 0) return -1;
        if (rc == 0) break;
        if (!h2_check_header(rec + 4, nl, rec + 4 + nl, vl)) return -1;
        rec[0] = (uint8_t)nl; rec[1] = (uint8_t)(nl >> 8); rec[2] = (uint8_t)vl; rec[3] = (uint8_t)(vl >> 8);
        st.hdr_len += 4 + nl + vl; st.n_headers++;
        pos += adv;
    }
    return 0;
}
// OnEndStream (:823-846): the stream leaves the pending map; the caller emits the message from its slot
__device__ __forceinline__ H2Res h2_end_stream(H2Conn& c, H2Stream* S, uint32_t P, H2Out& o, int32_t id) {
    const int k = h2_remove_stream(c, S, P, o, id);
    if (k < 0) return h2_ok();
    H2Res r = h2_ok(); r.kind = 1; r.slot = k; r.err_stream = id; return r;
}

__global__ void k_h2_conn_reset(H2Conn* conns, HpackState* hps, uint32_t conn, H2Pool pool) {
    h2_conn_init(conns[conn], pool.streams + (size_t)conn * pool.pending, pool.pending);
    HpackState& h = hps[conn]; h.max_size = 4096; h.size = 0; h.count = 0; h.head = 0; h.byte_head = 0;
}

__global__ void k_h2_consume(const uint8_t* bytes, const b2_run* runs, uint32_t n_runs, H2Conn* conns, HpackState* hps,
                             const DevMethod* methods, uint32_t n_methods, b2_h2_run_status* rs, b2_h2_msg* msgs, uint32_t msg_cap_per_run,
                             uint8_t* out, uint32_t region, H2Pool pool) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    const uint32_t P = pool.pending, kH2StreamBytes = pool.stream_bytes;
    H2Stream* const S = pool.streams + (size_t)(uint32_t)runs[r].socket_id * P;
    uint8_t* const slots = pool.slots + (size_t)(uint32_t)runs[r].socket_id * P * kH2StreamBytes;
    const uint32_t run_off = runs[r].offset;
    const uint8_t* in = bytes + run_off; const uint32_t n = runs[r].length;
    H2Conn& c = conns[(uint32_t)runs[r].socket_id];
    HpackState& hp = hps[(uint32_t)runs[r].socket_id];
    H2Out o; o.base = out + (size_t)r * region; o.ctrl_cap = region / 4; o.ctrl_len = 0; o.blob_off = region / 4; o.blob_end = region; o.overflow = false;
    b2_h2_msg* mout = msgs + (size_t)r * msg_cap_per_run;
    uint32_t n_msgs = 0, pos = 0, last_ok = 0, perr = B2_PARSE_ERROR_NOT_ENOUGH_DATA;
    bool no_room = false;
    for (;;) {
        if (o.overflow || no_room) { perr = B2_PARSE_ERROR_NO_RESOURCE; break; }
        if (c.conn_state == 0) {                                     // H2_CONNECTION_UNINITIALIZED, server side (:469-489)
            const char* pre = "PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n";
            const uint32_t k = (n - pos) < 24 ? (n - pos) : 24;
            bool match = true;
            for (uint32_t i = 0; i < k; i++) if (in[pos + i] != (uint8_t)pre[i]) { match = false; break; }
            if (!match) { perr = B2_PARSE_ERROR_TRY_OTHERS; break; }
            if (k < 24) break;
            c.conn_state = 1; pos += 24;
            // SerializeH2SettingsFrameAndWU of the default server settings (:230-259): ENABLE_PUSH=0, INITIAL_WINDOW_SIZE=256K, WU 1M-65535
            uint8_t* p = h2_ack_room(o, 9 + 12 + 13);
            if (p) {
                h2_put_head(p, 12, 4, 0, 0);
                p[9] = 0; p[10] = 2; put_be32(p + 11, 0);
                p[15] = 0; p[16] = 4; put_be32(p + 17, c.l_stream_window_size);
                h2_put_head(p + 21, 4, 8, 0, 0); put_be32(p + 30, 1024 * 1024 - 65535);
            }
            last_ok = pos;
            continue;
        }
        // ---- ConsumeFrameHead (:438-465)
        const uint32_t left = n - pos;
        if (left < 3) break;
        const uint32_t length = ((uint32_t)in[pos] << 16) | ((uint32_t)in[pos + 1] << 8) | in[pos + 2];
        if (length > c.l_max_frame_size) { perr = B2_PARSE_ERROR_ABSOLUTELY_WRONG; break; }
        if ((unsigned long long)(left - 3) < 6ull + length) break;
        const uint32_t type = in[pos + 3], flags = in[pos + 4], sid_raw = load_be32(in + pos + 5);
        if (sid_raw & 0x80000000u) { perr = B2_PARSE_ERROR_ABSOLUTELY_WRONG; break; }
        const int32_t sid = (int32_t)sid_raw;
        pos += 9;
        if (type > 9) { perr = B2_PARSE_ERROR_ABSOLUTELY_WRONG; break; }          // FindFrameHandler == NULL (:498-502)
        const uint8_t* pl = in + pos;                                // payload; handlers advance `used`
        uint32_t used = 0;
        H2Res res = h2_ok();
        switch (type) {
        case 0: {                                                    // ---- OnData (:700-723) + H2StreamContext::OnData (:725-779)
            uint32_t frag = length, padl = 0;
            if ((flags & 0x8) && length == 0) { res = h2_err(6); break; }   // no room for the pad-length byte (the reference would read past the frame)
            if (flags & 0x8) { frag--; padl = pl[used++]; }
            if (frag < padl) { res = h2_err(6); break; }
            frag -= padl;
            const int k = h2_find(S, P, sid);
            if (k < 0) {
                // stream unknown: the bytes are still counted against the connection window, then STREAM_CLOSED
                used += frag + padl;
                const long long acc = (long long)frag;
                const long long quota = (long long)(c.l_stream_window_size / (c.n_pending + 1));
                long long tmp_deferred = (long long)frag;
                if (acc >= quota) {
                    if (acc > (long long)c.l_stream_window_size) { h2_defer_wu(c, o, tmp_deferred); res = h2_err(5, sid); break; }   // (inner FLOW_CONTROL result is discarded)
                    const long long swu = tmp_deferred; tmp_deferred = 0;
                    if (swu > 0) { h2_write_wu(o, (uint32_t)sid, swu); const long long cw = swu + c.deferred_window_update; c.deferred_window_update = 0; h2_write_wu(o, 0, cw); }
                }
                h2_defer_wu(c, o, tmp_deferred);
                res = h2_err(5, sid);
                break;
            }
            H2Stream& st = S[k];
            if (st.body_len == 0 && (flags & 0x1) && frag) {
                // the usual unary call: one DATA frame that also ends the stream — the body stays where it is in the batch
                st.body_input_off = run_off + pos + used; st.body_len = frag;
            } else {
                if (kH2HdrBytes + st.body_len + frag > kH2StreamBytes) { no_room = true; break; }
                thread_copy(slots + (size_t)k * kH2StreamBytes + kH2HdrBytes + st.body_len, pl + used, frag);
                st.body_len += frag;
            }
            used += frag + padl;
            const long long acc = (long long)frag + st.deferred_wu; st.deferred_wu += frag;
            const long long quota = (long long)(c.l_stream_window_size / (c.n_pending + 1));
            if (acc >= quota) {
                if (acc > (long long)c.l_stream_window_size) { res = h2_err(3, sid); break; }
                const long long swu = st.deferred_wu; st.deferred_wu = 0;
                if (swu > 0) { h2_write_wu(o, (uint32_t)sid, swu); const long long cw = swu + c.deferred_window_update; c.deferred_window_update = 0; h2_write_wu(o, 0, cw); }
            }
            if (flags & 0x1) res = h2_end_stream(c, S, P, o, sid);
            break; }
        case 1: {                                                    // ---- OnHeaders (:545-613) + H2StreamContext::OnHeaders (:615-655)
            if (sid == 0) { res = h2_err(1); break; }
            const bool has_padding = flags & 0x8, has_priority = flags & 0x20;
            if (length < (has_priority ? 5u : 0u) + (has_padding ? 1u : 0u)) { res = h2_err(6); break; }
            uint32_t frag = length, padl = 0;
            if (has_padding) { padl = pl[used++]; frag--; }
            if (has_priority) { used += 5; frag -= 5; }
            if (frag < padl) { res = h2_err(6); break; }
            frag -= padl;
            int k;
            if (sid > c.last_received_stream_id) {                   // new stream
                if ((sid & 1) == 0) { res = h2_err(1); break; }
                c.last_received_stream_id = sid;
                k = h2_find(S, P, -1);
                if (k < 0) { no_room = true; break; }                // (device limit: B2_H2_MAX_PENDING)
                H2Stream& st = S[k];
                st.id = sid; st.hdr_len = 0; st.n_headers = 0; st.body_len = 0; st.stream_ended = 0; st.deferred_wu = 0; st.body_input_off = 0;
                st.remote_window_left = (long long)c.r_stream_window_size;
                c.n_pending++;
            } else {
                k = h2_find(S, P, sid);
                if (k < 0) { res = h2_err(1); break; }
            }
            H2Stream& st = S[k];
            if (h2_consume_headers(c, hp, st, slots + (size_t)k * kH2StreamBytes, pl + used, frag, no_room) < 0) { if (!no_room) res = h2_err(1); break; }
            used += frag + padl;
            if (flags & 0x4) { if (flags & 0x1) res = h2_end_stream(c, S, P, o, sid); }
            else if (flags & 0x1) st.stream_ended = 1;
            break; }
        case 2: res = h2_err(1); break;                              // OnPriority (:917-921)
        case 3: {                                                    // ---- OnResetStream (:781-821)
            if (length != 4) { res = h2_err(6); break; }
            used += 4;
            (void)h2_remove_stream(c, S, P, o, sid);                       // server side: the stream is dropped, no message
            break; }
        case 4: {                                                    // ---- OnSettings (:848-915)
            if (sid != 0) { res = h2_err(1); break; }
            if (flags & 0x1) { if (length != 0) res = h2_err(1); break; }
            const long long old_sw = (long long)c.r_stream_window_size;
            uint32_t t_hts, t_push, t_mcs, t_sws, t_mfs, t_mhl;
            if (!c.remote_settings_received) { t_hts = 4096; t_push = 0; t_mcs = 0xffffffffu; t_sws = 256 * 1024; t_mfs = 16384; t_mhl = 0xffffffffu; }
            else { t_hts = c.r_header_table_size; t_push = c.r_enable_push; t_mcs = c.r_max_concurrent_streams; t_sws = c.r_stream_window_size; t_mfs = c.r_max_frame_size; t_mhl = c.r_max_header_list_size; }
            bool okp = (length / 6) * 6 == length;                   // ParseH2Settings (:166-211)
            if (okp) for (uint32_t i = 0; i < length / 6; i++) {
                const uint32_t id = ((uint32_t)pl[used] << 8) | pl[used + 1], value = load_be32(pl + used + 2);
                used += 6;
                if (id == 1) t_hts = value;
                else if (id == 2) { if (value > 1) { okp = false; break; } t_push = value; }
                else if (id == 3) t_mcs = value;
                else if (id == 4) { if (value > (uint32_t)kH2MaxWindow) { okp = false; break; } t_sws = value; }
                else if (id == 5) { if (value > 16777215u || value < 16384u) { okp = false; break; } t_mfs = value; }
                else if (id == 6) t_mhl = value;
            }
            if (!c.remote_settings_received) {
                if (!okp) { res = h2_err(1); break; }                // parsed into a temporary: nothing is kept
                c.remote_window_left -= (kH2MaxWindow - 65535);
                c.remote_settings_received = 1;
            }
            // (after the first frame the reference parses in place: fields set before a bad pair stay)
            c.r_header_table_size = t_hts; c.r_enable_push = t_push; c.r_max_concurrent_streams = t_mcs;
            c.r_stream_window_size = t_sws; c.r_max_frame_size = t_mfs; c.r_max_header_list_size = t_mhl;
            if (!okp) { res = h2_err(1); break; }
            const long long diff = (long long)c.r_stream_window_size - old_sw;
            bool flow_ok = true;
            if (diff) for (uint32_t i = 0; i < P; i++) if (S[i].id >= 0) { if (!h2_add_window(S[i].remote_window_left, diff)) { flow_ok = false; break; } }
            if (!flow_ok) { res = h2_err(3); break; }
            uint8_t* p = h2_ack_room(o, 9); if (p) h2_put_head(p, 0, 4, 1, 0);
            break; }
        case 5: res = h2_err(1); break;                              // OnPushPromise (:923-927)
        case 6: {                                                    // ---- OnPing (:929-951)
            if (length != 8) { res = h2_err(6); break; }
            if (sid != 0) { res = h2_err(1); break; }
            if (flags & 0x1) break;                                  // (an ack's payload is left unread, as in the reference)
            uint8_t* p = h2_ack_room(o, 17);
            if (p) { h2_put_head(p, 8, 6, 1, 0); for (uint32_t i = 0; i < 8; i++) p[9 + i] = pl[i]; }
            used += 8;
            break; }
        case 7: {                                                    // ---- OnGoAway (:958-1004), server side: ignored
            if (length < 8) { res = h2_err(6); break; }
            if (sid != 0) { res = h2_err(1); break; }
            if (flags) { res = h2_err(1); break; }
            used += length;
            break; }
        case 8: {                                                    // ---- OnWindowUpdate (:1006-1041)
            if (length != 4) { res = h2_err(6); break; }
            const uint32_t inc = load_be32(pl); used += 4;
            if ((inc & 0x80000000u) || inc == 0) { res = h2_err(1); break; }
            if (sid == 0) { if (!h2_add_window(c.remote_window_left, (long long)inc)) res = h2_err(3); break; }
            const int k = h2_find(S, P, sid);
            if (k < 0) break;
            if (!h2_add_window(S[k].remote_window_left, (long long)inc)) res = h2_err(3);
            break; }
        case 9: {                                                    // ---- OnContinuation (:657-698)
            const int k = h2_find(S, P, sid);
            if (k < 0) { res = h2_err(1); break; }
            H2Stream& st = S[k];
            used += length;                                          // the payload moves into _remaining_header_fragment first
            if (h2_consume_headers(c, hp, st, slots + (size_t)k * kH2StreamBytes, pl, length, no_room) < 0) { if (!no_room) res = h2_err(1); break; }
            if ((flags & 0x4) && st.stream_ended) res = h2_end_stream(c, S, P, o, sid);
            break; }
        }
        if (no_room) continue;
        pos += used;
        if (res.kind == 2) {
            if (res.err_stream) {                                    // RST_STREAM, then the stream is forgotten (:507-527)
                uint8_t* p = h2_ack_room(o, 13);
                if (p) { h2_put_head(p, 4, 3, 0, (uint32_t)res.err_stream); put_be32(p + 9, res.err); }
                (void)h2_remove_stream(c, S, P, o, res.err_stream);
            } else {                                                 // GOAWAY (:528-538); parsing goes on
                uint8_t* p = h2_ack_room(o, 17);
                if (p) { h2_put_head(p, 8, 7, 0, 0); put_be32(p + 9, (uint32_t)c.last_received_stream_id); put_be32(p + 13, res.err); }
            }
            last_ok = pos;
            continue;
        }
        last_ok = pos;
        if (res.kind == 1) {
            // ---- the completed request, as ProcessHttpRequest first sees it
            const H2Stream& st = S[res.slot];
            const uint8_t* slot = slots + (size_t)res.slot * kH2StreamBytes;
            const bool in_input = st.body_input_off != 0;
            const uint32_t need = ((st.hdr_len + 15u) & ~15u) + (in_input ? 0u : ((st.body_len + 15u) & ~15u));
            if (n_msgs >= msg_cap_per_run || o.blob_off + need > o.blob_end) { no_room = true; continue; }
            b2_h2_msg m;
            m.run_idx = r; m.stream_id = (uint32_t)res.err_stream; m.reserved = 0;
            const uint32_t ho = o.blob_off, bo = ho + ((st.hdr_len + 15u) & ~15u);
            thread_copy(o.base + ho, slot, st.hdr_len);
            if (!in_input) thread_copy(o.base + bo, slot + kH2HdrBytes, st.body_len);
            o.blob_off += need;
            const uint32_t gbase = r * region;
            m.headers_off = gbase + ho; m.headers_len = st.hdr_len; m.n_headers = st.n_headers;
            m.body_off = in_input ? st.body_input_off : gbase + bo; m.body_len = st.body_len;
            m.http_method = B2_H2_NO_METHOD; m.content_type = 0; m.flags = 0; m.method_idx = -1;
            m.msg_off = 0; m.msg_len = 0; m.path_off = 0; m.path_len = 0;
            if (in_input) m.flags |= B2_H2_FLAG_BODY_IN_INPUT;
            const uint8_t* body_p = in_input ? bytes + st.body_input_off : slot + kH2HdrBytes;
            bool is_grpc = false;
            const uint8_t* path = nullptr; uint32_t path_len = 0;
            for (uint32_t q = 0; q < st.hdr_len;) {
                const uint32_t nl = slot[q] | ((uint32_t)slot[q + 1] << 8), vl = slot[q + 2] | ((uint32_t)slot[q + 3] << 8);
                const uint8_t* nm = slot + q + 4; const uint8_t* v = nm + nl;
                const uint32_t cn = cstr_len(nm, nl);
                if (lit_eq(nm, cn, ":method")) m.http_method = (uint32_t)h2_http_method(v, vl);
                else if (lit_eq(nm, cn, ":path")) {                  // URI::SetH2Path (uri.cpp:403-425): up to '?' / '#'
                    uint32_t e = 0; while (e < vl && v[e] && v[e] != '?' && v[e] != '#') e++;
                    path = v; path_len = e; m.path_off = gbase + ho + (uint32_t)(v - slot); m.path_len = e; m.flags |= B2_H2_FLAG_HAS_PATH;
                } else if (lit_eq(nm, cn, "content-type")) m.content_type = h2_content_type(v, vl, is_grpc);
                q += 4 + nl + vl;
            }
            if (is_grpc) {
                m.flags |= B2_H2_FLAG_GRPC;
                // RemoveGrpcPrefix (policy/http_rpc_protocol.cpp:264-277)
                if (st.body_len == 0) { m.flags |= B2_H2_FLAG_GRPC_PREFIX_OK; m.msg_off = m.body_off; }
                else if (st.body_len >= 5) {
                    const uint8_t* b = body_p;
                    if (b[0]) m.flags |= B2_H2_FLAG_GRPC_COMPRESSED;
                    if ((unsigned long long)load_be32(b + 1) + 5ull == st.body_len) { m.flags |= B2_H2_FLAG_GRPC_PREFIX_OK; m.msg_off = m.body_off + 5; m.msg_len = st.body_len - 5; }
                }
            }
            if (path) {
                // FindMethodPropertyByURIImpl (:1088-1138), "[service]/[method]" form: '/'-separated, empty fields skipped
                uint32_t f0 = 0; while (f0 < path_len && path[f0] == '/') f0++;
                uint32_t e0 = f0; while (e0 < path_len && path[e0] != '/') e0++;
                uint32_t f1 = e0; while (f1 < path_len && path[f1] == '/') f1++;
                uint32_t e1 = f1; while (e1 < path_len && path[e1] != '/') e1++;
                if (e0 > f0 && e1 > f1) {
                    bool no_service = false;
                    m.method_idx = find_method(methods, n_methods, path + f0, e0 - f0, path + f1, e1 - f1, no_service);
                }
            }
            mout[n_msgs++] = m;
        }
    }
    b2_h2_run_status st; st.consumed = last_ok; st.parse_error = perr; st.n_msgs = n_msgs; st.first_msg = o.blob_off - region / 4;      // blob bytes used (the host turns this field into the list index)
    st.ctrl_off = r * region; st.ctrl_len = o.ctrl_len; st.remote_max_frame_size = c.r_max_frame_size; st.remote_stream_window_size = c.r_stream_window_size;
    rs[r] = st;
}

// ---------------------------------------------------------------------------------------------------------
// Response side: H2UnsentResponse::AppendAndDestroySelf (:1688-1750) + PackH2Message (:1310-1380), one thread per connection.
__device__ __forceinline__ uint8_t lc(uint8_t c) { return (c >= 'A' && c <= 'Z') ? (uint8_t)(c + 32) : c; }
__device__ __forceinline__ uint8_t* hp_put_int(uint8_t* p, uint8_t msb, uint32_t prefix, uint32_t value) {       // EncodeInteger :479-496
    const uint32_t lim = (1u << prefix) - 1;
    if (value < lim) { *p++ = (uint8_t)(msb | value); return p; }
    value -= lim; *p++ = (uint8_t)(msb | lim);
    for (; value >= 128;) { *p++ = (uint8_t)((value & 0x7f) | 0x80); value >>= 7; }
    *p++ = (uint8_t)value;
    return p;
}
// the encoder's view of "is this header / this name in a table": static first, then the connection's encode table;
// names compare case-insensitively, entries with an empty value are never full matches (IndexTable::AddHeader :165-171)
__device__ __forceinline__ uint32_t hp_enc_find(const HpackState& t, const uint8_t* n, uint32_t nl, const uint8_t* v, uint32_t vl, bool want_value) {
    for (uint32_t i = 0; i < 61; i++) {                          // reverse insertion => the smallest index wins for names
        if (kHpackStaticName[i][1] != nl) continue;
        if (want_value && (vl == 0 || kHpackStaticValue[i][1] != vl)) continue;
        bool eq = true;
        for (uint32_t k = 0; k < nl && eq; k++) eq = lc(n[k]) == lc(kHpackStaticBlob[kHpackStaticName[i][0] + k]);
        for (uint32_t k = 0; want_value && k < vl && eq; k++) eq = v[k] == kHpackStaticBlob[kHpackStaticValue[i][0] + k];
        if (eq) return i + 1;
    }
    for (uint32_t i = 0; i < t.count; i++) {                     // newest first == the latest id of a duplicated header
        const uint32_t e = (t.head + i) & 127u;
        if (t.meta[e].nl != nl) continue;
        if (want_value && (vl == 0 || t.meta[e].vl != vl)) continue;
        bool eq = true;
        for (uint32_t k = 0; k < nl && eq; k++) eq = lc(n[k]) == lc(t.bytes[(t.meta[e].off + k) & 4095u]);
        for (uint32_t k = 0; want_value && k < vl && eq; k++) eq = v[k] == t.bytes[(t.meta[e].off + nl + k) & 4095u];
        if (eq) return 62 + i;
    }
    return 0;
}
// HPacker::Encode (:696-726); hp_add wants name||value contiguous: `tmp` (>= nl + vl bytes) is scratch
__device__ __forceinline__ uint8_t* hp_encode(HpackState& t, uint8_t* p, const uint8_t* n, uint32_t nl, const uint8_t* v, uint32_t vl, bool never_index, uint8_t* tmp) {
    if (!never_index) {
        const uint32_t idx = hp_enc_find(t, n, nl, v, vl, true);
        if (idx) return hp_put_int(p, 0x80, 7, idx);
    }
    const uint32_t name_index = hp_enc_find(t, n, nl, nullptr, 0, false);
    if (!never_index) {
        for (uint32_t k = 0; k < nl; k++) tmp[k] = n[k];
        for (uint32_t k = 0; k < vl; k++) tmp[nl + k] = v[k];
        (void)hp_add(t, tmp, nl, vl);
        p = hp_put_int(p, 0x40, 6, name_index);
    } else p = hp_put_int(p, 0x10, 4, name_index);
    if (name_index == 0) { p = hp_put_int(p, 0x00, 7, nl); for (uint32_t k = 0; k < nl; k++) *p++ = lc(n[k]); }
    p = hp_put_int(p, 0x00, 7, vl); for (uint32_t k = 0; k < vl; k++) *p++ = v[k];
    return p;
}
__device__ __forceinline__ uint32_t put_dec_i32_h2(uint8_t* p, int32_t v) {     // "%d"
    uint8_t tmp[12]; uint32_t n = 0; uint32_t u = v < 0 ? (uint32_t)(-(long long)v) : (uint32_t)v;
    do { tmp[n++] = (uint8_t)('0' + u % 10); u /= 10; } while (u);
    uint32_t o = 0; if (v < 0) p[o++] = '-';
    while (n) p[o++] = tmp[--n];
    return o;
}
constexpr uint32_t kH2FragCap = 1024;      // encoded header block of one response (":status", "content-type", trailers)
constexpr uint32_t kH2PackWarps = 4;
// One WARP per connection: lane 0 runs the serial part (window check, HPACK encode against the connection's table,
// deferred WINDOW_UPDATE) into shared memory, then the whole warp writes the frames — the DATA payload, which is
// nearly all of the bytes, with coalesced 16-byte copies.
__global__ void __launch_bounds__(kH2PackWarps * 32) k_h2_pack(const uint8_t* bytes, const uint8_t* last_input, const uint8_t* last_out, const uint8_t* last_unz, const b2_h2_response* resps,
                                                               const uint32_t* group_first, uint32_t n_groups, H2Conn* conns,
                                                               uint8_t* out, const uint32_t* out_offs, uint32_t* out_lens) {
    __shared__ __align__(16) uint8_t s_buf[kH2PackWarps][3][kH2FragCap];
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t g = blockIdx.x * kH2PackWarps + w;
    if (g >= n_groups) return;
    uint8_t* frag = s_buf[w][0]; uint8_t* trailer = s_buf[w][1]; uint8_t* tmp = s_buf[w][2];
    for (uint32_t i = group_first[g]; i < group_first[g + 1]; i++) {
        const b2_h2_response R = resps[i];
        uint8_t* o0 = out + out_offs[i]; uint8_t* o = o0;
        const bool grpc = R.flags & B2_H2_RESP_GRPC;
        const uint32_t data_size = R.body_len + (grpc ? 5u : 0u);
        uint32_t rst = 0, fl = 0, tl = 0, mfs = 0, cw = 0;
        if (lane == 0) {
            H2Conn& c = conns[R.conn];
            // MinusWindowSize(&_remote_window_left, _data.size()) (:283-296)
            if (c.remote_window_left < (long long)data_size) rst = 1;
            else {
                c.remote_window_left -= (long long)data_size;
                const bool never = c.r_header_table_size == 0;
                uint8_t num[16];
                uint8_t* f = frag;
                { const uint32_t nn = put_dec_i32_h2(num, R.status_code); f = hp_encode(c.enc, f, (const uint8_t*)":status", 7, num, nn, never, tmp); }
                if (R.content_type_len) f = hp_encode(c.enc, f, (const uint8_t*)"content-type", 12, ((R.flags & B2_H2_RESP_CT_IN_OUT) ? last_out : bytes) + R.content_type_off, R.content_type_len, never, tmp);
                uint8_t* t = trailer;
                if (grpc) {
                    const uint32_t nn = put_dec_i32_h2(num, R.grpc_status);
                    t = hp_encode(c.enc, t, (const uint8_t*)"grpc-status", 11, num, nn, never, tmp);
                    if (R.grpc_message_len) t = hp_encode(c.enc, t, (const uint8_t*)"grpc-message", 12, bytes + R.grpc_message_off, R.grpc_message_len, never, tmp);
                }
                fl = (uint32_t)(f - frag); tl = (uint32_t)(t - trailer); mfs = c.r_max_frame_size;
                if (c.deferred_window_update > 0) { cw = (uint32_t)c.deferred_window_update; c.deferred_window_update = 0; }   // ReleaseDeferredWindowUpdate
            }
        }
        rst = __shfl_sync(0xffffffffu, rst, 0); fl = __shfl_sync(0xffffffffu, fl, 0); tl = __shfl_sync(0xffffffffu, tl, 0);
        mfs = __shfl_sync(0xffffffffu, mfs, 0); cw = __shfl_sync(0xffffffffu, cw, 0);
        __syncwarp();
        if (rst) {                                                   // RST_STREAM(FLOW_CONTROL_ERROR) instead of the response (:1706-1712)
            if (lane == 0) { h2_put_head(o, 4, 3, 0, R.stream_id); put_be32(o + 9, 3); out_lens[i] = 13; }
            __syncwarp();
            continue;
        }
        // ---- PackH2Message (:1310-1380)
        const uint8_t hflags = (data_size == 0 && tl == 0) ? 0x1 : 0;
        if (fl <= mfs) {
            if (lane == 0) h2_put_head(o, fl, 1, hflags | 0x4, R.stream_id);
            for (uint32_t k = lane; k < fl; k += 32) o[9 + k] = frag[k];
            o += 9 + fl;
        } else {                                                     // (cannot happen with kH2FragCap < 16384 <= max_frame_size; kept for the shape)
            if (lane == 0) {
                uint8_t* q = o;
                h2_put_head(q, mfs, 1, hflags, R.stream_id); q += 9; for (uint32_t k = 0; k < mfs; k++) *q++ = frag[k];
                for (uint32_t at = mfs; at < fl;) { const uint32_t nn = min(fl - at, mfs); h2_put_head(q, nn, 9, at + nn == fl ? 0x4 : 0, R.stream_id); q += 9; for (uint32_t k = 0; k < nn; k++) *q++ = frag[at + k]; at += nn; }
            }
            o += fl + 9 * ((fl + mfs - 1) / mfs);
        }
        const uint8_t* body = ((R.flags & B2_H2_RESP_BODY_IN_INPUT) ? last_input : (R.flags & B2_H2_RESP_BODY_IN_OUT) ? last_out :
                                    (R.flags & B2_H2_RESP_BODY_IN_UNZ) ? last_unz : bytes) + R.body_off;
        for (uint32_t at = 0; at < data_size;) {
            const uint32_t nn = min(data_size - at, mfs);
            const uint8_t dflags = (at + nn == data_size && tl == 0) ? 0x1 : 0;
            if (lane == 0) h2_put_head(o, nn, 0, dflags, R.stream_id);
            o += 9;
            uint32_t k = 0;
            if (grpc && at < 5) { k = min(nn, 5u - at); if (lane < k) { const uint32_t q = at + lane; o[lane] = q == 0 ? 0 : (uint8_t)(R.body_len >> (8 * (4 - q))); } }   // AddGrpcPrefix: flag 0 + BE32 length
            warp_copy(o + k, body + (at + k - (grpc ? 5u : 0u)), nn - k, lane);
            o += nn; at += nn;
        }
        if (tl) { if (lane == 0) h2_put_head(o, tl, 1, 0x5, R.stream_id); for (uint32_t k = lane; k < tl; k += 32) o[9 + k] = trailer[k]; o += 9 + tl; }
        if (cw) { if (lane == 0) { h2_put_head(o, 4, 8, 0, 0); put_be32(o + 9, cw); } o += 13; }
        if (lane == 0) out_lens[i] = (uint32_t)(o - o0);
        __syncwarp();                                                // the shared buffers are reused by the next response
    }
}

// ---------------------------------------------------------------------------------------------------------
// The GzipDecompress step of ProcessHttpRequest (policy/http_rpc_protocol.cpp:1646-1683) for messages of the last batch.
// The value HttpHeader keeps for `name` (AppendHeader, http_header.cpp:100-116: case-insensitive names, a repeated field folded with
// "," onto a non-empty value, an empty value overwritten): 0 no such field, 1 exactly "gzip", 2 anything else.  Once the value is
// non-empty every further field appends a ",", so it equals "gzip" only when the first non-empty value is "gzip" and is the last field.
// `name` is upper case (ci_eq).
__device__ __forceinline__ uint32_t h2_encoding(const uint8_t* hdr, uint32_t len, const char* name) {
    bool present = false, nonempty = false, gzip = false;
    for (uint32_t q = 0; q + 4 <= len;) {
        const uint32_t nl = hdr[q] | ((uint32_t)hdr[q + 1] << 8), vl = hdr[q + 2] | ((uint32_t)hdr[q + 3] << 8);
        if (q + 4 + nl + vl > len) break;
        if (ci_eq(hdr + q + 4, nl, name)) {
            present = true;
            if (nonempty) gzip = false;
            else { nonempty = vl != 0; gzip = lit_eq(hdr + q + 4 + nl, vl, "gzip"); }
        }
        q += 4 + nl + vl;
    }
    return !present ? 0u : gzip ? 1u : 2u;
}
// B2_H2_UNZ_OK here = "to be inflated"
__device__ __forceinline__ uint32_t h2_unz_status(const b2_h2_msg& m, const uint8_t* out) {
    if (m.body_len == 0) return B2_H2_UNZ_NONE;
    uint32_t enc;
    if (m.flags & B2_H2_FLAG_GRPC) {
        if ((m.flags & (B2_H2_FLAG_GRPC_PREFIX_OK | B2_H2_FLAG_GRPC_COMPRESSED)) != (B2_H2_FLAG_GRPC_PREFIX_OK | B2_H2_FLAG_GRPC_COMPRESSED)) return B2_H2_UNZ_NONE;
        enc = h2_encoding(out + m.headers_off, m.headers_len, "GRPC-ENCODING");
        if (enc == 0) return B2_H2_UNZ_NO_ENCODING;
    } else {
        enc = h2_encoding(out + m.headers_off, m.headers_len, "CONTENT-ENCODING");
        if (enc == 0) return B2_H2_UNZ_NONE;
    }
    return enc == 1 ? B2_H2_UNZ_OK : B2_H2_UNZ_NOT_GZIP;
}
// One warp per message, its lane 0 decoding (the shape of k_pack_slow): a gzip-enabled client compresses every call, so a batch holds
// many independent DEFLATE streams, each a serial bit stream.  Measured against one thread per message on the grpc_h2 shape (256
// connections x 8 calls of 4 KiB, B200 at 1000 W, tools/h2_gzip_probe.py): 2.71 ms against 4.24 ms for the three stages.
// kWrite = false classifies and sizes (res.out_len = gz_input_stream<false>'s bound); k_h2_unz_offsets then places the slots;
// kWrite = true inflates into them.  GzipDecompressBase (gzip_compress.cpp:138-176) hands over what GzipInputStream yields and, for a
// body in one block, never fails (DESIGN §5).
constexpr uint32_t kH2UnzWarps = 4;
template <bool kWrite>
__global__ void __launch_bounds__(kH2UnzWarps * 32) k_h2_inflate(const uint8_t* in, const uint8_t* out, const b2_h2_msg* msgs, uint32_t n,
                                                                 b2_h2_unz_result* res, uint8_t* unz) {
    const uint32_t i = blockIdx.x * kH2UnzWarps + (threadIdx.x >> 5);
    if ((threadIdx.x & 31) || i >= n) return;
    const b2_h2_msg m = msgs[i];
    const bool grpc = m.flags & B2_H2_FLAG_GRPC;
    const uint8_t* src = ((m.flags & B2_H2_FLAG_BODY_IN_INPUT) ? in : out) + (grpc ? m.msg_off : m.body_off);
    const uint32_t len = grpc ? m.msg_len : m.body_len;
    bool big = false;
    if (!kWrite) {
        b2_h2_unz_result r; r.status = h2_unz_status(m, out); r.out_off = 0; r.out_len = 0; r.reserved = 0;
        if (r.status == B2_H2_UNZ_OK) {
            if (len > kGzMaxIn) r.status = B2_H2_UNZ_HOST;
            else {
                r.out_len = gz_input_stream<false>(src, len, B2_COMPRESS_TYPE_GZIP, nullptr, kGzMaxOut, &big);
                if (big) { r.status = B2_H2_UNZ_HOST; r.out_len = 0; }
            }
        }
        res[i] = r;
    } else {
        const b2_h2_unz_result r = res[i];
        if (r.status != B2_H2_UNZ_OK) return;
        uint8_t* dst = unz + r.out_off;
        const uint32_t got = gz_input_stream<true>(src, len, B2_COMPRESS_TYPE_GZIP, dst, r.out_len, &big);
        for (uint32_t k = got; k < r.out_len; k++) dst[k] = 0;     // a stream whose check failed delivers less than its bound: no stale bytes
        res[i].out_len = got;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Client side: H2UnsentRequest::New (:1382-1453, the header list) + AppendAndDestroySelf (:1496-1592) + PackH2Message (:1310-1380).
// The same split as k_h2_pack: one warp per connection, lane 0 runs the serial part (stream id, windows, HPACK encode against the
// connection's table) into shared memory, the warp writes the frames.
constexpr uint32_t kH2ReqFragCap = 2048;
__global__ void __launch_bounds__(kH2PackWarps * 32) k_h2_pack_req(const uint8_t* bytes, const b2_h2_request* reqs, const uint32_t* group_first, uint32_t n_groups,
                                                                   H2Conn* conns, uint8_t* out, b2_h2_request_result* results) {
    __shared__ __align__(16) uint8_t s_buf[kH2PackWarps][2][kH2ReqFragCap];
    const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t g = blockIdx.x * kH2PackWarps + w;
    if (g >= n_groups) return;
    uint8_t* frag = s_buf[w][0]; uint8_t* tmp = s_buf[w][1];
    for (uint32_t i = group_first[g]; i < group_first[g + 1]; i++) {
        const b2_h2_request R = reqs[i];
        uint8_t* o0 = out + results[i].out_off; uint8_t* o = o0;
        const bool grpc = R.flags & B2_H2_REQ_GRPC;
        const uint32_t data_size = R.body_len + (grpc ? 5u : 0u);
        uint32_t st = B2_H2_REQ_OK, sid = 0, fl = 0, mfs = 0, cw = 0, pre = 0;
        if (lane == 0) {
            H2Conn& c = conns[R.conn];
            if (!c.preface_sent) { c.preface_sent = 1; pre = 1; }
            if (c.last_sent_stream_id > 0x7FFFFFFFll) st = B2_H2_REQ_RUNOUT;                      // AllocateClientStreamId
            else {
                sid = (uint32_t)c.last_sent_stream_id; c.last_sent_stream_id += 2;
                // ConsumeWindowSize (:1199-1219) on a stream that starts with the peer's initial window (Init :1176-1181)
                if (data_size && ((long long)c.r_stream_window_size < (long long)data_size || c.remote_window_left < (long long)data_size)) st = B2_H2_REQ_ELIMIT;
                else {
                    c.remote_window_left -= (long long)data_size;
                    const bool never = c.r_header_table_size == 0;
                    uint8_t* f = frag;
                    f = (R.flags & B2_H2_REQ_GET) ? hp_encode(c.enc, f, (const uint8_t*)":method", 7, (const uint8_t*)"GET", 3, never, tmp)
                                                  : hp_encode(c.enc, f, (const uint8_t*)":method", 7, (const uint8_t*)"POST", 4, never, tmp);
                    f = (R.flags & B2_H2_REQ_HTTPS) ? hp_encode(c.enc, f, (const uint8_t*)":scheme", 7, (const uint8_t*)"https", 5, never, tmp)
                                                    : hp_encode(c.enc, f, (const uint8_t*)":scheme", 7, (const uint8_t*)"http", 4, never, tmp);
                    f = hp_encode(c.enc, f, (const uint8_t*)":path", 5, bytes + R.path_off, R.path_len, never, tmp);
                    f = hp_encode(c.enc, f, (const uint8_t*)":authority", 10, bytes + R.authority_off, R.authority_len, never, tmp);
                    if (R.content_type_len) f = hp_encode(c.enc, f, (const uint8_t*)"content-type", 12, bytes + R.content_type_off, R.content_type_len, never, tmp);
                    if (R.flags & B2_H2_REQ_ACCEPT) f = hp_encode(c.enc, f, (const uint8_t*)"accept", 6, (const uint8_t*)"*/*", 3, never, tmp);
                    if (R.flags & B2_H2_REQ_USER_AGENT) f = hp_encode(c.enc, f, (const uint8_t*)"user-agent", 10, (const uint8_t*)"brpc/1.0 curl/7.0", 17, never, tmp);
                    for (uint32_t at = 0; at + 4 <= R.extra_len;) {
                        const uint8_t* e = bytes + R.extra_off + at;
                        const uint32_t nl = e[0] | ((uint32_t)e[1] << 8), vl = e[2] | ((uint32_t)e[3] << 8);
                        if (at + 4 + nl + vl > R.extra_len) break;
                        f = hp_encode(c.enc, f, e + 4, nl, e + 4 + nl, vl, never, tmp);
                        at += 4 + nl + vl;
                    }
                    fl = (uint32_t)(f - frag); mfs = c.r_max_frame_size;
                    if (c.deferred_window_update > 0) { cw = (uint32_t)c.deferred_window_update; c.deferred_window_update = 0; }
                }
            }
        }
        st = __shfl_sync(0xffffffffu, st, 0); sid = __shfl_sync(0xffffffffu, sid, 0); fl = __shfl_sync(0xffffffffu, fl, 0);
        mfs = __shfl_sync(0xffffffffu, mfs, 0); cw = __shfl_sync(0xffffffffu, cw, 0); pre = __shfl_sync(0xffffffffu, pre, 0);
        __syncwarp();
        if (pre) {                                                   // preface + SerializeH2SettingsFrameAndWU(default client settings) (:1508-1526)
            if (lane < 24) o[lane] = (uint8_t)"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n"[lane];
            if (lane == 0) {
                uint8_t* p = o + 24;
                h2_put_head(p, 12, 4, 0, 0);
                p[9] = 0; p[10] = 2; put_be32(p + 11, 0);
                p[15] = 0; p[16] = 4; put_be32(p + 17, 256u * 1024u);
                h2_put_head(p + 21, 4, 8, 0, 0); put_be32(p + 30, 1024u * 1024u - 65535u);
            }
            o += 58;
        }
        if (st != B2_H2_REQ_OK) {
            if (lane == 0) { results[i].status = (int32_t)st; results[i].stream_id = sid; results[i].out_len = (uint32_t)(o - o0); }
            __syncwarp();
            continue;
        }
        const uint8_t hflags = data_size == 0 ? 0x1 : 0;
        if (fl <= mfs) {
            if (lane == 0) h2_put_head(o, fl, 1, hflags | 0x4, sid);
            for (uint32_t k = lane; k < fl; k += 32) o[9 + k] = frag[k];
            o += 9 + fl;
        } else {                                                     // (kH2ReqFragCap < 16384 <= max_frame_size: kept for the shape)
            if (lane == 0) {
                uint8_t* q = o;
                h2_put_head(q, mfs, 1, hflags, sid); q += 9; for (uint32_t k = 0; k < mfs; k++) *q++ = frag[k];
                for (uint32_t at = mfs; at < fl;) { const uint32_t nn = min(fl - at, mfs); h2_put_head(q, nn, 9, at + nn == fl ? 0x4 : 0, sid); q += 9; for (uint32_t k = 0; k < nn; k++) *q++ = frag[at + k]; at += nn; }
            }
            o += fl + 9 * ((fl + mfs - 1) / mfs);
        }
        const uint8_t* body = bytes + R.body_off;
        for (uint32_t at = 0; at < data_size;) {
            const uint32_t nn = min(data_size - at, mfs);
            if (lane == 0) h2_put_head(o, nn, 0, at + nn == data_size ? 0x1 : 0, sid);
            o += 9;
            uint32_t k = 0;
            if (grpc && at < 5) { k = min(nn, 5u - at); if (lane < k) { const uint32_t q = at + lane; o[lane] = q == 0 ? 0 : (uint8_t)(R.body_len >> (8 * (4 - q))); } }   // AddGrpcPrefix
            warp_copy(o + k, body + (at + k - (grpc ? 5u : 0u)), nn - k, lane);
            o += nn; at += nn;
        }
        if (cw) { if (lane == 0) { h2_put_head(o, 4, 8, 0, 0); put_be32(o + 9, cw); } o += 13; }
        if (lane == 0) { results[i].status = B2_H2_REQ_OK; results[i].stream_id = sid; results[i].out_len = (uint32_t)(o - o0); }
        __syncwarp();                                                // the shared buffers are reused by the next request
    }
}
// b2_h2_conn_peer_update: OnSettings' effect on _remote_settings (:848-915) and OnWindowUpdate on stream 0 (:1006-1041), mirrored by the host
__global__ void k_h2_peer_update(H2Conn* conns, uint32_t conn, b2_h2_peer_update u, int* rc) {
    H2Conn& c = conns[conn];
    *rc = 0;
    if (u.set & B2_H2_PEER_HEADER_TABLE_SIZE) c.r_header_table_size = u.header_table_size;
    if (u.set & B2_H2_PEER_MAX_FRAME_SIZE) c.r_max_frame_size = u.max_frame_size;
    if (u.set & B2_H2_PEER_STREAM_WINDOW) c.r_stream_window_size = u.stream_window_size;
    if (u.set & B2_H2_PEER_CONN_WINDOW_ADD) {
        if (u.conn_window_add < 0) c.remote_window_left += u.conn_window_add;
        else if (!h2_add_window(c.remote_window_left, u.conn_window_add)) *rc = -1;
    }
}
__global__ void k_h2_set_next_stream_id(H2Conn* conns, uint32_t conn, uint32_t next_id) { conns[conn].last_sent_stream_id = next_id; }
#endif
}  // namespace b2
