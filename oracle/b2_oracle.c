/*
 * b2_oracle.c — CPU ORACLE (test infrastructure, NOT product code).
 * See b2_oracle.h for the rules on who may call this and how it is pinned.
 *
 * Every function restates one reference function over flat byte buffers
 * (an IOBuf is just its byte string for the purposes of results); citations
 * are relative to /root/reference/.
 */
#include "b2_oracle.h"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------ */
/* CRC-32C.  src/butil/crc32c.cc:379-454 (Extend: init/xorout 0xffffffff,
 * reflected Castagnoli polynomial 0x82f63b78), crc32c.h:38-47 (Mask/Unmask). */
static uint32_t g_crc_tab[8][256];
static int g_crc_init = 0;
static void crc_init(void) {
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0x82f63b78u : (c >> 1);
        g_crc_tab[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; i++)
        for (int t = 1; t < 8; t++)
            g_crc_tab[t][i] = (g_crc_tab[t - 1][i] >> 8) ^ g_crc_tab[0][g_crc_tab[t - 1][i] & 0xff];
    g_crc_init = 1;
}
uint32_t orc_crc32c_extend(uint32_t init_crc, const void* data, size_t n) {
    if (!g_crc_init) crc_init();
    const uint8_t* p = (const uint8_t*)data;
    uint32_t l = init_crc ^ 0xffffffffu;
    while (n >= 8) {
        uint32_t a, b;
        memcpy(&a, p, 4); memcpy(&b, p + 4, 4);
        a ^= l;
        l = g_crc_tab[7][a & 0xff] ^ g_crc_tab[6][(a >> 8) & 0xff] ^ g_crc_tab[5][(a >> 16) & 0xff] ^
            g_crc_tab[4][a >> 24] ^ g_crc_tab[3][b & 0xff] ^ g_crc_tab[2][(b >> 8) & 0xff] ^
            g_crc_tab[1][(b >> 16) & 0xff] ^ g_crc_tab[0][b >> 24];
        p += 8; n -= 8;
    }
    while (n--) l = g_crc_tab[0][(l ^ *p++) & 0xff] ^ (l >> 8);
    return l ^ 0xffffffffu;
}
uint32_t orc_crc32c_mask(uint32_t crc) { return ((crc >> 15) | (crc << 17)) + 0xa282ead8u; }
uint32_t orc_crc32c_unmask(uint32_t m) { uint32_t rot = m - 0xa282ead8u; return (rot >> 17) | (rot << 15); }

/* ------------------------------------------------------------------------ */
/* Snappy raw format (format_description.txt of the snappy project), as the
 * reference vendors it: Snappy 1.1.3 (src/butil/third_party/snappy).  The
 * encoder follows that version's CompressFragment (snappy.cc:329-468): 64 KiB
 * fragments, a zeroed uint16 hash table of 256..16384 entries (>= fragment
 * size), hash = load32 * 0x1e35a7bd >> shift, skip heuristic skip++ >> 5, a
 * 15-byte input margin, EmitLiteral / EmitCopy (:156-233); so its bytes are
 * the reference's (pinned by tests/golden/snappy_vectors.json).  The decoder
 * gives RawUncompress's verdict (snappy.cc:716-787, :1145-1215): well formed,
 * input consumed exactly, exactly the announced length produced.             */
size_t orc_snappy_max_compressed_length(size_t n) { return 32 + n + n / 6; }   /* snappy.cc:55-77 */

static uint32_t sn_ld32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
static size_t sn_literal(uint8_t* op, const uint8_t* src, size_t len) {
    size_t n = len - 1, w = 1;
    if (n < 60) op[0] = (uint8_t)(n << 2);
    else {
        uint32_t count = 0;
        while (n > 0) { op[1 + count] = (uint8_t)(n & 0xff); n >>= 8; count++; }
        op[0] = (uint8_t)((59 + count) << 2); w += count;
    }
    memcpy(op + w, src, len);
    return w + len;
}
static size_t sn_copy_lt64(uint8_t* op, size_t offset, size_t len) {
    if (len < 12 && offset < 2048) { op[0] = (uint8_t)(1 + ((len - 4) << 2) + ((offset >> 8) << 5)); op[1] = (uint8_t)(offset & 0xff); return 2; }
    op[0] = (uint8_t)(2 + ((len - 1) << 2)); op[1] = (uint8_t)(offset & 0xff); op[2] = (uint8_t)(offset >> 8); return 3;
}
static size_t sn_copy(uint8_t* op, size_t offset, size_t len) {
    size_t w = 0;
    while (len >= 68) { w += sn_copy_lt64(op + w, offset, 64); len -= 64; }
    if (len > 64) { w += sn_copy_lt64(op + w, offset, 60); len -= 60; }
    return w + sn_copy_lt64(op + w, offset, len);
}
static size_t sn_fragment(const uint8_t* in, size_t n, uint8_t* out, uint16_t* table) {
    uint32_t table_size = 256, shift = 24;
    while (table_size < 16384 && table_size < n) { table_size <<= 1; shift--; }
    memset(table, 0, table_size * sizeof *table);
    size_t op = 0, ip = 0, next_emit = 0;
    if (n >= 15) {
        const size_t ip_limit = n - 15;
        uint32_t next_hash = (sn_ld32(in + 1) * 0x1e35a7bdu) >> shift;
        ip = 1;
        for (;;) {
            size_t candidate, next_ip = ip;
            uint32_t skip = 32;
            for (;;) {                                               /* a 4-byte match */
                ip = next_ip;
                const uint32_t hash = next_hash;
                next_ip = ip + (skip++ >> 5);
                if (next_ip > ip_limit) goto emit_remainder;
                next_hash = (sn_ld32(in + next_ip) * 0x1e35a7bdu) >> shift;
                candidate = table[hash];
                table[hash] = (uint16_t)ip;
                if (sn_ld32(in + ip) == sn_ld32(in + candidate)) break;
            }
            op += sn_literal(out + op, in + next_emit, ip - next_emit);
            for (;;) {                                               /* copies while the next position matches again */
                const size_t base = ip;
                size_t matched = 4;
                while (ip + matched < n && in[candidate + matched] == in[ip + matched]) matched++;
                ip += matched;
                op += sn_copy(out + op, base - candidate, matched);
                next_emit = ip;
                if (ip >= ip_limit) goto emit_remainder;
                table[(sn_ld32(in + ip - 1) * 0x1e35a7bdu) >> shift] = (uint16_t)(ip - 1);
                const uint32_t cur = sn_ld32(in + ip), cur_hash = (cur * 0x1e35a7bdu) >> shift;
                candidate = table[cur_hash];
                table[cur_hash] = (uint16_t)ip;
                if (cur != sn_ld32(in + candidate)) break;
            }
            next_hash = (sn_ld32(in + ip + 1) * 0x1e35a7bdu) >> shift;
            ++ip;
        }
    }
emit_remainder:
    if (next_emit < n) op += sn_literal(out + op, in + next_emit, n - next_emit);
    return op;
}
/* RawCompress: varint32 length, then the fragments; out holds orc_snappy_max_compressed_length(n) */
size_t orc_snappy_compress(const uint8_t* in, size_t n, uint8_t* out) {
    uint16_t table[16384];
    size_t op = 0, v = n;
    while (v >= 0x80) { out[op++] = (uint8_t)(v | 0x80); v >>= 7; }
    out[op++] = (uint8_t)v;
    for (size_t pos = 0; pos < n; pos += 65536) op += sn_fragment(in + pos, n - pos < 65536 ? n - pos : 65536, out + op, table);
    return op;
}
/* GetUncompressedLength: the varint32 preamble (SnappyDecompressor::ReadUncompressedLength, snappy.cc:690-711) */
static int sn_preamble(const uint8_t* in, size_t n, size_t* ulen, size_t* used) {
    uint32_t v = 0, shift = 0; size_t ip = 0;
    for (;;) {
        if (shift >= 32 || ip >= n) return 0;
        const uint32_t c = in[ip++];
        v |= (c & 0x7f) << shift;
        if (c < 128) break;
        shift += 7;
    }
    *ulen = v; if (used) *used = ip;
    return 1;
}
int orc_snappy_uncompressed_length(const uint8_t* in, size_t n, size_t* ulen) { return sn_preamble(in, n, ulen, NULL); }
/* RawUncompress into out[cap]: 1 and *got = the announced length when the stream is valid and fits, else 0 */
int orc_snappy_uncompress(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* got) {
    size_t ulen, ip, op = 0;
    if (!sn_preamble(in, n, &ulen, &ip) || ulen > cap) return 0;
    while (ip < n) {
        const uint32_t c = in[ip++];
        if ((c & 3) == 0) {                                          /* literal */
            uint64_t len = (c >> 2) + 1;
            if (len >= 61) {
                const size_t ll = len - 60;
                if (n - ip < ll) return 0;
                uint64_t v = 0;
                for (size_t k = 0; k < ll; k++) v |= (uint64_t)in[ip + k] << (8 * k);
                len = v + 1; ip += ll;
            }
            if (len > n - ip || len > ulen - op) return 0;           /* premature end of input / no room */
            memcpy(out + op, in + ip, len); ip += len; op += len;
        } else {                                                     /* copy */
            size_t len, offset;
            if ((c & 3) == 1) {
                if (n - ip < 1) return 0;
                len = ((c >> 2) & 7) + 4; offset = ((size_t)(c >> 5) << 8) | in[ip]; ip += 1;
            } else if ((c & 3) == 2) {
                if (n - ip < 2) return 0;
                len = (c >> 2) + 1; offset = in[ip] | ((size_t)in[ip + 1] << 8); ip += 2;
            } else {
                if (n - ip < 4) return 0;
                len = (c >> 2) + 1; offset = sn_ld32(in + ip); ip += 4;
            }
            if (offset == 0 || offset > op || len > ulen - op) return 0;
            for (size_t i = 0; i < len; i++) out[op + i] = out[op - offset + i];     /* may overlap its own output */
            op += len;
        }
    }
    if (op != ulen) return 0;
    *got = op;
    return 1;
}

/* ------------------------------------------------------------------------ */
/* protobuf wire reader: restates google::protobuf (pinned 27.3, MODULE.bazel:11)
 * parse_context.h semantics as used by ParsePbFromIOBuf (protocol.cpp:202-239):
 * ParseFromCodedStream() && ConsumedEntireMessage().                         */
typedef struct { const uint8_t* p; const uint8_t* end; } rd_t;

/* VarintParse<uint64>: at most 10 bytes, bits past 64 silently dropped. */
static int rd_varint(rd_t* r, uint64_t* out) {
    uint64_t v = 0;
    for (int i = 0; i < 10; i++) {
        if (r->p >= r->end) return 0;
        uint8_t b = *r->p++;
        v |= (uint64_t)(b & 0x7f) << (7 * i);
        if (b < 0x80) { *out = v; return 1; }
    }
    return 0;
}
/* ReadTag / ReadTagFallback: at most 5 bytes, bits past 32 dropped. */
static int rd_tag(rd_t* r, uint32_t* tag) {
    uint32_t v = 0;
    for (int i = 0; i < 5; i++) {
        if (r->p >= r->end) return 0;
        uint8_t b = *r->p++;
        v |= (uint32_t)(b & 0x7f) << (7 * i);
        if (b < 0x80) { *tag = v; return 1; }
    }
    return 0;
}
/* ReadSize / ReadSizeFallback: at most 5 bytes, 5th byte < 8, value <= INT_MAX-16;
 * the delimited field must end inside the enclosing message. */
static int rd_size(rd_t* r, uint32_t* n) {
    uint32_t v = 0;
    for (int i = 0; i < 5; i++) {
        if (r->p >= r->end) return 0;
        uint8_t b = *r->p++;
        if (i == 4 && b >= 8) return 0;
        v |= (uint32_t)(b & 0x7f) << (7 * i);
        if (b < 0x80) {
            if (v > 0x7fffffffu - 16u) return 0;
            if ((uint64_t)v > (uint64_t)(r->end - r->p)) return 0;
            *n = v; return 1;
        }
    }
    return 0;
}
/* UnknownFieldParse: skip one field by wire type.  `budget` is ParseContext's
 * depth_ at this nesting level (groups consume one level each). */
static int skip_field(rd_t* r, uint32_t tag, int budget) {
    uint64_t v; uint32_t n;
    switch (tag & 7) {
    case 0: return rd_varint(r, &v);
    case 1: if (r->end - r->p < 8) return 0; r->p += 8; return 1;
    case 2: if (!rd_size(r, &n)) return 0; r->p += n; return 1;
    case 3: {
        if (budget <= 0) return 0;
        for (;;) {
            uint32_t t;
            if (r->p >= r->end) return 0;           /* group not closed inside message */
            if (!rd_tag(r, &t)) return 0;
            if (t == 0) return 0;
            if ((t & 7) == 4) return (t >> 3) == (tag >> 3);
            if ((t >> 3) == 0) return 0;
            if (!skip_field(r, t, budget - 1)) return 0;
        }
    }
    case 5: if (r->end - r->p < 4) return 0; r->p += 4; return 1;
    default: return 0;   /* 4 = stray end-group, 6/7 = invalid */
    }
}
typedef int (*field_fn)(void* ctx, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base);
/* message loop; returns 1 when the message ended exactly at r->end */
static int parse_fields(rd_t* r, int budget, field_fn cb, void* ctx, const uint8_t* base) {
    while (r->p < r->end) {
        uint32_t tag;
        if (!rd_tag(r, &tag)) return 0;
        if (tag == 0 || (tag & 7) == 4) return 0;   /* parse stops early -> not consumed */
        if ((tag >> 3) == 0) return 0;
        int h = cb(ctx, tag >> 3, tag & 7, r, budget, base);
        if (h < 0) return 0;
        if (h == 0 && !skip_field(r, tag, budget)) return 0;
    }
    return 1;
}
static int sub_begin(rd_t* r, rd_t* sub, int budget) {   /* ParseMessage: --depth_ < 0 fails */
    uint32_t n;
    if (budget <= 0) return 0;
    if (!rd_size(r, &n)) return 0;
    sub->p = r->p; sub->end = r->p + n; r->p += n;
    return 1;
}
static int rd_bytes_span(rd_t* r, orc_span* s, const uint8_t* base) {
    uint32_t n;
    if (!rd_size(r, &n)) return 0;
    s->off = (uint32_t)(r->p - base); s->len = n; r->p += n;
    return 1;
}

/* RpcRequestMeta, baidu_rpc_meta.proto:41-50 */
static int cb_request(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_rpc_meta* m = (orc_rpc_meta*)c; uint64_t v; (void)budget;
    switch (fn) {
    case 1: if (wt != 2) return 0; if (!rd_bytes_span(r, &m->service_name, base)) return -1; m->has_service_name = 1; return 1;
    case 2: if (wt != 2) return 0; if (!rd_bytes_span(r, &m->method_name, base)) return -1; m->has_method_name = 1; return 1;
    case 3: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->log_id = (int64_t)v; m->has |= B2_HAS_LOG_ID; return 1;
    case 4: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->trace_id = (int64_t)v; m->has |= B2_HAS_TRACE_ID; return 1;
    case 5: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->span_id = (int64_t)v; m->has_span_id = 1; return 1;
    case 6: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->parent_span_id = (int64_t)v; m->has_parent_span_id = 1; return 1;
    case 7: if (wt != 2) return 0; if (!rd_bytes_span(r, &m->request_id, base)) return -1; m->has |= B2_HAS_REQUEST_ID; return 1;
    case 8: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->timeout_ms = (int32_t)(uint32_t)v; m->has |= B2_HAS_TIMEOUT_MS; return 1;
    }
    return 0;
}
/* RpcResponseMeta, baidu_rpc_meta.proto:52-55 */
static int cb_response(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_rpc_meta* m = (orc_rpc_meta*)c; uint64_t v; (void)budget;
    switch (fn) {
    case 1: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->error_code = (int32_t)(uint32_t)v; m->has_error_code = 1; return 1;
    case 2: if (wt != 2) return 0; if (!rd_bytes_span(r, &m->error_text, base)) return -1; m->has_error_text = 1; return 1;
    }
    return 0;
}
/* ChunkInfo, options.proto:90-93 */
static int cb_chunk(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_rpc_meta* m = (orc_rpc_meta*)c; uint64_t v; (void)budget; (void)base;
    switch (fn) {
    case 1: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->chunk_has_stream_id = 1; return 1;
    case 2: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->chunk_has_chunk_id = 1; return 1;
    }
    return 0;
}
/* StreamSettings, streaming_rpc_meta.proto:24-29 */
static int cb_stream_settings(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_rpc_meta* m = (orc_rpc_meta*)c; uint64_t v; (void)budget; (void)base;
    switch (fn) {
    case 1: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->ss_stream_id = (int64_t)v; m->ss_has_stream_id = 1; return 1;
    case 2: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->ss_need_feedback = v != 0; return 1;
    case 3: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->ss_writable = v != 0; return 1;
    case 4:
        if (wt == 0) { if (!rd_varint(r, &v)) return -1; m->ss_n_extra++; return 1; }
        if (wt == 2) {   /* packed encoding is accepted for a repeated scalar */
            rd_t sub; uint32_t n;
            if (!rd_size(r, &n)) return -1;
            sub.p = r->p; sub.end = r->p + n; r->p += n;
            while (sub.p < sub.end) { if (!rd_varint(&sub, &v)) return -1; m->ss_n_extra++; }
            return 1;
        }
        return 0;
    }
    return 0;
}
/* map<string,string> entry {1:key, 2:value}; contents are not surfaced */
static int cb_map_entry(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_span s; (void)c; (void)budget;
    if ((fn == 1 || fn == 2) && wt == 2) return rd_bytes_span(r, &s, base) ? 1 : -1;
    return 0;
}
/* RpcMeta, baidu_rpc_meta.proto:26-39 */
static int cb_rpc_meta(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_rpc_meta* m = (orc_rpc_meta*)c; uint64_t v; rd_t sub;
    switch (fn) {
    case 1: if (wt != 2) return 0; if (!sub_begin(r, &sub, budget)) return -1; m->has |= B2_HAS_REQUEST;
            return parse_fields(&sub, budget - 1, cb_request, m, base) ? 1 : -1;
    case 2: if (wt != 2) return 0; if (!sub_begin(r, &sub, budget)) return -1; m->has |= B2_HAS_RESPONSE;
            return parse_fields(&sub, budget - 1, cb_response, m, base) ? 1 : -1;
    case 3: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->compress_type = (int32_t)(uint32_t)v; m->has |= B2_HAS_COMPRESS_TYPE; return 1;
    case 4: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->correlation_id = (int64_t)v; m->has |= B2_HAS_CORRELATION_ID; return 1;
    case 5: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->attachment_size = (int32_t)(uint32_t)v; m->has |= B2_HAS_ATTACHMENT_SIZE; return 1;
    case 6: if (wt != 2) return 0; if (!sub_begin(r, &sub, budget)) return -1; m->has |= B2_HAS_CHUNK_INFO;
            return parse_fields(&sub, budget - 1, cb_chunk, m, base) ? 1 : -1;
    case 7: if (wt != 2) return 0; if (!rd_bytes_span(r, &m->authentication_data, base)) return -1; m->has |= B2_HAS_AUTH_DATA; return 1;
    case 8: if (wt != 2) return 0; if (!sub_begin(r, &sub, budget)) return -1; m->has |= B2_HAS_STREAM_SETTINGS;
            return parse_fields(&sub, budget - 1, cb_stream_settings, m, base) ? 1 : -1;
    case 9: if (wt != 2) return 0; if (!sub_begin(r, &sub, budget)) return -1; m->has |= B2_HAS_USER_FIELDS; m->n_user_fields++;
            return parse_fields(&sub, budget - 1, cb_map_entry, m, base) ? 1 : -1;
    case 10: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1;
            {   /* closed proto2 enum ContentType (options.proto:83-88): unknown numbers
                   go to the unknown-field set and leave the field unset */
                int32_t e = (int32_t)(uint32_t)v;
                if (e >= 0 && e <= 3) { m->content_type = e; m->has |= B2_HAS_CONTENT_TYPE; }
            }
            return 1;
    case 11: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->checksum_type = (int32_t)(uint32_t)v; m->has |= B2_HAS_CHECKSUM_TYPE; return 1;
    case 12: if (wt != 2) return 0; if (!rd_bytes_span(r, &m->checksum_value, base)) return -1; m->has |= B2_HAS_CHECKSUM_VALUE; return 1;
    }
    return 0;
}
int orc_parse_rpc_meta(const uint8_t* p, size_t n, orc_rpc_meta* m) {
    rd_t r = { p, p + n };
    memset(m, 0, sizeof *m);
    if (!parse_fields(&r, 100, cb_rpc_meta, m, p)) return 0;
    /* IsInitialized(): required fields of present sub-messages */
    if ((m->has & B2_HAS_REQUEST) && !(m->has_service_name && m->has_method_name)) return 0;
    if ((m->has & B2_HAS_CHUNK_INFO) && !(m->chunk_has_stream_id && m->chunk_has_chunk_id)) return 0;
    if ((m->has & B2_HAS_STREAM_SETTINGS) && !m->ss_has_stream_id) return 0;
    return 1;
}

/* StreamFrameMeta + Feedback, streaming_rpc_meta.proto:39-53 */
static int cb_feedback(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_stream_meta* m = (orc_stream_meta*)c; uint64_t v; (void)budget; (void)base;
    if (fn == 1 && wt == 0) { if (!rd_varint(r, &v)) return -1; m->consumed_size = (int64_t)v; m->feedback_has_consumed_size = 1; return 1; }
    return 0;
}
static int cb_stream_meta(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    orc_stream_meta* m = (orc_stream_meta*)c; uint64_t v; rd_t sub;
    switch (fn) {
    case 1: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->stream_id = (int64_t)v; m->has |= B2_SHAS_STREAM_ID; return 1;
    case 2: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->source_stream_id = (int64_t)v; m->has |= B2_SHAS_SOURCE_STREAM_ID; return 1;
    case 3: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1;
            { int32_t e = (int32_t)(uint32_t)v; if (e >= 0 && e <= 4) { m->frame_type = e; m->has |= B2_SHAS_FRAME_TYPE; } }
            return 1;
    case 4: if (wt != 0) return 0; if (!rd_varint(r, &v)) return -1; m->has |= B2_SHAS_HAS_CONTINUATION;
            if (v != 0) m->has |= B2_SVAL_HAS_CONTINUATION; else m->has &= ~B2_SVAL_HAS_CONTINUATION; return 1;
    case 5: if (wt != 2) return 0; if (!sub_begin(r, &sub, budget)) return -1; m->has |= B2_SHAS_FEEDBACK;
            return parse_fields(&sub, budget - 1, cb_feedback, m, base) ? 1 : -1;
    }
    return 0;
}
int orc_parse_stream_meta(const uint8_t* p, size_t n, orc_stream_meta* m) {
    rd_t r = { p, p + n };
    memset(m, 0, sizeof *m);
    if (!parse_fields(&r, 100, cb_stream_meta, m, p)) return 0;
    return (m->has & B2_SHAS_STREAM_ID) != 0;   /* required int64 stream_id = 1 */
}

/* EchoRequest, example/echo_c++/echo.proto:23-25 (required string message = 1) */
typedef struct { orc_span msg; int has; } echo_ctx;
static int cb_echo(void* c, uint32_t fn, uint32_t wt, rd_t* r, int budget, const uint8_t* base) {
    echo_ctx* e = (echo_ctx*)c; (void)budget;
    if (fn == 1 && wt == 2) { if (!rd_bytes_span(r, &e->msg, base)) return -1; e->has = 1; return 1; }
    return 0;
}
int orc_parse_echo_request(const uint8_t* p, size_t n, orc_span* message) {
    rd_t r = { p, p + n }; echo_ctx e; memset(&e, 0, sizeof e);
    if (!parse_fields(&r, 100, cb_echo, &e, p)) return 0;
    if (!e.has) return 0;
    *message = e.msg;
    return 1;
}

/* ------------------------------------------------------------------------ */
/* encoders: CodedOutputStream varint / tag writers */
typedef struct { uint8_t* p; uint8_t* end; int ovf; } wr_t;
static void wr_byte(wr_t* w, uint8_t b) { if (w->p < w->end) *w->p++ = b; else w->ovf = 1; }
static void wr_raw(wr_t* w, const void* s, size_t n) {
    if ((size_t)(w->end - w->p) < n) { w->ovf = 1; return; }
    memcpy(w->p, s, n); w->p += n;
}
static void wr_varint(wr_t* w, uint64_t v) { while (v >= 0x80) { wr_byte(w, (uint8_t)(v | 0x80)); v >>= 7; } wr_byte(w, (uint8_t)v); }
static size_t varint_len(uint64_t v) { size_t n = 1; while (v >= 0x80) { v >>= 7; n++; } return n; }
static void wr_i32(wr_t* w, uint32_t fn, int32_t v) { wr_varint(w, (fn << 3) | 0); wr_varint(w, (uint64_t)(int64_t)v); }  /* int32: sign-extended */
static void wr_i64(wr_t* w, uint32_t fn, int64_t v) { wr_varint(w, (fn << 3) | 0); wr_varint(w, (uint64_t)v); }
static void wr_len(wr_t* w, uint32_t fn, const void* s, size_t n) { wr_varint(w, (fn << 3) | 2); wr_varint(w, n); wr_raw(w, s, n); }
static void wr_be32(wr_t* w, uint32_t v) { uint8_t b[4] = { (uint8_t)(v >> 24), (uint8_t)(v >> 16), (uint8_t)(v >> 8), (uint8_t)v }; wr_raw(w, b, 4); } /* raw_pack.h:43-58 */

/* PackRpcHeader, baidu_rpc_protocol.cpp:75-81 */
static void pack_header(wr_t* w, const char* magic, uint32_t meta_size, uint32_t payload_size) {
    wr_raw(w, magic, 4); wr_be32(w, meta_size + payload_size); wr_be32(w, meta_size);
}

/* SerializeRpcMessage for EchoRequest with COMPRESS_TYPE_NONE/SNAPPY + checksum
 * (baidu_rpc_protocol.cpp:148-216); returns body length, fills checksum bytes */
static size_t serialize_echo_body(const uint8_t* msg, uint32_t len, int32_t compress_type,
                                  int32_t checksum_type, uint8_t* out, size_t cap, uint8_t cks[4], int* cks_len) {
    size_t pb_len = 1 + varint_len(len) + len, body_len = 0;
    *cks_len = 0;
    if (compress_type == B2_COMPRESS_TYPE_SNAPPY) {
        uint8_t* pb = (uint8_t*)malloc(pb_len ? pb_len : 1);
        wr_t w = { pb, pb + pb_len, 0 };
        wr_len(&w, 1, msg, len);
        if (orc_snappy_max_compressed_length(pb_len) > cap) { free(pb); return (size_t)-1; }
        body_len = orc_snappy_compress(pb, pb_len, out);
        free(pb);
    } else {
        wr_t w = { out, out + cap, 0 };
        wr_len(&w, 1, msg, len);
        if (w.ovf) return (size_t)-1;
        body_len = pb_len;
    }
    if (checksum_type == B2_CHECKSUM_TYPE_CRC32C) {      /* Crc32cCompute, crc32c_checksum.cpp:28-42 */
        uint32_t c = orc_crc32c_mask(orc_crc32c_extend(0, out, body_len));
        cks[0] = (uint8_t)(c >> 24); cks[1] = (uint8_t)(c >> 16); cks[2] = (uint8_t)(c >> 8); cks[3] = (uint8_t)c;
        *cks_len = 4;
    }
    return body_len;
}

/* PackRpcRequest, baidu_rpc_protocol.cpp:1045-1133 */
size_t orc_pack_echo_request(const orc_request_spec* s, uint8_t* out, size_t cap) {
    size_t body_cap = 64 + (size_t)s->message_len + s->message_len / 5;
    uint8_t* body = (uint8_t*)malloc(body_cap);
    uint8_t cks[4]; int cks_len = 0;
    size_t body_len = serialize_echo_body(s->message, s->message_len, s->compress_type, s->checksum_type,
                                          body, body_cap, cks, &cks_len);
    if (body_len == (size_t)-1) { free(body); return 0; }
    uint8_t req[1024]; wr_t rw = { req, req + sizeof req, 0 };
    wr_len(&rw, 1, s->service_name, strlen(s->service_name));
    wr_len(&rw, 2, s->method_name, strlen(s->method_name));
    if (s->has_log_id) wr_i64(&rw, 3, s->log_id);
    if (s->has_trace) { wr_i64(&rw, 4, s->trace_id); wr_i64(&rw, 5, s->span_id); wr_i64(&rw, 6, s->parent_span_id); }
    if (s->request_id && s->request_id[0]) wr_len(&rw, 7, s->request_id, strlen(s->request_id));
    if (s->timeout_ms > 0) wr_i32(&rw, 8, s->timeout_ms);
    uint8_t meta[1400]; wr_t mw = { meta, meta + sizeof meta, 0 };
    wr_len(&mw, 1, req, (size_t)(rw.p - req));
    wr_i32(&mw, 3, s->compress_type);
    wr_i64(&mw, 4, s->correlation_id);
    if (s->attachment_len) wr_i32(&mw, 5, (int32_t)s->attachment_len);
    wr_i32(&mw, 10, s->content_type);
    wr_i32(&mw, 11, s->checksum_type);
    wr_len(&mw, 12, cks, (size_t)cks_len);
    if (rw.ovf || mw.ovf) { free(body); return 0; }
    uint32_t meta_size = (uint32_t)(mw.p - meta);
    wr_t w = { out, out + cap, 0 };
    pack_header(&w, "PRPC", meta_size, (uint32_t)(body_len + s->attachment_len));
    wr_raw(&w, meta, meta_size);
    wr_raw(&w, body, body_len);
    if (s->attachment_len) wr_raw(&w, s->attachment, s->attachment_len);
    free(body);
    return w.ovf ? 0 : (size_t)(w.p - out);
}

/* PackStreamMessage, streaming_rpc_protocol.cpp:42-58 (fields set as in
 * SendStreamData :165-172 / stream.cpp:181-186) */
size_t orc_pack_stream_frame(int64_t stream_id, int64_t source_stream_id, int frame_type,
                             int has_continuation, int cont_value,
                             const uint8_t* data, uint32_t data_len, uint8_t* out, size_t cap) {
    uint8_t meta[64]; wr_t mw = { meta, meta + sizeof meta, 0 };
    wr_i64(&mw, 1, stream_id);
    if (source_stream_id >= 0) wr_i64(&mw, 2, source_stream_id);
    wr_i32(&mw, 3, frame_type);
    if (has_continuation) { wr_varint(&mw, (4 << 3) | 0); wr_varint(&mw, cont_value ? 1 : 0); }
    uint32_t meta_size = (uint32_t)(mw.p - meta);
    wr_t w = { out, out + cap, 0 };
    pack_header(&w, "STRM", meta_size, data_len);
    wr_raw(&w, meta, meta_size);
    if (data_len) wr_raw(&w, data, data_len);
    return w.ovf ? 0 : (size_t)(w.p - out);
}

/* ------------------------------------------------------------------------ */
/* Protocol::parse of baidu_std and streaming_rpc over a flat run.
 * ParseRpcMessage (policy/baidu_rpc_protocol.cpp:105-146) and
 * ParseStreamingMessage (policy/streaming_rpc_protocol.cpp:61-96) share the
 * 12-byte header logic; only the magic differs.                              */
typedef struct { int err; uint32_t pop; uint32_t body_size, meta_size; } cut_t;
static cut_t parse_prefixed(const uint8_t* p, uint64_t n, const char* magic, uint64_t max_body) {
    cut_t c = { B2_PARSE_OK, 0, 0, 0 };
    if (n >= 4) { if (memcmp(p, magic, 4) != 0) { c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; } }
    else        { if (memcmp(p, magic, (size_t)n) != 0) { c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; } }
    if (n < 12) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    uint32_t body = ((uint32_t)p[4] << 24) | ((uint32_t)p[5] << 16) | ((uint32_t)p[6] << 8) | p[7];   /* RawUnpacker, raw_pack.h:76-80 */
    uint32_t meta = ((uint32_t)p[8] << 24) | ((uint32_t)p[9] << 16) | ((uint32_t)p[10] << 8) | p[11];
    if ((uint64_t)body > max_body) { c.err = B2_PARSE_ERROR_TOO_BIG_DATA; return c; }
    if (n < 12 + (uint64_t)body) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    if (meta > body) { c.pop = 12 + body; c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; }   /* pop the message */
    c.pop = 12 + body; c.body_size = body; c.meta_size = meta;
    return c;
}
static const char* k_magic[5] = { NULL, "PRPC", "STRM", "HULU", "SOFA" };   /* handler index == ProtocolType */
static uint32_t le32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
static uint64_t le64(const uint8_t* p) { return (uint64_t)le32(p) | ((uint64_t)le32(p + 4) << 32); }

/* ParseHuluMessage, policy/hulu_pbrpc_protocol.cpp:178-223: "HULU", body_size and meta_size in HOST order (HuluRawUnpacker :110-135) */
static cut_t parse_hulu(const uint8_t* p, uint64_t n, uint64_t max_body) {
    cut_t c = { B2_PARSE_OK, 0, 0, 0 };
    if (memcmp(p, "HULU", n >= 4 ? 4 : (size_t)n) != 0) { c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; }
    if (n < 12) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    uint32_t body = le32(p + 4);
    if ((uint64_t)body > max_body) { c.err = B2_PARSE_ERROR_TOO_BIG_DATA; return c; }
    if (n < 12 + (uint64_t)body) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    uint32_t meta = le32(p + 8);
    if (meta > body) { c.pop = 12 + body; c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; }   /* pop the message */
    c.pop = 12 + body; c.body_size = body; c.meta_size = meta;
    return c;
}
/* ParseSofaMessage, policy/sofa_pbrpc_protocol.cpp:165-205: 24-byte header "SOFA" meta_size(32) body_size(64) msg_size(64) */
static cut_t parse_sofa(const uint8_t* p, uint64_t n, uint64_t max_body) {
    cut_t c = { B2_PARSE_OK, 0, 0, 0 };
    if (memcmp(p, "SOFA", n >= 4 ? 4 : (size_t)n) != 0) { c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; }
    if (n < 24) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    uint32_t meta = le32(p + 4); uint64_t body = le64(p + 8), msg = le64(p + 16);
    if (msg != (uint64_t)meta + body) { c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; }
    if (body > max_body) { c.err = B2_PARSE_ERROR_TOO_BIG_DATA; return c; }
    if (n < 24 + msg) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    c.pop = 24 + (uint32_t)msg; c.body_size = (uint32_t)msg; c.meta_size = meta;      /* descriptor: the bytes behind the header */
    return c;
}
/* ParseNsheadMessage, policy/nshead_protocol.cpp:154-182 over nshead_t (src/brpc/nshead.h:28-36): magic_num at +24, body_len at +32 */
static cut_t parse_nshead(const uint8_t* p, uint64_t n, uint64_t max_body) {
    cut_t c = { B2_PARSE_OK, 0, 0, 0 };
    if (n < 28) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    if (le32(p + 24) != 0xfb709394u) { c.err = B2_PARSE_ERROR_TRY_OTHERS; return c; }
    if (n < 36) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    uint32_t body = le32(p + 32);
    if ((uint64_t)body > max_body) { c.err = B2_PARSE_ERROR_TOO_BIG_DATA; return c; }
    if (n < 36 + (uint64_t)body) { c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA; return c; }
    c.pop = 36 + body; c.body_size = body; c.meta_size = 0;
    return c;
}
static cut_t parse_handler(int idx, const uint8_t* p, uint64_t n, uint64_t max_body) {
    if (idx == 3) return parse_hulu(p, n, max_body);
    if (idx == 4) return parse_sofa(p, n, max_body);
    if (idx == 12) return parse_nshead(p, n, max_body);
    return parse_prefixed(p, n, k_magic[idx], max_body);
}

/* InputMessenger::CutInputMessage, input_messenger.cpp:84-179, over the handlers enabled in `mask` (_handlers[i].parse != NULL),
 * probed in index order.  *pos advances by what the handlers popped.             */
static cut_t cut_input_message(const uint8_t* run, uint32_t len, uint32_t* pos, int* preferred,
                               int* index, uint64_t max_body, int created_by_connect, uint32_t mask) {
    const int max_index = 12;
    const int pref = *preferred;
    cut_t c;
    if (pref >= 0 && pref <= max_index && ((mask >> pref) & 1u)) {
        int cur_index = pref;
        do {
            c = parse_handler(cur_index, run + *pos, len - *pos, max_body);
            if (c.err == B2_PARSE_OK || c.err == B2_PARSE_ERROR_NOT_ENOUGH_DATA) {
                if (c.err == B2_PARSE_OK) *pos += c.pop;
                *preferred = cur_index; *index = cur_index; return c;
            } else if (c.err != B2_PARSE_ERROR_TRY_OTHERS) {
                return c;
            }
            *pos += c.pop;
            if (len - *pos >= 4 && memcmp(run + *pos, "RDMA", 4) == 0) { c.pop = 0; return c; }   /* :111-119 */
            if (created_by_connect) {                                                            /* :122-138 */
                if (cur_index == B2_PROTOCOL_BAIDU_STD && cur_index == pref) { cur_index = B2_PROTOCOL_STREAMING_RPC; continue; }
                else if (cur_index == B2_PROTOCOL_STREAMING_RPC && cur_index == pref) { cur_index = B2_PROTOCOL_BAIDU_STD; continue; }
                else { c.err = B2_PARSE_ERROR_ABSOLUTELY_WRONG; c.pop = 0; return c; }
            } else break;
        } while (1);
        *preferred = -1;
    }
    for (int i = 0; i <= max_index; i++) {
        if (i == pref || !((mask >> i) & 1u)) continue;
        c = parse_handler(i, run + *pos, len - *pos, max_body);
        if (c.err == B2_PARSE_OK || c.err == B2_PARSE_ERROR_NOT_ENOUGH_DATA) {
            if (c.err == B2_PARSE_OK) *pos += c.pop;
            *preferred = i; *index = i; return c;
        } else if (c.err != B2_PARSE_ERROR_TRY_OTHERS) {
            return c;
        }
        *pos += c.pop;
    }
    c.err = B2_PARSE_ERROR_TRY_OTHERS; c.pop = 0;
    return c;
}

/* ------------------------------------------------------------------------ */
/* Controller::SetFailed text, controller.cpp:468-495 + AppendServerIdentiy :407-428 */
static size_t fmt_error_text(char* out, size_t cap, const char* identity, int code, const char* reason, size_t reason_len) {
    size_t n = 0;
    if (identity) n += (size_t)snprintf(out + n, cap - n, "[%s]", identity);
    n += (size_t)snprintf(out + n, cap - n, "[E%d]", code);
    if (n + reason_len > cap) reason_len = cap - n;
    memcpy(out + n, reason, reason_len);
    return n + reason_len;
}
static const char* content_type_cstr(int32_t t) {   /* baidu_rpc_protocol.cpp:1135-1148 */
    switch (t) { case 0: return "pb"; case 1: return "json"; case 2: return "proto-json"; case 3: return "proto-text"; }
    return "unknown";
}
static const char* compress_type_cstr(int32_t t) {  /* compress.cpp:63-69 + global.cpp:400-411 */
    switch (t) { case 0: return "none"; case 1: return "snappy"; case 2: return "gzip"; case 3: return "zlib"; }
    return "unknown";
}
static const char* checksum_type_cstr(int32_t t) {  /* checksum.cpp:60-66 + global.cpp:414-418 */
    switch (t) { case 0: return "none"; case 1: return "crc32c"; }
    return "unknown";
}

/* SendRpcResponse (baidu_rpc_protocol.cpp:273-460): meta build :339-349 +
 * SerializeRpcHeaderAndMeta :83-103 + append body/attachment :384-389.     */
static size_t send_rpc_response(uint8_t* out, size_t cap, int32_t error_code,
                                const char* error_text, size_t error_text_len,
                                int64_t correlation_id, int32_t compress_type, int32_t content_type,
                                int32_t checksum_type, const uint8_t* cks, size_t cks_len,
                                const uint8_t* body, size_t body_len,
                                const uint8_t* att, size_t att_len, int append_body) {
    uint8_t rm[8192]; wr_t rw = { rm, rm + sizeof rm, 0 };
    wr_i32(&rw, 1, error_code);
    if (error_text_len) wr_len(&rw, 2, error_text, error_text_len);
    size_t meta_cap = 64 + (size_t)(rw.p - rm) + cks_len;
    uint8_t* meta = (uint8_t*)malloc(meta_cap); wr_t mw = { meta, meta + meta_cap, 0 };
    wr_len(&mw, 2, rm, (size_t)(rw.p - rm));
    wr_i32(&mw, 3, compress_type);
    wr_i64(&mw, 4, correlation_id);
    if (append_body && att_len > 0) wr_i32(&mw, 5, (int32_t)att_len);
    wr_i32(&mw, 10, content_type);
    wr_i32(&mw, 11, checksum_type);
    wr_len(&mw, 12, cks, cks_len);
    uint32_t meta_size = (uint32_t)(mw.p - meta);
    size_t payload = append_body ? body_len + att_len : 0;
    wr_t w = { out, out + cap, 0 };
    pack_header(&w, "PRPC", meta_size, (uint32_t)payload);
    wr_raw(&w, meta, meta_size);
    if (append_body) { wr_raw(&w, body, body_len); if (att_len) wr_raw(&w, att, att_len); }
    int bad = rw.ovf || mw.ovf || w.ovf;
    free(meta);
    return bad ? (size_t)-1 : (size_t)(w.p - out);
}

/* SendRpcResponse for a reply the HOST produced (the checker of b2_pack_responses): SerializeResponse :218-246 (compress, then
 * checksum over what goes on the wire), error / append_body rules :316-337, RpcMeta :339-380 incl. stream_settings
 * (Stream::FillSettings, stream.cpp:678-682) and user_fields in the order given, SerializeRpcHeaderAndMeta :83-103.
 * Returns the frame length, 0 when the reply cannot be packed (gzip / zlib), (size_t)-1 when out is too small. */
size_t orc_pack_response(const b2_reply* r, const uint8_t* bytes, uint8_t* out, size_t cap) {
    const int32_t err = r->error_code == -1 ? B2_EINTERNAL : r->error_code;
    const int append_body = err == 0;
    if (append_body && r->compress_type != B2_COMPRESS_TYPE_NONE && r->compress_type != B2_COMPRESS_TYPE_SNAPPY) return 0;
    uint8_t* body = NULL; size_t body_len = 0; uint8_t cks4[4];
    const uint8_t* cks = bytes + r->checksum_value_off; size_t cks_len = r->checksum_value_len;
    if (append_body) {
        if (r->compress_type == B2_COMPRESS_TYPE_SNAPPY) {
            body = (uint8_t*)malloc(orc_snappy_max_compressed_length(r->body_len));
            body_len = orc_snappy_compress(bytes + r->body_off, r->body_len, body);
        } else { body = (uint8_t*)malloc(r->body_len ? r->body_len : 1); memcpy(body, bytes + r->body_off, r->body_len); body_len = r->body_len; }
        if (r->checksum_type == B2_CHECKSUM_TYPE_CRC32C) {
            const uint32_t c = orc_crc32c_mask(orc_crc32c_extend(0, body, body_len));
            cks4[0] = (uint8_t)(c >> 24); cks4[1] = (uint8_t)(c >> 16); cks4[2] = (uint8_t)(c >> 8); cks4[3] = (uint8_t)c;
            cks = cks4; cks_len = 4;
        }
    }
    const size_t att_len = append_body ? r->attachment_len : 0;
    size_t meta_cap = 256 + r->error_text_len + cks_len + 11u * (size_t)r->n_extra_streams;
    { const uint8_t* uf = bytes + r->user_fields_off;
      for (uint32_t k = 0; k < r->n_user_fields; k++) { uint32_t kl, vl; memcpy(&kl, uf, 4); memcpy(&vl, uf + 4, 4); meta_cap += 24u + kl + vl; uf += 8u + kl + vl; } }
    uint8_t* rm = (uint8_t*)malloc(32 + r->error_text_len); wr_t rw = { rm, rm + 32 + r->error_text_len, 0 };
    wr_i32(&rw, 1, err);
    if (r->error_text_len) wr_len(&rw, 2, bytes + r->error_text_off, r->error_text_len);
    uint8_t* meta = (uint8_t*)malloc(meta_cap); wr_t mw = { meta, meta + meta_cap, 0 };
    wr_len(&mw, 2, rm, (size_t)(rw.p - rm));
    wr_i32(&mw, 3, r->compress_type);
    wr_i64(&mw, 4, r->correlation_id);
    if (att_len) wr_i32(&mw, 5, (int32_t)att_len);
    if (r->flags & B2_RSP_HAS_STREAM) {
        size_t sc = 32 + 11u * (size_t)r->n_extra_streams; uint8_t* ss = (uint8_t*)malloc(sc); wr_t sw = { ss, ss + sc, 0 };
        wr_i64(&sw, 1, r->stream_id);
        wr_varint(&sw, (2 << 3) | 0); wr_varint(&sw, (r->flags & B2_RSP_STREAM_NEED_FEEDBACK) ? 1 : 0);
        wr_varint(&sw, (3 << 3) | 0); wr_varint(&sw, (r->flags & B2_RSP_STREAM_WRITABLE) ? 1 : 0);
        for (uint32_t k = 0; k < r->n_extra_streams; k++) { int64_t v; memcpy(&v, bytes + r->extra_streams_off + 8u * k, 8); wr_i64(&sw, 4, v); }
        wr_len(&mw, 8, ss, (size_t)(sw.p - ss));
        if (sw.ovf) mw.ovf = 1;
        free(ss);
    }
    { const uint8_t* uf = bytes + r->user_fields_off;
      for (uint32_t k = 0; k < r->n_user_fields; k++) {
          uint32_t kl, vl; memcpy(&kl, uf, 4); memcpy(&vl, uf + 4, 4);
          size_t ec = 24u + kl + vl; uint8_t* e = (uint8_t*)malloc(ec); wr_t ew = { e, e + ec, 0 };
          wr_len(&ew, 1, uf + 8, kl); wr_len(&ew, 2, uf + 8 + kl, vl);
          wr_len(&mw, 9, e, (size_t)(ew.p - e));
          free(e); uf += 8u + kl + vl;
      } }
    wr_i32(&mw, 10, r->content_type);
    wr_i32(&mw, 11, r->checksum_type);
    wr_len(&mw, 12, cks, cks_len);
    const uint32_t meta_size = (uint32_t)(mw.p - meta);
    wr_t w = { out, out + cap, 0 };
    pack_header(&w, "PRPC", meta_size, (uint32_t)(body_len + att_len));
    wr_raw(&w, meta, meta_size);
    if (append_body) { wr_raw(&w, body, body_len); if (att_len) wr_raw(&w, bytes + r->attachment_off, att_len); }
    const int bad = rw.ovf || mw.ovf || w.ovf;
    free(rm); free(meta); free(body);
    return bad ? (size_t)-1 : (size_t)(w.p - out);
}

static const b2_method* find_method(const orc_config* cfg, const uint8_t* svc, uint32_t svc_len,
                                    const uint8_t* mth, uint32_t mth_len, int* idx, int* no_service) {
    /* baidu_rpc_protocol.cpp:738-756: a service name without '.' is looked up as a
     * short name first (jprotobuf) and replaced by the full name */
    const uint8_t* full = svc; uint32_t full_len = svc_len;
    *no_service = 0; *idx = -1;
    if (memchr(svc, '.', svc_len) == NULL) {
        const b2_method* sp = NULL;
        for (uint32_t i = 0; i < cfg->n_methods; i++)
            if (strlen(cfg->methods[i].service_name) == svc_len && memcmp(cfg->methods[i].service_name, svc, svc_len) == 0) { sp = &cfg->methods[i]; break; }
        if (!sp) { *no_service = 1; return NULL; }
        full = (const uint8_t*)sp->service_full_name; full_len = (uint32_t)strlen(sp->service_full_name);
    }
    /* Server::FindMethodPropertyByFullName(service, method), server.cpp:1970-1988:
     * key is the concatenation service + '.' + method */
    for (uint32_t i = 0; i < cfg->n_methods; i++) {
        const b2_method* m = &cfg->methods[i];
        size_t a = strlen(m->service_full_name), b = strlen(m->method_name);
        size_t klen = a + 1 + b;
        if (klen != (size_t)full_len + 1 + mth_len) continue;
        char* key = (char*)malloc(klen + 1), *cand = (char*)malloc(klen + 1);
        memcpy(key, m->service_full_name, a); key[a] = '.'; memcpy(key + a + 1, m->method_name, b);
        memcpy(cand, full, full_len); cand[full_len] = '.'; memcpy(cand + full_len + 1, mth, mth_len);
        int eq = memcmp(key, cand, klen) == 0;
        free(key); free(cand);
        if (eq) { *idx = (int)i; return m; }
    }
    return NULL;
}

/* ProcessRpcRequest (baidu_rpc_protocol.cpp:568-866) -> echo service
 * (example/echo_c++/server.cpp:44-84) -> SendRpcResponse, for one cut message. */
static int process_rpc_request(const orc_config* cfg, const uint8_t* frame, b2_msg_desc* d,
                               uint8_t* resp, size_t resp_cap, size_t* resp_len) {
    const uint8_t* meta_p = frame + 12;
    const uint8_t* payload = meta_p + d->meta_size;
    const uint32_t req_size = d->body_size - d->meta_size;
    orc_rpc_meta m;
    *resp_len = 0;
    d->method_idx = -1; d->error_code = 0;
    if (!orc_parse_rpc_meta(meta_p, d->meta_size, &m)) { d->status = B2_MSG_BAD_META; return 0; }   /* :577-582 */
    d->correlation_id = m.correlation_id; d->log_id = m.log_id;
    d->attachment_size = m.attachment_size; d->compress_type = m.compress_type;
    d->checksum_type = m.checksum_type; d->content_type = (uint8_t)m.content_type;
    d->has_bits = (uint16_t)m.has;

    char reason[2048]; int rl; char text[2300]; size_t tl;
    const uint8_t* req_cks = meta_p + m.checksum_value.off; size_t req_cks_len = m.checksum_value.len;
    if (!(m.has & B2_HAS_CHECKSUM_VALUE)) req_cks_len = 0;
    int err = 0;
    const b2_method* mp = NULL; int midx = -1, no_service = 0;
    int64_t att = m.attachment_size;
    do {
        if ((m.has & B2_HAS_ATTACHMENT_SIZE) && (int64_t)req_size < att) {                           /* :700-707 */
            err = B2_EREQUEST;
            rl = snprintf(reason, sizeof reason, "attachment_size=%d is larger than request_size=%d", m.attachment_size, (int)req_size);
            break;
        }
        const uint8_t* svc = meta_p + m.service_name.off; const uint8_t* mth = meta_p + m.method_name.off;
        uint32_t svc_len = m.service_name.len, mth_len = m.method_name.len;
        if (!(m.has & B2_HAS_REQUEST)) { svc_len = 0; mth_len = 0; }
        mp = find_method(cfg, svc, svc_len, mth, mth_len, &midx, &no_service);
        if (no_service) {                                                                              /* :741-746 */
            err = B2_ENOSERVICE;
            rl = snprintf(reason, sizeof reason, "Fail to find service=%.*s", (int)strnlen((const char*)svc, svc_len), (const char*)svc);
            break;
        }
        if (!mp) {                                                                                     /* :752-757 */
            err = B2_ENOMETHOD;
            rl = snprintf(reason, sizeof reason, "Fail to find method=%.*s/%.*s",
                          (int)strnlen((const char*)svc, svc_len), (const char*)svc,
                          (int)strnlen((const char*)mth, mth_len), (const char*)mth);
            break;
        }
        d->method_idx = (int16_t)midx;
    } while (0);
    if (!err && mp->handler == B2_HANDLER_HOST) { d->status = B2_MSG_HOST; return 0; }

    const uint8_t* body = NULL; size_t body_len = 0; uint8_t* owned = NULL; uint8_t* unz = NULL;
    const uint8_t* out_att = NULL; size_t out_att_len = 0;
    uint8_t cks_buf[4]; const uint8_t* cks = req_cks; size_t cks_len = req_cks_len;
    int32_t r_compress = 0, r_checksum = 0;
    if (!err) {
        /* :797-802 split payload / attachment */
        int64_t bwo = (int64_t)req_size - att;
        if (bwo > (int64_t)req_size) bwo = req_size;
        const uint8_t* req_buf = payload; size_t req_buf_len = (size_t)bwo;
        const uint8_t* in_att = payload + req_buf_len; size_t in_att_len = att > 0 ? (size_t)att : 0;
        /* DeserializeRpcMessage :498-566 */
        int ok = 1;
        if (m.content_type != B2_CONTENT_TYPE_PB) { d->status = B2_MSG_UNSUPPORTED; return 0; }
        /* scope decision (SURVEY §2 row 10): non-pb content types are outside this path; so are replies a method wants
         * gzip / zlib COMPRESSED (bit-exact deflate is zlib-version specific) — such requests are surfaced untouched, before any checksum work */
        if (mp->response_compress_type != B2_COMPRESS_TYPE_NONE && mp->response_compress_type != B2_COMPRESS_TYPE_SNAPPY) { d->status = B2_MSG_UNSUPPORTED; return 0; }
        /* device limit (one thread walks a DEFLATE stream): big gzip / zlib bodies go to the host as they are */
        if (m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB) {
            if (req_buf_len > ORC_GZ_MAX_IN) { d->status = B2_MSG_UNSUPPORTED; return 0; }
            if (!(m.checksum_type == B2_CHECKSUM_TYPE_CRC32C && req_cks_len != 4) &&
                orc_gzip_sizing_bound(req_buf, req_buf_len, m.compress_type, ORC_GZ_MAX_OUT) > ORC_GZ_MAX_OUT) { d->status = B2_MSG_UNSUPPORTED; return 0; }
        }
        if (m.checksum_type == B2_CHECKSUM_TYPE_CRC32C) {                  /* Crc32cVerify, crc32c_checksum.cpp:44-61 */
            if (req_cks_len != 4) ok = 0;   /* reference CHECK_EQ-aborts here; treated as a failed verify */
            else {
                uint32_t expected = ((uint32_t)req_cks[0] << 24) | ((uint32_t)req_cks[1] << 16) | ((uint32_t)req_cks[2] << 8) | req_cks[3];
                ok = orc_crc32c_extend(0, req_buf, req_buf_len) == orc_crc32c_unmask(expected);
            }
        }
        orc_span msg = { 0, 0 };
        const uint8_t* pb = req_buf; size_t pb_len = req_buf_len;
        if (ok) {
            if (m.compress_type == B2_COMPRESS_TYPE_NONE) {
            } else if (m.compress_type == B2_COMPRESS_TYPE_SNAPPY) {         /* SnappyDecompress, snappy_compress.cpp:51-70 */
                size_t ulen = 0;
                if (!orc_snappy_uncompressed_length(req_buf, req_buf_len, &ulen)) ok = 0;
                else {
                    unz = (uint8_t*)malloc(ulen ? ulen : 1);
                    size_t got = 0;
                    if (!orc_snappy_uncompress(req_buf, req_buf_len, unz, ulen, &got)) ok = 0;
                    pb = unz; pb_len = got;
                }
            } else if (m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB) {
                /* GzipDecompress / ZlibDecompress(const IOBuf&, Message*), gzip_compress.cpp:75-89: the parser reads what the
                 * GzipInputStream yields; a corrupt stream is end-of-input to it, not an error */
                size_t got = 0;
                if (orc_gzip_input_stream(req_buf, req_buf_len, m.compress_type, &unz, &got)) return -1;
                pb = unz; pb_len = got;
            } else ok = 0;                                                   /* FindCompressHandler == NULL */
        }
        if (ok) ok = orc_parse_echo_request(pb, pb_len, &msg);
        if (!ok) {                                                            /* :819-829 */
            err = B2_EREQUEST;
            rl = snprintf(reason, sizeof reason,
                          "Fail to parse request=%s, ContentType=%s, CompressType=%s, ChecksumType=%s, request_size=%d",
                          mp->request_type_name, content_type_cstr(m.content_type), compress_type_cstr(m.compress_type),
                          checksum_type_cstr(m.checksum_type), (int)req_size);
        } else {
            /* EchoServiceImpl::Echo: response->set_message(request->message()) */
            r_compress = mp->response_compress_type; r_checksum = mp->response_checksum_type;
            size_t cap = 64 + (size_t)msg.len + msg.len / 5;
            owned = (uint8_t*)malloc(cap);
            int cl = 0;
            body_len = serialize_echo_body(pb + msg.off, msg.len, r_compress, r_checksum, owned, cap, cks_buf, &cl);
            if (body_len == (size_t)-1) { free(owned); free(unz); d->status = B2_MSG_UNSUPPORTED; return 0; }
            body = owned;
            if (cl) { cks = cks_buf; cks_len = 4; }
            if (mp->echo_attachment) { out_att = in_att; out_att_len = in_att_len; }
        }
    }
    size_t n;
    if (err) {
        tl = fmt_error_text(text, sizeof text, cfg->server_identity, err, reason, (size_t)rl);
        n = send_rpc_response(resp, resp_cap, err, text, tl, m.correlation_id, 0, B2_CONTENT_TYPE_PB, 0,
                              req_cks, req_cks_len, NULL, 0, NULL, 0, 0);
        d->status = B2_MSG_ERROR_REPLIED; d->error_code = err;
    } else {
        n = send_rpc_response(resp, resp_cap, 0, NULL, 0, m.correlation_id, r_compress, B2_CONTENT_TYPE_PB, r_checksum,
                              cks, cks_len, body, body_len, out_att, out_att_len, 1);
        d->status = B2_MSG_ECHOED;
    }
    free(owned); free(unz);
    if (n == (size_t)-1) return -1;
    *resp_len = n;
    return 0;
}

/* ProcessRpcResponse (baidu_rpc_protocol.cpp:911-1013) for a channel whose response type is EchoResponse.
 * d->error_code = what Controller::SetFailed receives (0 = success); the message bytes are reported
 * in place (batch offset) or, for a snappy response, decompressed into resp. */
static int process_rpc_response(const uint8_t* frame, b2_msg_desc* d, uint8_t* resp, size_t resp_cap, size_t* resp_len) {
    const uint8_t* meta_p = frame + 12;
    const uint8_t* payload = meta_p + d->meta_size;
    const uint32_t res_size = d->body_size - d->meta_size;
    orc_rpc_meta m;
    *resp_len = 0; d->method_idx = -1; d->error_code = 0;
    if (!orc_parse_rpc_meta(meta_p, d->meta_size, &m)) { d->status = B2_MSG_BAD_META; return 0; }   /* :914-918: dropped */
    d->correlation_id = m.correlation_id; d->log_id = m.log_id; d->attachment_size = m.attachment_size;
    d->compress_type = m.compress_type; d->checksum_type = m.checksum_type; d->content_type = (uint8_t)m.content_type;
    d->has_bits = (uint16_t)m.has; d->status = B2_MSG_RESPONSE;
    if (m.error_code != 0) { d->error_code = m.error_code; return 0; }                               /* :960-965 */
    int64_t att = m.attachment_size;
    size_t body_len = res_size;
    if (m.has & B2_HAS_ATTACHMENT_SIZE) {
        if (att > (int64_t)res_size) { d->error_code = B2_ERESPONSE; return 0; }                      /* :971-976 */
        int64_t bwo = (int64_t)res_size - att; if (bwo > (int64_t)res_size) bwo = res_size;
        body_len = (size_t)bwo;
    }
    if (m.content_type != B2_CONTENT_TYPE_PB) { d->status = B2_MSG_UNSUPPORTED; return 0; }
    if (m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB) {      /* device limit, as on the request side */
        const size_t cl = (m.has & B2_HAS_CHECKSUM_VALUE) ? m.checksum_value.len : 0;
        if (body_len > ORC_GZ_MAX_IN) { d->status = B2_MSG_UNSUPPORTED; return 0; }
        if (!(m.checksum_type == B2_CHECKSUM_TYPE_CRC32C && cl != 4) &&
            orc_gzip_sizing_bound(payload, body_len, m.compress_type, ORC_GZ_MAX_OUT) > ORC_GZ_MAX_OUT) { d->status = B2_MSG_UNSUPPORTED; return 0; }
    }
    int ok = 1;
    const uint8_t* cks = meta_p + m.checksum_value.off; size_t cks_len = (m.has & B2_HAS_CHECKSUM_VALUE) ? m.checksum_value.len : 0;
    if (m.checksum_type == B2_CHECKSUM_TYPE_CRC32C) {
        if (cks_len != 4) ok = 0;
        else {
            uint32_t expected = ((uint32_t)cks[0] << 24) | ((uint32_t)cks[1] << 16) | ((uint32_t)cks[2] << 8) | cks[3];
            ok = orc_crc32c_extend(0, payload, body_len) == orc_crc32c_unmask(expected);
        }
    }
    orc_span msg = { 0, 0 };
    if (ok && m.compress_type == B2_COMPRESS_TYPE_NONE) {
        ok = orc_parse_echo_request(payload, body_len, &msg);       /* EchoResponse has the same schema */
        if (ok) { d->resp_off = d->frame_off + 12 + d->meta_size + msg.off; d->resp_len = msg.len; }
    } else if (ok && m.compress_type == B2_COMPRESS_TYPE_SNAPPY) {
        size_t ulen = 0, got = 0;
        if (!orc_snappy_uncompressed_length(payload, body_len, &ulen) || ulen > 32 * (uint64_t)body_len + 64 || ulen > resp_cap) ok = 0;
        else if (!orc_snappy_uncompress(payload, body_len, resp, ulen, &got)) ok = 0;
        else ok = orc_parse_echo_request(resp, got, &msg);
        if (ok) { d->status = B2_MSG_RESPONSE_UNZ; *resp_len = got; d->resp_len = msg.len; d->resp_off = msg.off; /* + slot, by caller */ }
    } else if (ok && (m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB)) {
        uint8_t* u = NULL; size_t got = 0;                                                           /* gzip_compress.cpp:75-89 */
        if (orc_gzip_input_stream(payload, body_len, m.compress_type, &u, &got)) return -1;
        if (got > resp_cap) { free(u); return -1; }
        memcpy(resp, u, got); free(u);
        ok = orc_parse_echo_request(resp, got, &msg);
        if (ok) { d->status = B2_MSG_RESPONSE_UNZ; *resp_len = got; d->resp_len = msg.len; d->resp_off = msg.off; }
    } else if (ok) ok = 0;                                                                           /* no such handler */
    if (!ok) { d->error_code = B2_EREQUEST; d->resp_off = 0; d->resp_len = 0; d->status = B2_MSG_RESPONSE; }   /* :999-1007 */
    return 0;
}

/* ParseStreamingMessage's meta step, streaming_rpc_protocol.cpp:95-100 */
static void process_stream_frame(const orc_config* cfg, const uint8_t* frame, b2_msg_desc* d, uint8_t* resp, size_t resp_cap, size_t* resp_len) {
    orc_stream_meta sm;
    d->method_idx = -1; d->error_code = 0; *resp_len = 0;
    if (!orc_parse_stream_meta(frame + 12, d->meta_size, &sm)) { d->status = B2_MSG_BAD_STREAM_META; return; }
    d->status = B2_MSG_STREAM_FRAME;
    d->correlation_id = sm.stream_id; d->log_id = sm.source_stream_id;
    d->compress_type = sm.frame_type; d->has_bits = (uint16_t)sm.has;
    d->attachment_size = (int32_t)(uint32_t)((uint64_t)sm.consumed_size & 0xffffffffu);
    d->checksum_type = (int32_t)(uint32_t)((uint64_t)sm.consumed_size >> 32);
    if (cfg->stream_handler == B2_STREAM_SNAPPY_UNCOMPRESS && (sm.has & B2_SHAS_FRAME_TYPE) && sm.frame_type == 3) {
        /* policy::SnappyDecompress(IOBuf, IOBuf), snappy_compress.cpp:77-82, on the frame payload */
        const uint8_t* data = frame + 12 + d->meta_size; const size_t n = d->body_size - d->meta_size;
        size_t ulen = 0, got = 0;
        if (!orc_snappy_uncompressed_length(data, n, &ulen) || ulen > 32 * (uint64_t)n + 64 || ulen > resp_cap ||
            !orc_snappy_uncompress(data, n, resp, ulen, &got)) { d->error_code = B2_EREQUEST; return; }
        *resp_len = got;
    }
}


/* ---- rpc_dump replay source (SURVEY 8f rank 4) --------------------------------------------------------------------------
 * A dump file is a sequence of records "PRPC" BE32(meta+request) BE32(meta) RpcDumpMeta request (RpcDumpContext::Serialize,
 * src/brpc/rpc_dump.cpp:237-258), read back by SampleIterator::Pop (:322-361).  rpc_replay (tools/rpc_replay/rpc_replay.cpp:148-200) sends
 * every sample through a Channel of its protocol_type with cntl->reset_sampled_request(sample); for baidu_std PackRpcRequest then takes the
 * replay branch (baidu_rpc_protocol.cpp:1067-1075): service/method names from the sample, compress_type from the sample when it has one,
 * no checksum fields; the request bytes are the sample's (the last attachment_size bytes travel as the attachment). */
typedef struct { uint32_t has; orc_span service_name, method_name; int32_t compress_type, protocol_type, attachment_size; } dump_meta_t;
static int parse_dump_meta(const uint8_t* p, size_t n, dump_meta_t* o) {      /* rpc_dump.proto:23-48, all optional */
    rd_t r = { p, p + n };
    memset(o, 0, sizeof *o);
    while (r.p < r.end) {
        uint32_t tag;
        if (!rd_tag(&r, &tag)) return 0;
        if (tag == 0 || (tag & 7) == 4 || (tag >> 3) == 0) return 0;
        uint32_t fn = tag >> 3, wt = tag & 7; uint64_t v; int handled = 0;
        if (wt == 2 && (fn == 1 || fn == 2 || (fn >= 7 && fn <= 9))) {
            uint32_t len;
            if (!rd_size(&r, &len)) return 0;
            if (fn == 1) { o->service_name.off = (uint32_t)(r.p - p); o->service_name.len = len; o->has |= 1; }
            else if (fn == 2) { o->method_name.off = (uint32_t)(r.p - p); o->method_name.len = len; o->has |= 2; }
            r.p += len; handled = 1;
        } else if (wt == 0 && fn >= 3 && fn <= 6) {
            if (!rd_varint(&r, &v)) return 0;
            int32_t e = (int32_t)(uint32_t)v; handled = 1;
            if (fn == 4) { if (e >= 0 && e <= 4) { o->compress_type = e; o->has |= 4; } }          /* closed enum CompressType, options.proto:69-75 */
            else if (fn == 5) { if (e >= 0 && e <= 27) { o->protocol_type = e; o->has |= 8; } }      /* closed enum ProtocolType, :38-67 */
            else if (fn == 6) { o->attachment_size = e; o->has |= 16; }
        }
        if (!handled && !skip_field(&r, tag, 100)) return 0;
    }
    return 1;
}
static int process_dump_record(const uint8_t* frame, b2_msg_desc* d, int64_t correlation_id, uint8_t* resp, size_t resp_cap, size_t* resp_len) {
    dump_meta_t m;
    *resp_len = 0; d->method_idx = -1;
    if (!parse_dump_meta(frame + 12, d->meta_size, &m)) { d->status = B2_MSG_BAD_META; return 0; }     /* "Fail to parse RpcDumpMeta": format error */
    d->protocol = (uint8_t)m.protocol_type; d->compress_type = m.compress_type; d->attachment_size = m.attachment_size; d->has_bits = (uint16_t)m.has;
    d->correlation_id = correlation_id;
    if (m.protocol_type != B2_PROTOCOL_BAIDU_STD) { d->status = B2_MSG_UNSUPPORTED; return 0; }
    const uint32_t req = d->body_size - d->meta_size;
    const uint32_t att = m.attachment_size > 0 ? (uint32_t)m.attachment_size : 0;
    uint8_t rq[1200]; wr_t rw = { rq, rq + sizeof rq, 0 };
    wr_len(&rw, 1, frame + 12 + m.service_name.off, m.service_name.len);
    wr_len(&rw, 2, frame + 12 + m.method_name.off, m.method_name.len);
    uint8_t meta[1400]; wr_t mw = { meta, meta + sizeof meta, 0 };
    wr_len(&mw, 1, rq, (size_t)(rw.p - rq));
    wr_i32(&mw, 3, m.compress_type);
    wr_i64(&mw, 4, correlation_id);
    if (att) wr_i32(&mw, 5, (int32_t)att);
    wr_i32(&mw, 10, 0);
    if (rw.ovf || mw.ovf) { d->status = B2_MSG_UNSUPPORTED; return 0; }
    uint32_t ml = (uint32_t)(mw.p - meta);
    wr_t w = { resp, resp + resp_cap, 0 };
    pack_header(&w, "PRPC", ml, req);
    wr_raw(&w, meta, ml); wr_raw(&w, frame + 12 + d->meta_size, req);
    if (w.ovf) return -1;
    d->status = B2_MSG_REPLAY; *resp_len = (size_t)(w.p - resp);
    return 0;
}

/* InputMessenger::ProcessNewMessage, input_messenger.cpp:206-322, per run. */
int orc_process_batch(const orc_config* cfg, const uint8_t* bytes, uint32_t nbytes,
                      const b2_run* runs, uint32_t n_runs, b2_run_status* rs,
                      b2_msg_desc* msgs, uint32_t msg_cap, uint32_t* n_msgs,
                      uint8_t* resp, uint32_t resp_cap, uint32_t* resp_bytes) {
    uint32_t nm = 0; size_t rb = 0;
    uint64_t max_body = cfg->max_body_size ? cfg->max_body_size : (64ull << 20);
    const uint32_t mask = cfg->protocols ? cfg->protocols : ((1u << 1) | (1u << 2));
    (void)nbytes;
    for (uint32_t r = 0; r < n_runs; r++) {
        const uint8_t* run = bytes + runs[r].offset;
        const uint32_t len = runs[r].length;
        uint32_t pos = 0; int preferred = runs[r].preferred_proto; int index = -1;
        memset(&rs[r], 0, sizeof rs[r]);
        rs[r].first_msg = nm; rs[r].resp_off = (uint32_t)rb;
        for (;;) {
            uint32_t before = pos;
            const int client = (runs[r].flags & B2_RUN_CLIENT) != 0;
            cut_t c;
            if (runs[r].flags & B2_RUN_RPC_DUMP) {          /* SampleIterator::Pop: baidu_std header, malformed = format error, nothing popped */
                memset(&c, 0, sizeof c); index = B2_PROTOCOL_BAIDU_STD;
                const uint32_t n = len - pos; const uint8_t* p = run + pos;
                if (n < 12) c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA;
                else if (memcmp(p, "PRPC", 4) != 0) c.err = B2_PARSE_ERROR_ABSOLUTELY_WRONG;
                else {
                    uint32_t body = ((uint32_t)p[4] << 24) | ((uint32_t)p[5] << 16) | ((uint32_t)p[6] << 8) | p[7];
                    uint32_t meta = ((uint32_t)p[8] << 24) | ((uint32_t)p[9] << 16) | ((uint32_t)p[10] << 8) | p[11];
                    if ((uint64_t)body > max_body) c.err = B2_PARSE_ERROR_ABSOLUTELY_WRONG;
                    else if ((uint64_t)n < 12ull + body) c.err = B2_PARSE_ERROR_NOT_ENOUGH_DATA;
                    else if (meta > body) c.err = B2_PARSE_ERROR_ABSOLUTELY_WRONG;
                    else { c.err = B2_PARSE_OK; c.pop = 12 + body; c.body_size = body; c.meta_size = meta; pos += c.pop; preferred = B2_PROTOCOL_BAIDU_STD; }
                }
            } else c = cut_input_message(run, len, &pos, &preferred, &index, max_body, client, mask);
            if (c.err != B2_PARSE_OK) { rs[r].parse_error = (uint32_t)c.err; break; }
            if (nm >= msg_cap) return -1;
            b2_msg_desc* d = &msgs[nm];
            memset(d, 0, sizeof *d);
            d->run_idx = r; d->frame_off = runs[r].offset + (pos - c.pop);
            d->body_size = c.body_size; d->meta_size = c.meta_size; d->protocol = (uint8_t)index;
            (void)before;
            size_t rl = 0;
            if (runs[r].flags & B2_RUN_RPC_DUMP) {
                d->protocol = 0;
                if (process_dump_record(bytes + d->frame_off, d, (int64_t)(runs[r].socket_id + rs[r].n_msgs), resp + rb, resp_cap - rb, &rl) != 0) return -1;
                d->resp_off = (uint32_t)rb; d->resp_len = (uint32_t)rl;
            } else if (index == B2_PROTOCOL_BAIDU_STD && client) {
                if (process_rpc_response(bytes + d->frame_off, d, resp + rb, resp_cap - rb, &rl) != 0) return -1;
                if (d->status == B2_MSG_RESPONSE_UNZ) d->resp_off += (uint32_t)rb;       /* message inside the decompressed bytes */
            } else if (index == B2_PROTOCOL_BAIDU_STD) {
                if (process_rpc_request(cfg, bytes + d->frame_off, d, resp + rb, resp_cap - rb, &rl) != 0) return -1;
                d->resp_off = (uint32_t)rb; d->resp_len = (uint32_t)rl;
            } else if (index == B2_PROTOCOL_STREAMING_RPC) {
                process_stream_frame(cfg, bytes + d->frame_off, d, resp + rb, resp_cap - rb, &rl);
                d->resp_off = (uint32_t)rb; d->resp_len = (uint32_t)rl;
            } else {
                /* hulu_pbrpc / sofa_pbrpc / nshead: the path frames them; ProcessHuluRequest & co. stay on the host */
                d->status = B2_MSG_FRAMED; d->method_idx = -1;
            }
            rb += rl; nm++; rs[r].n_msgs++;
        }
        rs[r].consumed = pos; rs[r].preferred_proto = preferred;
        rs[r].resp_bytes = (uint32_t)rb - rs[r].resp_off;
    }
    *n_msgs = nm; *resp_bytes = (uint32_t)rb;
    return 0;
}

/* index of the method FindMethodPropertyByFullName(service, method) resolves, -1 if none (used by the h2 oracle) */
int orc_find_method_idx(const orc_config* cfg, const uint8_t* svc, uint32_t svc_len, const uint8_t* mth, uint32_t mth_len) {
    int idx = -1, no_service = 0;
    find_method(cfg, svc, svc_len, mth, mth_len, &idx, &no_service);
    return idx;
}
