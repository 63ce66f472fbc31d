/* b2_oracle_h2_gzip.c — CPU ORACLE (test infrastructure): the GzipDecompress step of ProcessHttpRequest
 * (src/brpc/policy/http_rpc_protocol.cpp:1646-1683) for the messages orc_h2_consume produces, on top of the gzip restatement of
 * b2_oracle_gzip.c (orc_gzip_input_stream, orc_gzip_sizing_bound).  Built as oracle/liboracle_h2gzip.so, linked against liboracle.so. */
#include "b2_oracle_h2_gzip.h"
#include <stdlib.h>
#include <string.h>

static int ci_eq(const uint8_t* a, uint32_t n, const char* lit) {       /* lit in upper case */
    const size_t l = strlen(lit); if (l != n) return 0;
    for (size_t i = 0; i < l; i++) { uint8_t x = a[i]; if (x >= 'a' && x <= 'z') x = (uint8_t)(x - 32); if (x != (uint8_t)lit[i]) return 0; }
    return 1;
}
/* req_header.GetHeader(name) after H2StreamContext::ConsumeHeaders passed every field through HttpHeader::AppendHeader
 * (http_header.cpp:100-116): names compare case-insensitively over their whole length (CaseIgnoredEqual), a repeated field is
 * folded with "," onto a non-empty value and overwrites an empty one.  *present = 0: GetHeader returns NULL.  The value is malloc'ed. */
static uint8_t* get_header(const uint8_t* hdr, uint32_t len, const char* name, int* present, uint32_t* vlen) {
    uint8_t* v = NULL; uint32_t n = 0;
    *present = 0;
    for (uint32_t q = 0; q + 4 <= len;) {
        const uint32_t nl = hdr[q] | ((uint32_t)hdr[q + 1] << 8), vl = hdr[q + 2] | ((uint32_t)hdr[q + 3] << 8);
        if (q + 4 + nl + vl > len) break;
        if (ci_eq(hdr + q + 4, nl, name)) {
            const uint8_t* val = hdr + q + 4 + nl;
            *present = 1;
            if (n == 0) { v = (uint8_t*)realloc(v, vl + 1); memcpy(v, val, vl); n = vl; }
            else { v = (uint8_t*)realloc(v, n + 1 + vl + 1); v[n] = ','; memcpy(v + n + 1, val, vl); n += 1 + vl; }
        }
        q += 4 + nl + vl;
    }
    *vlen = n;
    return v;
}

/* policy::GzipDecompress(const IOBuf&, IOBuf*) = GzipDecompressBase (gzip_compress.cpp:138-176): it copies out whatever
 * GzipInputStream::Next hands over, then fails when the sub-stream was not read to its end (wrapper.ByteCount() != data.size())
 * or when one more Next() succeeds.  With the body in ONE block the sub-stream's only Next() is taken by the first Inflate()
 * (an empty body has nothing to take), and every way GzipInputStream's Next() returns false leaves it returning false from then
 * on (a zlib error stays in zerror_, an exhausted sub-stream leaves next_out NULL): it never fails.  tests/_gzipstream.py pins this
 * against the system zlib. */
static int gzip_decompress_base(const uint8_t* in, uint32_t n, uint8_t** out, size_t* out_len) {
    if (orc_gzip_input_stream(in, n, B2_COMPRESS_TYPE_GZIP, out, out_len) != 0) return -1;
    return 1;
}

int orc_h2_decompress(const b2_h2_msg* msgs, uint32_t n, const uint8_t* in, const uint8_t* blob, uint8_t* out, uint32_t out_cap,
                      b2_h2_unz_result* res) {
    uint64_t off = 0;
    for (uint32_t i = 0; i < n; i++) {
        const b2_h2_msg* m = &msgs[i];
        b2_h2_unz_result* r = &res[i];
        memset(r, 0, sizeof *r);
        if (m->body_len == 0) { r->status = B2_H2_UNZ_NONE; continue; }          /* req_body.empty(): nothing is decompressed */
        const int grpc = (m->flags & B2_H2_FLAG_GRPC) != 0;
        int present = 0; uint32_t vl = 0; uint8_t* v = NULL;
        if (grpc) {
            if (!(m->flags & B2_H2_FLAG_GRPC_PREFIX_OK)) { r->status = B2_H2_UNZ_NONE; continue; }   /* "Invalid gRPC request" comes first */
            if (!(m->flags & B2_H2_FLAG_GRPC_COMPRESSED)) { r->status = B2_H2_UNZ_NONE; continue; }
            v = get_header(blob + m->headers_off, m->headers_len, "GRPC-ENCODING", &present, &vl);
            if (!present) { r->status = B2_H2_UNZ_NO_ENCODING; free(v); continue; }
        } else {
            v = get_header(blob + m->headers_off, m->headers_len, "CONTENT-ENCODING", &present, &vl);
            if (!present) { r->status = B2_H2_UNZ_NONE; free(v); continue; }
        }
        const int gzip = vl == 4 && memcmp(v, "gzip", 4) == 0;                     /* *encoding == common->GZIP */
        free(v);
        if (!gzip) { r->status = B2_H2_UNZ_NOT_GZIP; continue; }
        const uint8_t* src = ((m->flags & B2_H2_FLAG_BODY_IN_INPUT) ? in : blob) + (grpc ? m->msg_off : m->body_off);
        const uint32_t len = grpc ? m->msg_len : m->body_len;
        /* the device's limits and slot placement: bound = its sizing pass, slots back to back in message order */
        if (len > ORC_GZ_MAX_IN) { r->status = B2_H2_UNZ_HOST; continue; }
        const size_t bound = orc_gzip_sizing_bound(src, len, B2_COMPRESS_TYPE_GZIP, ORC_GZ_MAX_OUT);
        if (bound > ORC_GZ_MAX_OUT) { r->status = B2_H2_UNZ_HOST; continue; }
        if (off + bound > out_cap) { r->status = B2_H2_UNZ_NO_ROOM; off += bound; continue; }
        uint8_t* got = NULL; size_t got_len = 0;
        const int ok = gzip_decompress_base(src, len, &got, &got_len);
        if (ok < 0) return -1;
        if (got_len > bound) { free(got); return -1; }                            /* the sizing pass must bound the bytes */
        r->out_off = (uint32_t)off;
        if (ok) { r->status = B2_H2_UNZ_OK; r->out_len = (uint32_t)got_len; memcpy(out + off, got, got_len); }
        else r->status = B2_H2_UNZ_FAILED;
        memset(out + off + (ok ? got_len : 0), 0, bound - (ok ? got_len : 0));
        free(got);
        off += bound;
    }
    return 0;
}
