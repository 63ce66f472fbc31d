/* b2_oracle_h2_gzip.h — CPU ORACLE (test infrastructure) of b2_h2_decompress_requests (oracle/b2_oracle_h2_gzip.c). */
#ifndef B2_ORACLE_H2_GZIP_H_
#define B2_ORACLE_H2_GZIP_H_
#include "b2_oracle.h"
#ifdef __cplusplus
extern "C" {
#endif
/* The GzipDecompress step of ProcessHttpRequest (policy/http_rpc_protocol.cpp:1646-1683) for messages of orc_h2_consume (header
 * records and bodies in `blob`; a body with B2_H2_FLAG_BODY_IN_INPUT, as the device reports it, in `in`): what b2_h2_decompress_requests
 * returns, res and the bytes of out up to the end of the last inflated message.  0, or -1 when out of memory. */
int orc_h2_decompress(const b2_h2_msg* msgs, uint32_t n, const uint8_t* in, const uint8_t* blob, uint8_t* out, uint32_t out_cap,
                      b2_h2_unz_result* res);
#ifdef __cplusplus
}
#endif
#endif
