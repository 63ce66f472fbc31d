// GpuH2Messenger with gzip-compressed gRPC calls (needs a GPU): echo calls are inflated on the device and answered from the
// inflated message, a compressed call to a method the device does not serve reaches the host callback with the inflated message,
// and every byte written back equals the oracle's (orc_h2_consume -> orc_h2_decompress -> orc_h2_pack_response), same chunking.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>
#include <string>
#include <vector>
#include "../../brpc_b200/host/h2_messenger.h"
#include "../../oracle/b2_oracle_h2_gzip.h"

#define CHECK(c) do { if (!(c)) { fprintf(stderr, "CHECK failed %s:%d: %s\n", __FILE__, __LINE__, #c); exit(1); } } while (0)

static std::string h2_frame(int type, int flags, uint32_t sid, const std::string& payload) {
    std::string f; const uint32_t n = (uint32_t)payload.size();
    f.push_back((char)(n >> 16)); f.push_back((char)(n >> 8)); f.push_back((char)n); f.push_back((char)type); f.push_back((char)flags);
    f.push_back((char)(sid >> 24)); f.push_back((char)(sid >> 16)); f.push_back((char)(sid >> 8)); f.push_back((char)sid);
    return f + payload;
}
static std::string hp_lit(const std::string& n, const std::string& v) {      // literal header field without indexing, new name (RFC 7541 6.2.2)
    std::string o; o.push_back(0); o.push_back((char)n.size()); o += n; o.push_back((char)v.size()); o += v; return o;
}
static std::string gzip_of(const std::string& s) {
    z_stream z; memset(&z, 0, sizeof z);
    CHECK(deflateInit2(&z, 6, Z_DEFLATED, 15 | 16, 8, Z_DEFAULT_STRATEGY) == Z_OK);
    std::string out(deflateBound(&z, s.size()) + 32, '\0');
    z.next_in = (Bytef*)s.data(); z.avail_in = (uInt)s.size(); z.next_out = (Bytef*)&out[0]; z.avail_out = (uInt)out.size();
    CHECK(deflate(&z, Z_FINISH) == Z_STREAM_END);
    out.resize(z.total_out); deflateEnd(&z);
    return out;
}
static std::string plain(int c, int k) {                 // compressible text, a few sizes
    std::string s;
    const size_t n = 20 + 311 * k + (k == 7 ? 30000 : 0);
    while (s.size() < n) s += "conn " + std::to_string(c) + " call " + std::to_string(k) + " gzip echo payload; ";
    s.resize(n);
    return s;
}

static int g_host = 0;
static std::vector<std::string> g_expect_host;
static void HostProcess(b2::InputMessageBase* base) {
    b2::H2Message* m = static_cast<b2::H2Message*>(base);
    CHECK(m->unz_status == B2_H2_UNZ_OK);
    CHECK(m->body.length() > 5 && m->message.to_string() == g_expect_host[g_host]);
    g_host++;
    delete m;
}

int main() {
    b2_options opt; memset(&opt, 0, sizeof opt);
    opt.device = 0; opt.max_batch_bytes = 8 << 20; opt.max_msgs = 1 << 14; opt.max_runs = 64; opt.max_resp_bytes = 32 << 20;
    b2::GpuH2Messenger messenger(opt);
    b2_method echo = { "example.EchoService", "EchoService", "Echo", "example.EchoRequest", B2_HANDLER_ECHO, 1, 0, 0 };
    CHECK(messenger.AddMethod(echo) == 0);
    messenger.SetHostProcess(HostProcess);
    const int kConns = 5, kCalls = 10;
    std::vector<std::string> streams(kConns);
    for (int c = 0; c < kConns; c++) {
        std::string& st = streams[c];
        st = "PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n"; st += h2_frame(4, 0, 0, "");
        for (int k = 0; k < kCalls; k++) {
            const uint32_t sid = 1 + 2 * k;
            const bool other = c == 1 && k % 3 == 1;                                     // compressed, but no device-served method
            const bool compressed = (c + k) % 4 != 3;                                    // the rest travel uncompressed on the same connections
            std::string hb = hp_lit(":method", "POST") + hp_lit(":scheme", "http") + hp_lit(":path", other ? "/example.Other/Call" : "/example.EchoService/Echo") +
                             hp_lit("content-type", "application/grpc") + hp_lit("te", "trailers") + hp_lit("grpc-encoding", "gzip");
            const std::string msg = plain(c, k);
            if (other) g_expect_host.push_back(msg);
            const std::string wire = compressed ? gzip_of(msg) : msg;
            std::string body; body.push_back(compressed ? 1 : 0);
            body.push_back((char)(wire.size() >> 24)); body.push_back((char)(wire.size() >> 16)); body.push_back((char)(wire.size() >> 8)); body.push_back((char)wire.size());
            body += wire;
            st += h2_frame(1, 0x4, sid, hb);
            const size_t step = k % 3 == 2 ? 9 : 16000;                                  // several DATA frames: the body is assembled in the slot
            for (size_t at = 0; at < body.size(); at += step) st += h2_frame(0, at + step >= body.size() ? 0x1 : 0, sid, body.substr(at, step));
        }
    }
    std::vector<b2::Socket*> socks; std::vector<size_t> pos(kConns, 0);
    std::vector<orc_h2_conn*> oc(kConns); std::vector<std::string> obuf(kConns), expect(kConns);
    for (int c = 0; c < kConns; c++) { socks.push_back(messenger.AddConnection(700 + c)); oc[c] = orc_h2_conn_new(); }
    orc_config cfg; memset(&cfg, 0, sizeof cfg); b2_method ms[1] = { echo }; cfg.methods = ms; cfg.n_methods = 1;
    unsigned seed = 4242; int rounds = 0, total = 0, n_unz = 0;
    std::vector<b2_h2_msg> om(256); std::vector<b2_h2_unz_result> ores(256);
    std::vector<uint8_t> octrl(1 << 16), oblob(1 << 21), opack(1 << 18), ounz(4 << 20);
    for (bool more = true; more; rounds++) {
        more = false;
        for (int c = 0; c < kConns; c++) {
            seed = seed * 1103515245u + 12345u;
            const size_t n = std::min(streams[c].size() - pos[c], (size_t)(seed >> 16) % 6000);
            socks[c]->_read_buf.append(streams[c].data() + pos[c], n); obuf[c].append(streams[c].data() + pos[c], n); pos[c] += n;
            if (pos[c] < streams[c].size()) more = true;
        }
        const int n = messenger.ProcessNewMessages(socks);
        CHECK(n >= 0); total += n;
        for (int c = 0; c < kConns; c++) {                       // the same round through the oracle
            if (obuf[c].empty()) continue;
            uint32_t cons = 0, nm = 0, cl = 0, bl = 0, mfs = 0, sws = 0;
            const uint32_t err = orc_h2_consume(oc[c], &cfg, (const uint8_t*)obuf[c].data(), (uint32_t)obuf[c].size(), &cons, om.data(), 256, &nm,
                                                octrl.data(), (uint32_t)octrl.size(), &cl, oblob.data(), (uint32_t)oblob.size(), &bl, &mfs, &sws);
            CHECK(err == B2_PARSE_ERROR_NOT_ENOUGH_DATA);
            CHECK(orc_h2_decompress(om.data(), nm, nullptr, oblob.data(), ounz.data(), (uint32_t)ounz.size(), ores.data()) == 0);
            expect[c].append((const char*)octrl.data(), cl);
            for (uint32_t k = 0; k < nm; k++) {
                const bool compressed = om[k].flags & B2_H2_FLAG_GRPC_COMPRESSED;
                CHECK(ores[k].status == (compressed ? B2_H2_UNZ_OK : B2_H2_UNZ_NONE));
                if (om[k].method_idx != 0) continue;            // the host callback's business
                const std::string ct = "application/grpc";
                const std::string m = compressed ? std::string((const char*)ounz.data() + ores[k].out_off, ores[k].out_len)
                                                 : std::string((const char*)oblob.data() + om[k].msg_off, om[k].msg_len);
                n_unz += compressed;
                const std::string blob = ct + m;
                b2_h2_response r; memset(&r, 0, sizeof r);
                r.stream_id = om[k].stream_id; r.status_code = 200; r.flags = B2_H2_RESP_GRPC; r.content_type_len = (uint32_t)ct.size();
                r.body_off = (uint32_t)ct.size(); r.body_len = (uint32_t)m.size();
                const uint32_t pn = orc_h2_pack_response(oc[c], &r, (const uint8_t*)blob.data(), opack.data());
                expect[c].append((const char*)opack.data(), pn);
            }
            obuf[c].erase(0, cons);
        }
    }
    for (int c = 0; c < kConns; c++) {
        CHECK(!socks[c]->Failed() && socks[c]->_read_buf.length() == obuf[c].size());
        CHECK(socks[c]->_write_buf.to_string() == expect[c]);
        orc_h2_conn_free(oc[c]);
    }
    CHECK(total == kConns * kCalls && g_host == (int)g_expect_host.size() && g_host > 0 && n_unz > 20);
    printf("h2 gzip messenger ok: %d calls in %d rounds, %d inflated echo calls, %d inflated host calls, every written byte identical to the oracle\n",
           total, rounds, n_unz, g_host);
    return 0;
}
