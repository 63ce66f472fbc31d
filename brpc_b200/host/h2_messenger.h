// b2::GpuH2Messenger — C++ host side of the h2/gRPC path, the counterpart of GpuInputMessenger for sockets whose protocol is
// h2 (ParseH2Message, src/brpc/policy/http2_rpc_protocol.cpp:1103-1138).  One ProcessNewMessages() round hands every readable
// connection's buffer to b2_h2_process_batch, pops what the parser consumed, writes the bytes the reference would WriteAck,
// answers gRPC calls of device-served (echo) methods through b2_h2_pack_responses without the payload ever leaving the GPU,
// and gives every other completed request to the host callback the way ProcessHttpRequest would receive an H2StreamContext.
// gzip-compressed calls are inflated on the device first (b2_h2_decompress_requests, ProcessHttpRequest's GzipDecompress step):
// an echo call is answered from the inflated message, uncompressed, and the host callback gets the inflated message too.
#pragma once
#include <algorithm>
#include <utility>
#include "input_messenger.h"

namespace b2 {

struct H2Message : public InputMessageBase {           // an H2StreamContext after OnEndStream
    int stream_id = 0;
    std::vector<std::pair<std::string, std::string>> headers;   // every decoded field, in order
    IOBuf body;                                         // the raw DATA payloads (compressed, for a compressed call)
    IOBuf message;                                      // the inflated request when unz_status == B2_H2_UNZ_OK, else empty
    uint32_t unz_status = B2_H2_UNZ_NONE;               // b2_h2_decompress_requests' verdict (B2_H2_UNZ_*)
    b2_h2_msg desc;
};

class GpuH2Messenger {
public:
    typedef void (*Process)(InputMessageBase* msg);
    // max_conns / max_pending / stream_bytes: the device's h2 stream pool (b2_h2_configure); a gRPC client keeps up to 100 calls in flight
    explicit GpuH2Messenger(const b2_options& opt, uint32_t out_cap = 32u << 20, uint32_t max_conns = B2_H2_MAX_CONNS, uint32_t max_pending = B2_H2_MAX_PENDING,
                            uint32_t stream_bytes = B2_H2_STREAM_BYTES) : _cap(opt.max_batch_bytes), _out_cap(out_cap), _max_conns(max_conns), _msg_cap(opt.max_msgs) {
        if (b2_ctx_create(&opt, &_ctx) != B2_OK) throw std::runtime_error(std::string("b2_ctx_create: ") + b2_last_error());
        _batch = static_cast<uint8_t*>(b2_block_alloc(_cap)); _out = static_cast<uint8_t*>(b2_block_alloc(_out_cap));
        _pack = static_cast<uint8_t*>(b2_block_alloc(_out_cap));
        const uint64_t resp_bytes = opt.max_resp_bytes ? opt.max_resp_bytes : (uint64_t)opt.max_batch_bytes + (uint64_t)opt.max_msgs * 64 + (1u << 20);   // (b2_ctx_create's default)
        _unz_cap = (uint32_t)std::min<uint64_t>(_out_cap, resp_bytes);
        _unz = static_cast<uint8_t*>(b2_block_alloc(_unz_cap));
        if (!_batch || !_out || !_pack || !_unz || b2_h2_configure(_ctx, max_conns, max_pending, stream_bytes) != B2_OK) {
            b2_block_free(_batch); b2_block_free(_out); b2_block_free(_pack); b2_block_free(_unz); b2_ctx_destroy(_ctx);      // (nothing leaks when construction fails)
            throw std::runtime_error(std::string("GpuH2Messenger: ") + b2_last_error());
        }
        for (uint32_t k = max_conns; k-- > 0;) _free_conns.push_back(k);
    }
    ~GpuH2Messenger() { b2_block_free(_batch); b2_block_free(_out); b2_block_free(_pack); b2_block_free(_unz); b2_ctx_destroy(_ctx); }
    GpuH2Messenger(const GpuH2Messenger&) = delete;

    int AddMethod(const b2_method& m) { const int i = b2_register_method(_ctx, &m); if (i >= 0) { _handlers.resize(i + 1); _handlers[i] = m.handler; } return i; }
    void SetHostProcess(Process p) { _process = p; }
    // a new server-side connection: H2Context is created when the first bytes arrive (:1108-1120)
    // Device connection slots are a free list: RemoveConnection gives the slot back.  nullptr = no slot left (the caller keeps such a
    // connection on the host parser) or the device refused the reset.
    Socket* AddConnection(uint64_t id) {
        auto it = _sockets.find(id);
        if (it != _sockets.end()) return it->second.get();
        if (_free_conns.empty()) return nullptr;
        const uint32_t slot = _free_conns.back();
        if (b2_h2_conn_reset(_ctx, slot) != B2_OK) return nullptr;
        _free_conns.pop_back();
        _conn_of[id] = slot;
        return (_sockets[id] = std::unique_ptr<Socket>(new Socket(id))).get();
    }
    void RemoveConnection(uint64_t id) {
        auto it = _conn_of.find(id);
        if (it == _conn_of.end()) return;
        _free_conns.push_back(it->second); _conn_of.erase(it); _sockets.erase(id);
    }

    // One round over the readable connections.  Returns the number of completed requests, -1 on an ABI error.
    int ProcessNewMessages(const std::vector<Socket*>& readable) {
        std::vector<b2_run> runs; std::vector<Socket*> live;
        size_t total = 0;
        for (Socket* s : readable) {
            if (s->Failed() || s->_read_buf.empty()) continue;
            const size_t n = s->_read_buf.length();
            if (n + 16 > _cap) { s->SetFailed(22, "Close socket: pending h2 bytes exceed the batch capacity"); continue; }
            if (total + n + 16 > _cap) continue;                  // served next round; later (smaller) connections still fit
            s->_read_buf.copy_to(_batch + total, n, 0);
            b2_run r; r.socket_id = _conn_of[s->id()]; r.offset = (uint32_t)total; r.length = (uint32_t)n; r.preferred_proto = -1; r.flags = 0;
            runs.push_back(r); live.push_back(s);
            total = (total + n + 15) & ~(size_t)15;
        }
        if (runs.empty()) return 0;
        // (the ABI splits msg_cap evenly over the runs: give every connection what a full batch of minimal requests could complete)
        const size_t per_run = std::max<size_t>(64, std::min<size_t>(_msg_cap / runs.size(), 4096));
        std::vector<b2_h2_run_status> rs(runs.size()); std::vector<b2_h2_msg> msgs(per_run * runs.size()); uint32_t n_msgs = 0;
        if (b2_h2_process_batch(_ctx, _batch, (uint32_t)total, runs.data(), (uint32_t)runs.size(), rs.data(), msgs.data(), (uint32_t)msgs.size(),
                                &n_msgs, _out, _out_cap) != B2_OK) return -1;
        // ProcessHttpRequest's GzipDecompress step for the round's candidates: compressed gRPC messages, and bodies of other requests
        std::vector<b2_h2_msg> cand; std::vector<uint32_t> cand_of(n_msgs, UINT32_MAX);
        for (uint32_t m = 0; m < n_msgs; m++) {
            const b2_h2_msg& d = msgs[m];
            const bool grpc = d.flags & B2_H2_FLAG_GRPC;
            if (grpc ? (d.flags & B2_H2_FLAG_GRPC_PREFIX_OK) && (d.flags & B2_H2_FLAG_GRPC_COMPRESSED) : d.body_len != 0) { cand_of[m] = (uint32_t)cand.size(); cand.push_back(d); }
        }
        std::vector<b2_h2_unz_result> unz(cand.size());
        if (!cand.empty() && b2_h2_decompress_requests(_ctx, cand.data(), (uint32_t)cand.size(), _unz, _unz_cap, unz.data()) != B2_OK) return -1;
        std::vector<b2_h2_response> resps; std::vector<Socket*> resp_sock;
        for (size_t i = 0; i < runs.size(); i++) {
            Socket* s = live[i]; const b2_h2_run_status& st = rs[i];
            s->AddInputBytes(st.consumed); s->AddInputMessages(st.n_msgs);
            if (st.ctrl_len) { IOBuf ack; ack.append(_out + st.ctrl_off, st.ctrl_len); s->Write(&ack); }      // WriteAck (:144-150)
            for (uint32_t m = st.first_msg; m < st.first_msg + st.n_msgs; m++) {
                const b2_h2_msg& d = msgs[m];
                const b2_h2_unz_result* u = cand_of[m] != UINT32_MAX ? &unz[cand_of[m]] : nullptr;
                const bool inflated = u && u->status == B2_H2_UNZ_OK;
                const bool device_echo = (d.flags & B2_H2_FLAG_GRPC) && (d.flags & B2_H2_FLAG_GRPC_PREFIX_OK) && (!(d.flags & B2_H2_FLAG_GRPC_COMPRESSED) || inflated) &&
                                         d.method_idx >= 0 && d.method_idx < (int)_handlers.size() && _handlers[d.method_idx] == B2_HANDLER_ECHO;
                uint32_t ct_off = 0, ct_len = 0;
                if (device_echo) FindHeader(d, "content-type", &ct_off, &ct_len);
                if (device_echo && ct_len) {
                    // SendHttpResponse for gRPC: status 200, the request's content-type, the echoed message, grpc-status 0
                    b2_h2_response r; memset(&r, 0, sizeof r);
                    r.conn = (uint32_t)runs[i].socket_id; r.stream_id = d.stream_id; r.status_code = 200;
                    r.flags = B2_H2_RESP_GRPC | B2_H2_RESP_CT_IN_OUT | (inflated ? B2_H2_RESP_BODY_IN_UNZ : (d.flags & B2_H2_FLAG_BODY_IN_INPUT) ? B2_H2_RESP_BODY_IN_INPUT : B2_H2_RESP_BODY_IN_OUT);
                    r.content_type_off = ct_off; r.content_type_len = ct_len;
                    r.body_off = inflated ? u->out_off : d.msg_off; r.body_len = inflated ? u->out_len : d.msg_len;
                    resps.push_back(r); resp_sock.push_back(s);
                } else if (_process) {
                    H2Message* msg = new H2Message; msg->socket = s; msg->stream_id = (int)d.stream_id; msg->desc = d;
                    for (uint32_t q = 0; q < d.headers_len;) {
                        const uint8_t* p = _out + d.headers_off + q; const uint32_t nl = p[0] | (p[1] << 8), vl = p[2] | (p[3] << 8);
                        msg->headers.emplace_back(std::string((const char*)p + 4, nl), std::string((const char*)p + 4 + nl, vl)); q += 4 + nl + vl;
                    }
                    const uint8_t* body = (d.flags & B2_H2_FLAG_BODY_IN_INPUT) ? _batch + d.body_off : _out + d.body_off;
                    msg->body.append(body, d.body_len);
                    if (u) { msg->unz_status = u->status; if (inflated) msg->message.append(_unz + u->out_off, u->out_len); }
                    _process(msg);
                }
            }
            s->_read_buf.pop_front(st.consumed);
            if (st.parse_error != B2_PARSE_ERROR_NOT_ENOUGH_DATA)
                s->SetFailed(22 /*EINVAL*/, std::string("Close socket: ") + ParseErrorToString((ParseError)st.parse_error));
        }
        if (!resps.empty()) {
            // responses of one connection must be adjacent: they already are (runs are visited in order)
            std::vector<uint32_t> offs(resps.size()), lens(resps.size());
            if (b2_h2_pack_responses(_ctx, nullptr, 0, resps.data(), (uint32_t)resps.size(), _pack, _out_cap, offs.data(), lens.data()) != B2_OK) return -1;
            for (size_t k = 0; k < resps.size(); k++) { IOBuf out; out.append(_pack + offs[k], lens[k]); resp_sock[k]->Write(&out); }
        }
        return (int)n_msgs;
    }
    b2_ctx* ctx() { return _ctx; }

private:
    void FindHeader(const b2_h2_msg& d, const char* name, uint32_t* off, uint32_t* len) const {   // last occurrence wins, like HttpHeader::set_content_type
        const size_t want = strlen(name);
        for (uint32_t q = 0; q < d.headers_len;) {
            const uint8_t* p = _out + d.headers_off + q; const uint32_t nl = p[0] | (p[1] << 8), vl = p[2] | (p[3] << 8);
            if (nl == want && memcmp(p + 4, name, want) == 0) { *off = d.headers_off + q + 4 + nl; *len = vl; }
            q += 4 + nl + vl;
        }
    }
    b2_ctx* _ctx = nullptr; uint8_t* _batch = nullptr; uint8_t* _out = nullptr; uint8_t* _pack = nullptr; uint8_t* _unz = nullptr; size_t _cap; uint32_t _out_cap, _unz_cap = 0, _max_conns; size_t _msg_cap;
    std::vector<uint32_t> _free_conns;
    Process _process = nullptr; std::vector<int> _handlers;
    std::unordered_map<uint64_t, std::unique_ptr<Socket>> _sockets;
    std::unordered_map<uint64_t, uint32_t> _conn_of;
};

}  // namespace b2
