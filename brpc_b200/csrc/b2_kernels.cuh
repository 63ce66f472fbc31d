// b2_kernels.cuh — the sm_100a kernels of the brpc message-processing hot path.
//
// Data layout in HBM (all offsets < 4 GiB, one batch):
//   bytes  : the batch buffer; run r occupies [runs[r].offset, +length), offset % 16 == 0
//   tiles  : every run is split in TILE-byte tiles; tile t of the batch = (run, k)
//   msgs   : b2_msg_desc[ ], 64 B each, per-run order, runs in order
//   resp   : response region; message i owns the 16-byte aligned slot
//            [slot_off[i], slot_off[i+1]) and its frame starts at slot_off[i] + pad
//            so that the echoed payload keeps its (mod 16) alignment -> 16 B copies
//
// Pipeline (one launch each, same stream):
//   k_tile_search  warp/tile   speculative first frame start of every tile (k >= 1)
//   k_tile_walk    thread/tile header chain inside the tile -> (exit, count)
//   k_resolve      CTA/run     verifies the speculation chain from tile 0 (exact),
//                              falls back to a scalar walk where it fails, run status
//   (run prefix)   first_msg of every run: the last CTA of k_resolve
//   k_frame_table  16 thr/tile copies the frame offsets k_tile_walk kept (re-walks only what k_resolve changed)
//   k_decode       thread/msg  RpcMeta / StreamFrameMeta / EchoRequest decode -> desc, aux, slot
//   k_scan_*       exclusive scan of the slot sizes
//   k_pack         warp/msg    response header+meta, payload copy (+CRC32C)
//   (finalize)     per-run response span + counters: prologue of k_pack_slow
#pragma once
#include <cuda_runtime.h>
#include "b2_core.cuh"
#include "b2_inflate.cuh"

namespace b2 {

enum TileKind : uint8_t { kRanOff = 0, kStop = 1, kAmbig = 2 };

struct __align__(16) TileRec {
    uint32_t entry;      // first step position (run-relative), kNone = no candidate
    uint32_t exit;       // position after the last step that started in this tile
    uint32_t count;      // messages cut by those steps
    uint8_t kind;        // TileKind
    int8_t last_proto;   // protocol of the last message (0 = none)
    uint8_t live;        // set by k_resolve: the true chain enters this tile at `entry`
    int8_t pf_in;        // set by k_resolve: preferred index at the first step
};

struct __align__(16) MsgAux {     // device-internal side record of k_decode -> k_pack
    uint32_t msg_off;    // echoed message: offset from the frame start
    uint32_t msg_len;
    uint32_t att_len;    // echoed attachment bytes (contiguous after body_wo_att)
    uint32_t att_off;    // offset from the frame start
    uint32_t cks_off;    // request checksum_value span (offset from frame start)
    uint32_t cks_len;
    uint32_t svc_off, svc_len;
    uint32_t mth_off, mth_len;
    uint32_t pad;        // bytes between slot start and frame start (0..15)
    uint32_t err_kind;   // ErrKind for B2_MSG_ERROR_REPLIED
};
// k_decode -> k_pack_tma: everything the bandwidth path needs for one OK echo reply
struct __align__(16) PackJob {
    uint32_t src_off;    // batch offset of the first payload byte that TMA moves (16-byte aligned)
    uint32_t bulk_len;   // payload bytes moved by TMA, rounded up to 16 (0 = payload fits in the head)
    uint16_t head_len;   // bytes of the head record: pad + prefix + payload bytes up to the 16-byte boundary
    uint8_t pad;         // slot start -> frame start
    uint8_t fast;        // 1 = take the TMA path
    uint32_t slot_len;   // roundup16(pad + resp_len)
};
constexpr uint32_t kHeadBytes = 96;               // head record stride; prefix <= 64 on the TMA path

enum ErrKind : uint32_t { kErrNone = 0, kErrAttachment, kErrNoService, kErrNoMethod, kErrParseRequest };

struct DevMethod {                // registered method table (global memory, tiny)
    char full_method[200];        // "example.EchoService.Echo"
    uint32_t full_method_len;
    char service_short[64];  uint32_t service_short_len;
    char service_full[120];  uint32_t service_full_len;
    char request_type[96];   uint32_t request_type_len;
    int32_t handler, echo_attachment, response_checksum_type, response_compress_type;
};
struct DevConfig {
    uint64_t max_body_size;
    uint32_t tile_bytes, tile_shift;
    uint32_t n_methods;
    uint32_t identity_len;
    uint32_t stream_handler;      // B2_STREAM_*
    uint32_t spec_k;              // speculative frame offsets kept per tile: kSpecK, or kSpecKDense when tiles hold many small frames
    uint32_t by_ref;              // B2_RESP_BY_REF: OK echo replies are {prefix, reference into the request bytes}
    uint32_t verify_done;         // k_crc_verify already checked the CRC-carrying echoes: k_pack_slow skips its own verify pass
    uint32_t proto_mask;          // handlers of the messenger (bit = ProtocolType): default baidu_std | streaming_rpc; b2_set_protocols adds hulu / sofa / nshead
    uint32_t fused;               // the fused decode+pack kernel serves this batch: replies sit at their request's own offset, slow ones in the overflow area
    uint32_t ovf_base;            // ... which starts here in the resp region
    uint32_t pull_vecs;           // 16-byte vectors per stashed row: 8 (128 B), or 6 (96 B) with B2_RESP_BY_REF — the decoder then needs header + meta + 6 body bytes only
    uint32_t pull;                // B2_INPUT_PULL: `bytes` is mapped host memory; the walk stashes each frame's first 128 bytes in HBM
    char identity[64];            // "ip:port" of Controller::AppendServerIdentiy
};

struct BatchPtrs {
    const uint8_t* bytes;
    const b2_run* runs;
    const uint32_t* run_tile_base;   // [n_runs+1] first tile of each run
    const uint4* tile_info;          // [n_tiles] {run offset, run length, tile index inside the run, run index | run flags << 24}: host-built with
                                     // the batch so that a tile thread needs ONE load, not a tile->run->runs[] chain, before it can touch the bytes
    TileRec* tiles;
    uint32_t* tile_base;             // [n_tiles] run-relative index of the tile's first message
    uint32_t* tile_scratch;          // [3 * n_tiles] k_resolve spill when a run's tiles exceed shared memory
    uint32_t* tile_spec;             // [kSpecK * n_tiles] frame offsets found by the speculative walk (first kSpecK of a tile)
    b2_run_status* run_status;
    uint32_t* frame_off;             // [max_msgs] frame offsets (batch-relative), bit 31 = protocol - 1
    uint32_t* frame_run;             // [max_msgs] run index of every message
    uint32_t* frame_row;             // [max_msgs] B2_INPUT_PULL: index of the frame's stashed row (kNone = read the bytes in place)
    uint4* rows;                     // [n_tiles * spec_k][8] B2_INPUT_PULL: the 128 bytes at (frame start & ~15), fetched ONCE over PCIe by the walk
    b2_msg_desc* msgs;
    MsgAux* aux;
    PackJob* jobs;                   // [max_msgs]
    uint4* refs;                     // [max_msgs] b2_resp_ref {prefix_len, src_off, src_len, 0} (B2_RESP_BY_REF)
    uint32_t* slow_idx;              // [max_msgs] messages k_pack_slow has to serve (unordered), count in totals[3]
    uint8_t* heads;                  // [max_msgs * kHeadBytes] reply prefixes pre-shifted to their slot alignment
    uint32_t* slot;                  // [max_msgs+1] slot sizes -> exclusive offsets
    uint32_t* scan_tmp;              // block sums
    uint8_t* resp;
    uint8_t* unz;                    // [2 * max_resp] scratch at the message's slot offset: decompressed request bodies (first half),
                                     // serialized replies awaiting compression (second half)
    uint16_t* snappy_tab;            // [kSnappyWarps][16384] hash tables of the snappy encoder, one per warp
    unsigned long long* counters;    // int64[B2_N_COUNTERS]
    uint32_t* totals;                // [0]=n_msgs [1]=resp_bytes [2]=overflow flags [3]=slow count [4],[5]=last-CTA tickets
                                     // [6]=slow queue ticket [7]=verify count [8]=verify queue ticket
    const DevMethod* methods;
    const uint32_t* crc_adv;         // warp CRC tables: hot [20][256] then tree [5][4][256]
    uint32_t n_runs, n_tiles, max_msgs, max_resp;
};

// ---------------------------------------------------------------------------
// tile walk: the CutInputMessage chain of the steps that START inside
// [entry, tile_end).  kSpec: the preferred index at the first step is unknown
// (speculation); a handler that pops bytes makes the outcome depend on it, so
// the tile is handed to the resolver (kAmbig).
template <bool kSpec, typename Emit>
B2_HD void walk_tile(const uint8_t* run, uint32_t len, uint32_t entry, int pf_in, uint32_t tile_end,
                     uint64_t max_body, bool client, TileRec& t, Emit emit, uint32_t mask = kProtoMaskDefault) {
    uint32_t pos = entry, count = 0;
    int pf = kSpec ? -1 : pf_in, last = 0;
    uint8_t kind = kRanOff;
    while (pos < tile_end) {
        const Step s = cut_input_message(run, len, pos, pf, max_body, client, mask);
        if (kSpec && count == 0 && (s.popped || (s.index != 12 && nshead_claims(run, len, pos, max_body, mask)))) { kind = kAmbig; break; }
        if (s.err != B2_PARSE_OK) { kind = kStop; break; }
        emit(count, s);
        count++; last = s.index; pf = s.index; pos = s.new_pos;
    }
    t.entry = entry; t.exit = pos; t.count = count; t.kind = kind; t.last_proto = (int8_t)last;
}
struct NoEmit { B2_HD void operator()(uint32_t, const Step&) const {} };
constexpr uint32_t kSpecK = 16;            // speculative frame offsets kept per tile; tiles with more frames are re-walked by k_frame_table
constexpr uint32_t kSpecKDense = 128;      // ... when the previous batches say a tile holds more than kSpecK frames (small requests)
constexpr uint8_t kKindRewalked = 0x80;    // k_resolve re-walked the tile: its speculative offsets are void
struct EmitSpec {
    uint32_t* out; uint32_t run_off, cap;
    __device__ __forceinline__ void operator()(uint32_t i, const Step& s) const {
        if (i < cap) out[i] = (run_off + s.frame_pos) | ((uint32_t)(s.index != 1) << 31);
    }
};

#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t find_run(const uint32_t* base, uint32_t n_runs, uint32_t tile) {
    uint32_t lo = 0, hi = n_runs;          // largest r with base[r] <= tile
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(base + mid) <= tile) lo = mid; else hi = mid; }
    return lo;
}
__device__ __forceinline__ bool is_magic(uint32_t w) { return w == kMagicPRPC || w == kMagicSTRM; }
#ifndef B2_SEARCH_FIRST
#define B2_SEARCH_FIRST 2
#endif

// --- k_tile_search: one warp per tile ---------------------------------------
// Finds the first position p in the tile where a frame of either protocol parses
// completely (header sane, whole body inside the run) and is followed by another
// magic or the run tail.  Pure speculation: k_resolve accepts it only if the true
// chain arrives exactly there.
__global__ void __launch_bounds__(256, 6) k_tile_search(BatchPtrs B, DevConfig C) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B.n_tiles) return;
    const uint4 ti = __ldg(B.tile_info + warp);
    const uint32_t k = ti.z;
    const uint8_t* base = B.bytes + ti.x;
    const uint32_t len = ti.y;
    uint32_t entry = kNone;
    if (k == 0) {
        entry = 0;
    } else {
        const uint32_t t0 = k << C.tile_shift;
        const uint32_t t1 = min(t0 + C.tile_bytes, len);
        // four 512-byte windows per trip: all eight loads of a lane are issued before the first use
        for (uint32_t c0 = t0; c0 < t1 && entry == kNone; c0 += (c0 == t0 ? 512u * B2_SEARCH_FIRST : 2048u)) {
            const int nwin = c0 == t0 ? B2_SEARCH_FIRST : 4;      // the first trip (B2_SEARCH_FIRST x 512 bytes) usually holds the entry; later trips go 4 wide
            uint4 v[4]; uint32_t nx[4];
            #pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t p0 = c0 + u * 512 + lane * 16;
                v[u] = make_uint4(0, 0, 0, 0); nx[u] = 0;
                if (u < nwin && p0 < t1) {
                    v[u] = __ldg(reinterpret_cast<const uint4*>(base + p0));        // bytes buffer is padded: safe past len
                    nx[u] = __ldg(reinterpret_cast<const uint32_t*>(base + p0 + 16));
                }
            }
            #pragma unroll
            for (int u = 0; u < 4; u++) {
                if (entry != kNone || u >= nwin) break;
                // lane owns 16 positions [p0, p0+16); needs 3 more bytes for the last windows
                const uint32_t w0 = c0 + u * 512, p0 = w0 + lane * 16;
                const uint32_t w[5] = { v[u].x, v[u].y, v[u].z, v[u].w, nx[u] };
                uint32_t mask = 0, mkind = 0;                        // mask: a magic starts at this position; mkind: 2 bits each — 0 PRPC/STRM, 1 HULU, 2 SOFA
                const bool ext = (C.proto_mask & ((1u << 3) | (1u << 4))) != 0;
                #pragma unroll
                for (int k4 = 0; k4 < 4; k4++) {
                    // byte prefilter: only positions holding 'P' or 'S' (first byte of "PRPC" / "STRM" / "SOFA"; 'H' for "HULU") are looked at
                    uint32_t e = __vcmpeq4(w[k4], 0x50505050u) | __vcmpeq4(w[k4], 0x53535353u);
                    if (ext) e |= __vcmpeq4(w[k4], 0x48484848u);
                    while (e) {
                        const int b = (__ffs(e) - 1) >> 3;
                        e &= ~(0xffu << (8 * b));
                        const int j = 4 * k4 + b;
                        const uint32_t word = __funnelshift_r(w[k4], w[k4 + 1], b * 8);
                        const bool other = ext && ((word == kMagicHULU && (C.proto_mask & 8u)) || (word == kMagicSOFA && (C.proto_mask & 16u)));
                        if ((is_magic(word) || other) && p0 + j + 4 <= len && p0 + j < t1) { mask |= 1u << j; if (other) mkind |= (word == kMagicHULU ? 1u : 2u) << (2 * j); }
                    }
                }
                // candidates in position order: lanes ascending, bits ascending.  A candidate is taken when its header is
                // sane (meta_size <= body_size <= max_body_size): the twelve header bytes are already in registers — the
                // lane's own 16 bytes plus its neighbour's — so no further load is needed; k_resolve is the exactness gate.
                uint32_t any = __ballot_sync(0xffffffffu, mask != 0);
                const uint32_t n5 = __shfl_down_sync(0xffffffffu, v[u].y, 1), n6 = __shfl_down_sync(0xffffffffu, v[u].z, 1);
                while (any && entry == kNone) {
                    const int src = __ffs(any) - 1;
                    uint32_t m = __shfl_sync(0xffffffffu, mask, src);
                    const uint32_t kinds = __shfl_sync(0xffffffffu, mkind, src);
                    while (m && entry == kNone) {
                        const int jj = __ffs(m) - 1;
                        const uint32_t p = w0 + src * 16 + jj;
                        m &= m - 1;
                        const uint32_t kind = (kinds >> (2 * jj)) & 3u;
                        if (kind == 2) { entry = p; break; }                 // "SOFA": taken on the magic alone (k_resolve is the exactness gate)
                        uint32_t body_le = 0, meta_le = 0;
                        if (src < 31) {
                            const uint32_t q = (uint32_t)(jj + 4) >> 2, sh = ((uint32_t)(jj + 4) & 3u) * 8u;   // body_size sits at byte jj + 4
                            const uint32_t a1 = w[1], a2 = w[2], a3 = w[3], a4 = w[4];
                            const uint32_t x0 = q == 1 ? a1 : q == 2 ? a2 : q == 3 ? a3 : a4;
                            const uint32_t x1 = q == 1 ? a2 : q == 2 ? a3 : q == 3 ? a4 : n5;
                            const uint32_t x2 = q == 1 ? a3 : q == 2 ? a4 : q == 3 ? n5 : n6;
                            body_le = __shfl_sync(0xffffffffu, __funnelshift_r(x0, x1, sh), src);
                            meta_le = __shfl_sync(0xffffffffu, __funnelshift_r(x1, x2, sh), src);
                        } else if (p + 12 <= len) {                      // (the header straddles two windows: read it)
                            body_le = load_le32(base + p + 4); meta_le = load_le32(base + p + 8);
                        } else continue;
                        const uint32_t body = kind == 1 ? body_le : __byte_perm(body_le, 0, 0x0123), meta = kind == 1 ? meta_le : __byte_perm(meta_le, 0, 0x0123);   // hulu: host order
                        if (meta <= body && (uint64_t)body <= C.max_body_size) entry = p;
                    }
                    any &= any - 1;
                }
            }
        }
    }
    if (lane == 0) B.tiles[warp].entry = entry;
}

// The speculative walk of k_tile_walk: same result as walk_tile<true>, but (1) a step whose twelve header bytes show a known
// magic and sane sizes is decided from registers (the generic CutInputMessage restatement is called for everything else:
// short tails, oversize bodies, meta > body, unknown bytes), and (2) while the header at `pos` is still on its way from
// DRAM the header at pos + (length of the previous frame) is requested too — requests of one connection tend to repeat
// their size, so the dependent chain "header -> next position -> header" often advances two frames per round trip.
struct HdrWords { uint32_t w0, w1, w2, w3; };
__device__ __forceinline__ HdrWords load_hdr_words(const uint8_t* p) {          // the 16 aligned-ish bytes around p (buffer is padded)
    const uint32_t* q = reinterpret_cast<const uint32_t*>((uintptr_t)p & ~(uintptr_t)3);
    HdrWords h; h.w0 = __ldg(q); h.w1 = __ldg(q + 1); h.w2 = __ldg(q + 2); h.w3 = __ldg(q + 3);
    return h;
}
template <typename Emit>
__device__ __forceinline__ void walk_tile_spec(const uint8_t* run, uint32_t len, uint32_t entry, uint32_t tile_end,
                                               uint64_t max_body, bool client, TileRec& t, Emit emit, uint32_t mask) {
    uint32_t pos = entry, count = 0, prev_len = 0, pre_pos = kNone;
    int pf = -1, last = 0;
    uint8_t kind = kRanOff;
    HdrWords pre; pre.w0 = pre.w1 = pre.w2 = pre.w3 = 0;
    while (pos < tile_end) {
        Step s;
        bool fast = false;
        if (len - pos >= 12) {
            const HdrWords h = pre_pos == pos ? pre : load_hdr_words(run + pos);
            const uint32_t guess = pos + prev_len;
            // (guess <= len - 12, written so that a guess past the run's end — the last tile's end lies beyond it — cannot wrap around)
            if (prev_len && guess < tile_end && (uint64_t)guess + 12 <= len) { pre = load_hdr_words(run + guess); pre_pos = guess; }   // in flight while h is used
            else pre_pos = kNone;
            const uint32_t sh = 8u * (pos & 3u);                      // run offsets are 16-byte aligned: alignment of run + pos is pos & 3
            const uint32_t h0 = sh ? __funnelshift_r(h.w0, h.w1, sh) : h.w0, h1 = sh ? __funnelshift_r(h.w1, h.w2, sh) : h.w1,
                           h2 = sh ? __funnelshift_r(h.w2, h.w3, sh) : h.w2;
            const int idx = h0 == kMagicPRPC ? 1 : h0 == kMagicSTRM ? 2 : 0;
            const uint32_t body = __byte_perm(h1, 0, 0x0123), meta = __byte_perm(h2, 0, 0x0123);
            // (a preferred nshead handler is asked first and may claim these bytes: pf == 12 goes the generic way)
            if (idx && ((mask >> idx) & 1u) && pf != 12 && (uint64_t)body <= max_body && (uint64_t)(len - pos) >= 12ull + body && meta <= body) {
                s.err = B2_PARSE_OK; s.index = idx; s.pf = idx; s.frame_pos = pos; s.new_pos = pos + 12 + body; s.body = body; s.meta = meta; s.popped = false;
                fast = true;
            }
        }
        if (!fast) s = cut_input_message(run, len, pos, pf, max_body, client, mask);
        if (count == 0 && (s.popped || (s.index != 12 && nshead_claims(run, len, pos, max_body, mask)))) { kind = kAmbig; break; }
        if (s.err != B2_PARSE_OK) { kind = kStop; break; }
        emit(count, s);
        count++; last = s.index; pf = s.index; prev_len = s.new_pos - pos; pos = s.new_pos;
    }
    t.entry = entry; t.exit = pos; t.count = count; t.kind = kind; t.last_proto = (int8_t)last;
}

// --- k_tile_walk: one thread per tile ---------------------------------------
__global__ void __launch_bounds__(128) k_tile_walk(BatchPtrs B, DevConfig C) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B.n_tiles) return;
    const uint4 ti = __ldg(B.tile_info + t);
    const uint32_t k = ti.z;
    b2_run run; run.offset = ti.x; run.length = ti.y; run.flags = ti.w >> 24;
    TileRec rec;
    rec.entry = B.tiles[t].entry; rec.exit = 0; rec.count = 0; rec.kind = kStop; rec.last_proto = 0; rec.live = 0; rec.pf_in = -1;
    if (rec.entry != kNone) {
        // the frame offsets met on the way are kept: if k_resolve accepts the tile as is, k_frame_table only has to copy them
        EmitSpec e; e.out = B.tile_spec + (size_t)t * C.spec_k; e.run_off = run.offset; e.cap = C.spec_k;
        walk_tile_spec(B.bytes + run.offset, run.length, rec.entry, (k + 1) << C.tile_shift, C.max_body_size, (run.flags & B2_RUN_CLIENT) != 0, rec, e, run_mask(C.proto_mask, run.flags));
    }
    B.tiles[t] = rec;
}

// --- k_tile_walk_pull: B2_INPUT_PULL, eight lanes per tile ----------------------------------------------
// The batch lives in mapped host memory: every load is a PCIe read (~2 us, <= 575 M requests/s, ~50 GB/s).  The walk
// is the only stage that HAS to touch each frame, so it fetches, per hop, the 128 bytes at (position & ~15) with ONE
// coalesced load of the tile's eight lanes, decides the step from the header inside them (same rules as
// walk_tile_spec) and stashes the row in HBM; k_decode then finds header, RpcMeta and the first body bytes of every
// message in that stash and never goes back over the link.  One ~128-byte read per message is all that crosses.
__global__ void __launch_bounds__(128) k_tile_walk_pull(BatchPtrs B, DevConfig C) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t t = g >> 3, sub = threadIdx.x & 7u, lane = threadIdx.x & 31u;
    if (t >= B.n_tiles) return;                                       // (whole groups of eight leave together)
    const uint32_t gmask = 0xffu << (lane & 24u), l0 = lane & 24u;
    const uint4 ti = __ldg(B.tile_info + t);
    const uint32_t k = ti.z, len = ti.y;
    const uint8_t* run = B.bytes + ti.x;
    const bool client = ((ti.w >> 24) & B2_RUN_CLIENT) != 0;
    const uint32_t pmask = run_mask(C.proto_mask, ti.w >> 24);
    const uint32_t tile_end = (k + 1) << C.tile_shift, cap = C.spec_k;
    uint32_t* spec = B.tile_spec + (size_t)t * cap;
    uint4* rows = B.rows + (size_t)t * cap * 8;
    TileRec rec;
    rec.entry = B.tiles[t].entry; rec.exit = 0; rec.count = 0; rec.kind = kStop; rec.last_proto = 0; rec.live = 0; rec.pf_in = -1;
    if (rec.entry != kNone) {
        uint32_t pos = rec.entry, count = 0; int pf = -1, last = 0; uint8_t kind = kRanOff;
        while (pos < tile_end) {
            bool fast = false; uint32_t new_pos = pos, frame_pos = pos; int idx = 0, err = B2_PARSE_OK; bool popped = false;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (len - pos >= 12) {
                if (sub < C.pull_vecs) v = __ldg(reinterpret_cast<const uint4*>(run + (pos & ~15u)) + sub);      // (the buffer has 1 KiB of slack past its end)
                // the 12 header bytes start at byte (pos & 15) of the row: words from lanes 0 and 1 of the group
                const uint32_t a0 = __shfl_sync(gmask, v.x, l0), a1 = __shfl_sync(gmask, v.y, l0), a2 = __shfl_sync(gmask, v.z, l0), a3 = __shfl_sync(gmask, v.w, l0);
                const uint32_t b0 = __shfl_sync(gmask, v.x, l0 + 1), b1 = __shfl_sync(gmask, v.y, l0 + 1), b2 = __shfl_sync(gmask, v.z, l0 + 1);
                const uint32_t q = (pos & 15u) >> 2, sh = 8u * (pos & 3u);
                const uint32_t w0 = q == 0 ? a0 : q == 1 ? a1 : q == 2 ? a2 : a3, w1 = q == 0 ? a1 : q == 1 ? a2 : q == 2 ? a3 : b0;
                const uint32_t w2 = q == 0 ? a2 : q == 1 ? a3 : q == 2 ? b0 : b1, w3 = q == 0 ? a3 : q == 1 ? b0 : q == 2 ? b1 : b2;
                const uint32_t h0 = sh ? __funnelshift_r(w0, w1, sh) : w0, h1 = sh ? __funnelshift_r(w1, w2, sh) : w1, h2 = sh ? __funnelshift_r(w2, w3, sh) : w2;
                idx = h0 == kMagicPRPC ? 1 : h0 == kMagicSTRM ? 2 : 0;
                const uint32_t body = __byte_perm(h1, 0, 0x0123), meta = __byte_perm(h2, 0, 0x0123);
                if (idx && ((pmask >> idx) & 1u) && pf != 12 && (uint64_t)body <= C.max_body_size && (uint64_t)(len - pos) >= 12ull + body && meta <= body) { fast = true; new_pos = pos + 12 + body; }
            }
            if (count == 0 && ((pmask >> 12) & 1u)) {          // unknown preferred index + an nshead handler that would claim the bytes: the resolver decides
                int amb = 0;
                if (sub == 0) amb = nshead_claims(run, len, pos, C.max_body_size, pmask) ? 1 : 0;
                if (__shfl_sync(gmask, amb, l0)) { kind = kAmbig; break; }
            }
            if (!fast) {                                              // short tails, oversize bodies, meta > body, unknown bytes: the generic restatement
                Step s; s.err = 0; s.index = 0; s.new_pos = 0; s.frame_pos = 0; s.popped = false;
                if (sub == 0) s = cut_input_message(run, len, pos, pf, C.max_body_size, client, pmask);
                err = __shfl_sync(gmask, s.err, l0); idx = __shfl_sync(gmask, s.index, l0); new_pos = __shfl_sync(gmask, s.new_pos, l0);
                frame_pos = __shfl_sync(gmask, s.frame_pos, l0); popped = __shfl_sync(gmask, (int)s.popped, l0) != 0;
                if (count == 0 && popped) { kind = kAmbig; break; }
                if (err != B2_PARSE_OK) { kind = kStop; break; }
                if (sub < C.pull_vecs) v = __ldg(reinterpret_cast<const uint4*>(run + (frame_pos & ~15u)) + sub);
            }
            if (count < cap) {
                if (sub == 0) spec[count] = (ti.x + frame_pos) | ((uint32_t)(idx != 1) << 31);
                if (sub < C.pull_vecs) rows[(size_t)count * 8 + sub] = v;
            }
            count++; last = idx; pf = idx; pos = new_pos;
        }
        rec.exit = pos; rec.count = count; rec.kind = kind; rec.last_proto = (int8_t)last;
    }
    if (sub == 0) B.tiles[t] = rec;
}

// --- run prefix: exclusive scan of n_msgs over runs, done by the LAST CTA of k_resolve to finish -------
__device__ __forceinline__ void run_prefix_body(const BatchPtrs& B, uint32_t* s_warp, uint32_t* s_carry) {
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) *s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < B.n_runs; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        uint32_t v = i < B.n_runs ? __ldcg(&B.run_status[i].n_msgs) : 0, x = v;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= (uint32_t)d) x += y; }
        if (lane == 31) s_warp[wid] = x;
        __syncthreads();
        uint32_t wbase = 0, wtot = 0;
        for (uint32_t w = 0; w < nw; w++) { const uint32_t t = s_warp[w]; if (w < wid) wbase += t; wtot += t; }
        const uint32_t carry = *s_carry;
        if (i < B.n_runs) B.run_status[i].first_msg = carry + wbase + x - v;
        __syncthreads();
        if (threadIdx.x == 0) *s_carry = carry + wtot;
        __syncthreads();
    }
    if (threadIdx.x == 0) { B.totals[0] = *s_carry; if (*s_carry > B.max_msgs) B.totals[2] |= 1u; }
}

// --- k_resolve: one CTA per run ---------------------------------------------
// Verifies the speculation chain from position 0 with the true preferred index.
// A tile's summary is used only when the chain arrives exactly at its speculated
// entry (by induction every used summary is what a sequential walk would have
// produced); otherwise the tile is re-walked here, scalar, from the true entry.
//   phase 1 (all threads): per tile, the link to the next tile on the chain
//   phase 2 (thread 0)   : hop along the links, one shared-memory load per hop;
//                          broken links / pf-sensitive tiles take the scalar path
//   phase 3 (all threads): message-index base and preferred index of every live tile
constexpr uint32_t kLinkOk = 0x80000000u;      // | next tile index
constexpr uint32_t kLinkStop = 0x40000000u;    // chain ends inside this tile (non-OK step)
constexpr uint32_t kLinkEnd = 0x20000000u;     // chain leaves the run's tiles (pos == len)
constexpr uint32_t kLinkBroken = 0x10000000u;  // | next tile index: its entry is not where we arrive
constexpr uint32_t kLinkRewalk = 0x08000000u;  // this tile itself must be re-walked (no entry / ambiguous)

__device__ __forceinline__ uint32_t make_link(const TileRec& t, const TileRec* tiles, uint32_t nt, uint32_t shift) {
    if (t.entry == kNone || t.kind == kAmbig) return kLinkRewalk;
    if (t.kind == kStop) return kLinkStop;
    const uint32_t j = t.exit >> shift;
    if (j >= nt) return kLinkEnd;
    return (tiles[j].entry == t.exit ? kLinkOk : kLinkBroken) | j;
}

__global__ void __launch_bounds__(256) k_resolve(BatchPtrs B, DevConfig C, uint32_t use_scratch) {
    extern __shared__ uint32_t sm[];
    const uint32_t r = blockIdx.x;
    const b2_run run = B.runs[r];
    const uint8_t* base = B.bytes + run.offset;
    const uint32_t len = run.length;
    const uint32_t tb = B.run_tile_base[r], nt = B.run_tile_base[r + 1] - tb;
    TileRec* tiles = B.tiles + tb;
    const bool fits = !use_scratch;                              // decided per LAUNCH by the host: no dynamic shared memory was allocated otherwise
    uint32_t* link = fits ? sm : B.tile_scratch + 3ull * tb;     // [nt]
    uint32_t* cp = link + nt;                                     // [nt] count << 2 | last_proto
    uint32_t* live = cp + nt;                                     // [nt]
    __shared__ uint32_t s_final_pos, s_warp_sum[8], s_warp_pf[8], s_carry_sum, s_carry_pf;
    // The speculation rests on the cut at a position not depending on the preferred index (only the ORDER of the handlers does, and the tiles
    // where bytes get popped on the way are re-walked).  On a CLIENT-side socket with more than baidu_std / streaming_rpc enabled that does
    // not hold: the channel's protocol is fixed, a frame of another handler is an error there (input_messenger.cpp:122-138), so what a
    // tile holds depends on the message before it.  Such runs take the exact chain: every tile re-walked in order with the true index.
    const uint32_t rmask = run_mask(C.proto_mask, run.flags);
    const bool pf_decides = (run.flags & B2_RUN_CLIENT) && !(rmask & kProtoMaskDump) && (rmask & ~((1u << B2_PROTOCOL_BAIDU_STD) | (1u << B2_PROTOCOL_STREAMING_RPC))) != 0;
    for (uint32_t k = threadIdx.x; k < nt; k += blockDim.x) {
        const TileRec t = tiles[k];
        link[k] = ((k == 0 && t.entry != 0) || pf_decides) ? kLinkRewalk : make_link(t, tiles, nt, C.tile_shift);
        cp[k] = (t.count << 4) | ((uint32_t)t.last_proto & 15u);     // (protocol indices go up to 12: nshead)
        live[k] = 0;
    }
    // dense shortcut: the leading stretch of tiles whose verified link goes to the next tile is
    // live without hopping (the common case: frames smaller than a tile, speculation all correct)
    __shared__ uint32_t s_first_bad;
    if (threadIdx.x == 0) s_first_bad = nt ? nt - 1 : 0;
    __syncthreads();
    {
        uint32_t mine = nt;
        for (uint32_t k = threadIdx.x; k + 1 < nt; k += blockDim.x)
            if (link[k] != (kLinkOk | (k + 1))) { mine = k; break; }
        if (mine < nt) atomicMin(&s_first_bad, mine);
    }
    __syncthreads();
    const uint32_t first_bad = s_first_bad;
    for (uint32_t k = threadIdx.x; k < first_bad; k += blockDim.x) live[k] = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t k = first_bad, pos = 0;
        bool via_ok = first_bad > 0;                 // arrived through a verified link: pos == tiles[k].entry
        while (k < nt) {
            uint32_t v = link[k];
            if (v & kLinkRewalk) {
                if (via_ok) pos = tiles[k].entry;
                // the true chain enters tile k at `pos` but the speculation has nothing usable there
                int pf = run.preferred_proto;
                for (uint32_t j = k; j-- > 0;) if (live[j] && (cp[j] >> 4)) { pf = (int)(cp[j] & 15u); break; }
                TileRec t; t.live = 0; t.pf_in = 0;
                walk_tile<false>(base, len, pos, pf, (k + 1) << C.tile_shift, C.max_body_size, (run.flags & B2_RUN_CLIENT) != 0, t, NoEmit(), run_mask(C.proto_mask, run.flags));
                tiles[k].entry = t.entry; tiles[k].exit = t.exit; tiles[k].count = t.count; tiles[k].kind = t.kind | kKindRewalked; tiles[k].last_proto = t.last_proto;
                cp[k] = (t.count << 4) | ((uint32_t)t.last_proto & 15u);
                v = make_link(t, tiles, nt, C.tile_shift);
                link[k] = v;
            }
            live[k] = 1;
            if (v & kLinkOk) { k = v & 0x07ffffffu; via_ok = true; continue; }
            if (v & kLinkBroken) {
                const uint32_t j = v & 0x07ffffffu;
                pos = tiles[k].exit; k = j; link[j] = kLinkRewalk; via_ok = false;
                continue;
            }
            pos = tiles[k].exit;                     // kLinkStop / kLinkEnd
            break;
        }
        // tiles reached through kLinkOk never set `pos`; recover it from the last live tile
        s_final_pos = pos;
        if (k < nt) s_final_pos = tiles[k].exit;
        if (nt == 0) s_final_pos = 0;
    }
    __syncthreads();
    // phase 3: exclusive sum of live counts; pf_in = protocol of the last message before the tile
    if (threadIdx.x == 0) { s_carry_sum = 0; s_carry_pf = 0; }
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t k0 = 0; k0 < nt; k0 += blockDim.x) {
        const uint32_t k = k0 + threadIdx.x;
        const uint32_t lv = k < nt ? live[k] : 0;
        const uint32_t c = lv ? (cp[k] >> 4) : 0;
        const uint32_t pr = (lv && c) ? (cp[k] & 15u) : 0;
        uint32_t x = c, y = pr;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t xs = __shfl_up_sync(0xffffffffu, x, d), ys = __shfl_up_sync(0xffffffffu, y, d);
            if (lane >= d) { x += xs; if (!y) y = ys; }
        }
        if (lane == 31) { s_warp_sum[wid] = x; s_warp_pf[wid] = y; }
        __syncthreads();
        uint32_t wsum = 0, wpf = 0;
        for (uint32_t w = 0; w < wid; w++) { wsum += s_warp_sum[w]; if (s_warp_pf[w]) wpf = s_warp_pf[w]; }
        const uint32_t carry_sum = s_carry_sum, carry_pf = s_carry_pf;
        // exclusive values for this tile
        const uint32_t incl_pf = y ? y : (wpf ? wpf : carry_pf);
        uint32_t excl_pf = __shfl_up_sync(0xffffffffu, incl_pf, 1);
        if (lane == 0) excl_pf = wpf ? wpf : carry_pf;
        if (k < nt && lv) {
            B.tile_base[tb + k] = carry_sum + wsum + x - c;
            tiles[k].live = 1;
            tiles[k].pf_in = (int8_t)(excl_pf ? (int)excl_pf : run.preferred_proto);
        }
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) { s_carry_sum = carry_sum + wsum + x; s_carry_pf = incl_pf; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const uint32_t pos = s_final_pos;
        const int pf_true = s_carry_pf ? (int)s_carry_pf : run.preferred_proto;
        // the step that ends ProcessNewMessage's loop, with the true preferred index (never OK:
        // every tile walk stops only on a non-OK step or past the last tile, where no bytes remain)
        const Step s = cut_input_message(base, len, pos, pf_true, C.max_body_size, (run.flags & B2_RUN_CLIENT) != 0, run_mask(C.proto_mask, run.flags));
        b2_run_status st;
        st.consumed = s.new_pos; st.parse_error = (uint32_t)s.err; st.n_msgs = s_carry_sum; st.first_msg = 0;
        st.preferred_proto = s.pf; st.n_unanswered = 0; st.resp_off = 0; st.resp_bytes = 0;
        B.run_status[r] = st;
    }
    // the last CTA to get here turns the per-run counts into first_msg (was a separate launch)
    __shared__ uint32_t s_ticket, s_pw[8], s_pc;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(B.totals + 4, 1u);
    __syncthreads();
    if (s_ticket == gridDim.x - 1) { __threadfence(); run_prefix_body(B, s_pw, &s_pc); }
}

// --- k_frame_table ------------------------------------------------------------
struct EmitFrame {
    uint32_t* out; uint32_t* out_run; uint32_t run_off; uint32_t run_idx; uint32_t cap_left; uint32_t* out_row;
    __device__ __forceinline__ void operator()(uint32_t i, const Step& s) const {
        if (i < cap_left) { out[i] = (run_off + s.frame_pos) | ((uint32_t)(s.index != 1) << 31); out_run[i] = run_idx; if (out_row) out_row[i] = kNone; }
    }
};
// kSpecK threads per tile: a live tile that k_resolve accepted as speculated hands over the offsets k_tile_walk
// kept (plain copy, no header loads); a tile that was re-walked or holds more than kSpecK frames is walked again by
// its first thread.
__global__ void __launch_bounds__(256) k_frame_table(BatchPtrs B, DevConfig C) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t spec_k = C.spec_k;
    const uint32_t t = g / spec_k, j = g % spec_k;
    if (t >= B.n_tiles) return;
    const TileRec rec = B.tiles[t];
    if (!rec.live || rec.count == 0) return;
    if (B.totals[2] & 1u) return;
    const uint4 ti = __ldg(B.tile_info + t);
    const uint32_t r = ti.w & 0xffffffu;
    const uint32_t first = B.run_status[r].first_msg + B.tile_base[t];
    if (!(rec.kind & kKindRewalked) && rec.count <= spec_k) {
        if (j < rec.count && first + j < B.max_msgs) {
            B.frame_off[first + j] = B.tile_spec[(size_t)t * spec_k + j]; B.frame_run[first + j] = r;
            if (C.pull) B.frame_row[first + j] = t * spec_k + j;
        }
        return;
    }
    if (j != 0) return;
    const uint32_t k = ti.z;
    b2_run run; run.offset = ti.x; run.length = ti.y; run.flags = ti.w >> 24;
    TileRec tmp;
    EmitFrame e; e.out = B.frame_off + first; e.out_run = B.frame_run + first; e.run_off = run.offset; e.run_idx = r; e.cap_left = B.max_msgs - first;
    e.out_row = C.pull ? B.frame_row + first : nullptr;
    walk_tile<false>(B.bytes + run.offset, run.length, rec.entry, rec.pf_in, (k + 1) << C.tile_shift, C.max_body_size, (run.flags & B2_RUN_CLIENT) != 0, tmp, e, run_mask(C.proto_mask, run.flags));
}

// --- k_decode: one thread per message ----------------------------------------
// four bytes at any alignment from two aligned words (reads up to 3 bytes past p + 3: every buffer compared here
// has that much slack — staged rows, the padded batch buffer, the char arrays inside DevMethod)
__device__ __forceinline__ uint32_t ld32_any(const uint8_t* p) {
    const uint32_t* q = reinterpret_cast<const uint32_t*>((uintptr_t)p & ~(uintptr_t)3);
    const uint32_t sh = 8u * (uint32_t)((uintptr_t)p & 3u);
    return sh ? __funnelshift_r(q[0], q[1], sh) : q[0];
}
__device__ __forceinline__ bool bytes_eq(const uint8_t* a, const char* b, uint32_t n) {
    const uint8_t* bb = reinterpret_cast<const uint8_t*>(b);
    uint32_t i = 0;
    for (; i + 4 <= n; i += 4) if (ld32_any(a + i) != ld32_any(bb + i)) return false;
    const uint32_t rem = n - i;
    if (rem == 0) return true;
    const uint32_t mask = (1u << (8 * rem)) - 1u;
    return ((ld32_any(a + i) ^ ld32_any(bb + i)) & mask) == 0;
}
// Server::FindMethodPropertyByFullName(service, method): key = service + '.' + method (server.cpp:1970-1988)
__device__ __forceinline__ int find_method(const DevMethod* ms, uint32_t n, const uint8_t* svc, uint32_t svc_len,
                                           const uint8_t* mth, uint32_t mth_len, bool& no_service) {
    no_service = false;
    bool has_dot = false;
    for (uint32_t i = 0; i < svc_len && !has_dot; i += 4) {               // four bytes per step: any '.' among the valid ones
        uint32_t e = __vcmpeq4(ld32_any(svc + i), 0x2e2e2e2eu);
        if (svc_len - i < 4) e &= (1u << (8 * (svc_len - i))) - 1u;
        has_dot = e != 0;
    }
    const char* full = nullptr; uint32_t full_len = 0;
    if (!has_dot) {                                   // jprotobuf short service name (baidu_rpc_protocol.cpp:738-748)
        int sp = -1;
        for (uint32_t m = 0; m < n; m++)
            if (ms[m].service_short_len == svc_len && bytes_eq(svc, ms[m].service_short, svc_len)) { sp = (int)m; break; }
        if (sp < 0) { no_service = true; return -1; }
        full = ms[sp].service_full; full_len = ms[sp].service_full_len;
    }
    for (uint32_t m = 0; m < n; m++) {
        const DevMethod& d = ms[m];
        const uint32_t sl = has_dot ? svc_len : full_len;
        if (d.full_method_len != sl + 1 + mth_len) continue;
        bool eq = has_dot ? bytes_eq(svc, d.full_method, sl) : bytes_eq((const uint8_t*)full, d.full_method, sl);
        eq = eq && d.full_method[sl] == '.' && bytes_eq(mth, d.full_method + sl + 1, mth_len);
        if (eq) return (int)m;
    }
    return -1;
}
__device__ __forceinline__ uint32_t strnlen_dev(const uint8_t* s, uint32_t n) { uint32_t i = 0; while (i < n && s[i]) i++; return i; }

__device__ __forceinline__ uint32_t cstr_len_compress(int32_t t) { return t == 0 ? 4 : t == 1 ? 6 : (t == 2 || t == 3) ? 4 : 7; }   // none snappy gzip zlib unknown
__device__ __forceinline__ uint32_t cstr_len_checksum(int32_t t) { return t == 0 ? 4 : t == 1 ? 6 : 7; }                          // none crc32c unknown

// bytes of "[identity][E<code>]" + reason
__device__ __forceinline__ uint32_t error_text_len(const DevConfig& C, const DevMethod* ms, const b2_msg_desc& d, const MsgAux& a,
                                                   const uint8_t* frame) {
    uint32_t n = (C.identity_len ? C.identity_len + 2 : 0) + 3 + dec_len((uint32_t)d.error_code);
    const uint32_t req_size = d.body_size - d.meta_size;
    switch (a.err_kind) {
    case kErrAttachment:   // "attachment_size=%d is larger than request_size=%d"
        n += 16 + dec_len_i32(d.attachment_size) + 29 + dec_len(req_size); break;
    case kErrNoService:    // "Fail to find service=%s"
        n += 21 + strnlen_dev(frame + a.svc_off, a.svc_len); break;
    case kErrNoMethod:     // "Fail to find method=%s/%s"
        n += 20 + strnlen_dev(frame + a.svc_off, a.svc_len) + 1 + strnlen_dev(frame + a.mth_off, a.mth_len); break;
    case kErrParseRequest: // "Fail to parse request=%s, ContentType=%s, CompressType=%s, ChecksumType=%s, request_size=%d"
        n += 22 + ms[d.method_idx].request_type_len + 14 + 2 /*pb*/ + 15 + cstr_len_compress(d.compress_type) + 15 +
             cstr_len_checksum(d.checksum_type) + 15 + dec_len(req_size); break;
    }
    return n;
}

__device__ __forceinline__ bool snappy_preamble(const uint8_t* in, uint32_t n, uint32_t& ulen, uint32_t& used);
__host__ __device__ __forceinline__ uint32_t snappy_max_compressed_length(uint32_t n) { return 32 + n + n / 6; }   // snappy.cc:55-77
// k_decode stages the first kRowBytes of every frame (header + RpcMeta + first body bytes) in
// shared memory with coalesced 4-byte loads (one row per lane) and decodes from there; the head
// records are assembled in shared memory and leave with coalesced 16-byte stores.
#ifndef B2_ROW_BYTES
#define B2_ROW_BYTES 160
#endif
constexpr uint32_t kRowBytes = B2_ROW_BYTES, kRowVecs = kRowBytes / 16;
constexpr uint32_t kDecodeWarps = 4;
#ifndef B2_DECODE_MIN_BLOCKS
#define B2_DECODE_MIN_BLOCKS 6
#endif
struct DecodeWarpSmem {
    alignas(16) uint8_t head[32][kHeadBytes];
    alignas(16) uint4 row[32][kRowVecs + 1];       // +1: odd 16-byte stride spreads the rows over the banks
};

// k_fused: a reply that cannot sit at its request's offset (errors, CRC'd / compressed bodies, outputs of decoders) gets a slot in the
// overflow area behind the batch-shaped part of the resp region; order there is first come, first served (replies are iovec-style)
__device__ __forceinline__ uint32_t fused_overflow_slot(const BatchPtrs& B, const DevConfig& C, uint32_t slot_len) {
    const uint32_t so = atomicAdd(B.totals + 9, slot_len);
    if ((uint64_t)C.ovf_base + so + slot_len > B.max_resp) { atomicOr(B.totals + 2, 2u); return 0; }
    return C.ovf_base + so;
}
constexpr uint16_t kDeferred = 0xffff;        // b2_msg_desc.status between k_fused and k_pack_slow: decode not done yet (a gzip / zlib body)
struct DecodeOut { uint32_t prefix, rs; bool fast, slow; };        // k_fused: reply prefix length, where the reply starts in resp, disposition
// decode_one = decode_one_impl<kFused, false>, which stops short (returns true, nothing written) at a gzip / zlib body: sizing one walks a
// DEFLATE stream, and that code must not sit inside the hot instantiation (registers, spills).  Such a message is decoded again by the
// out-of-line decode_one_gz = decode_one_impl<kFused, true>.
template <bool kFused, bool kGz>
__device__ __forceinline__ bool decode_one_impl(const BatchPtrs& B, const DevConfig& C, uint32_t i, uint32_t fo_raw,
                                                const uint8_t* srow, uint8_t* shead, uint32_t row_bytes, uint32_t run_idx, DecodeOut* out);
template <bool kFused>
__device__ __noinline__ void decode_one_gz(BatchPtrs B, DevConfig C, uint32_t i, uint32_t fo_raw,
                                           const uint8_t* srow, uint8_t* shead, uint32_t row_bytes, uint32_t run_idx, DecodeOut* out);
template <bool kFused = false>
__device__ __forceinline__ void decode_one(const BatchPtrs& B, const DevConfig& C, uint32_t i, uint32_t fo_raw,
                                           const uint8_t* srow, uint8_t* shead, uint32_t row_bytes, uint32_t run_idx = kNone, DecodeOut* out = nullptr) {
    if (decode_one_impl<kFused, false>(B, C, i, fo_raw, srow, shead, row_bytes, run_idx, out)) {
        if (kFused) {
            // k_fused keeps no call in its loop at all: the message is parked (kDeferred) and decoded by k_pack_slow, which runs behind it
            b2_msg_desc d; d.run_idx = run_idx; d.frame_off = fo_raw; d.status = kDeferred; d.resp_len = 0; d.resp_off = 0;
            B.msgs[i] = d;
            out->fast = false; out->prefix = 0; out->rs = 0; out->slow = true;
        } else decode_one_gz<kFused>(B, C, i, fo_raw, srow, shead, row_bytes, run_idx, out);
    }
}

// one warp round: 32 consecutive messages starting at i0 (staging, decode, head write-out)
__device__ __forceinline__ void decode_round(const BatchPtrs& B, const DevConfig& C, DecodeWarpSmem& S, uint32_t i0, uint32_t n_msgs, uint32_t lane) {
    const uint32_t i = i0 + lane;
    const uint32_t fo_raw = i < n_msgs ? B.frame_off[i] : 0;
    const uint32_t my_row = (C.pull && i < n_msgs) ? B.frame_row[i] : kNone;      // B2_INPUT_PULL: the walk stashed this frame's first 128 bytes
    const uint32_t nm = min(32u, n_msgs - i0);
    // stage: row m <- the 16-byte aligned vectors covering frame m's first bytes; half a warp per row
    const uint32_t sub = lane & 15, half = lane >> 4;
    for (uint32_t m2 = 0; m2 < nm; m2 += 2) {
        const uint32_t m = m2 + half;
        const uint32_t f = __shfl_sync(0xffffffffu, fo_raw, m & 31) & 0x7fffffffu;
        const uint32_t row = __shfl_sync(0xffffffffu, my_row, m & 31);
        if (m < nm && sub < kRowVecs && (row == kNone || sub < C.pull_vecs)) {
            // cp.async (LDGSTS): global -> shared without a register round trip, so all 16 trips are in flight together
            const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&S.row[m][sub]);
            const uint4* src = row == kNone ? reinterpret_cast<const uint4*>(B.bytes + (f & ~15u)) + sub       // (buffer is padded past its end)
                                            : B.rows + (size_t)row * 8 + sub;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    bool is_slow = false, is_verify = false;
    if (i < n_msgs) {
        decode_one(B, C, i, fo_raw, reinterpret_cast<const uint8_t*>(S.row[lane]) + (fo_raw & 15u), S.head[lane], my_row == kNone ? kRowBytes : 16u * C.pull_vecs);
        const uint32_t f = B.jobs[i].fast; is_slow = f == 0; is_verify = f == 2;
    }
    const uint32_t slow_mask = __ballot_sync(0xffffffffu, is_slow);
    if (slow_mask) {                                                    // k_pack_slow returns at once when totals[3] stays 0
        uint32_t sbase = 0;
        if (lane == 0) sbase = atomicAdd(B.totals + 3, (uint32_t)__popc(slow_mask));
        sbase = __shfl_sync(0xffffffffu, sbase, 0);
        if (is_slow) B.slow_idx[sbase + __popc(slow_mask & ((1u << lane) - 1u))] = i;
    }
    const uint32_t ver_mask = __ballot_sync(0xffffffffu, is_verify);
    if (ver_mask) {                                                     // verify list: same array, filled from the top
        uint32_t vbase = 0;
        if (lane == 0) vbase = atomicAdd(B.totals + 7, (uint32_t)__popc(ver_mask));
        vbase = __shfl_sync(0xffffffffu, vbase, 0);
        if (is_verify) B.slow_idx[B.max_msgs - 1 - (vbase + __popc(ver_mask & ((1u << lane) - 1u)))] = i;
    }
    __syncwarp();
    // heads of 32 consecutive messages are contiguous: coalesced 16-byte stores
    {
        const uint4* hs = reinterpret_cast<const uint4*>(&S.head[0][0]);
        uint4* hd = reinterpret_cast<uint4*>(B.heads + (size_t)i0 * kHeadBytes);
        for (uint32_t k = lane; k < nm * (kHeadBytes / 16); k += 32) hd[k] = hs[k];
    }
    __syncwarp();
}

// persistent: a fixed grid (multiple of the SM count) strides over the device-side message count
__global__ void __launch_bounds__(kDecodeWarps * 32, B2_DECODE_MIN_BLOCKS) k_decode(BatchPtrs B, DevConfig C) {
    __shared__ DecodeWarpSmem smem[kDecodeWarps];
    const uint32_t n_msgs = B.totals[0];
    if (B.totals[2] & 1u) return;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t i0 = (blockIdx.x * kDecodeWarps + wid) * 32; i0 < n_msgs; i0 += gridDim.x * kDecodeWarps * 32)
        decode_round(B, C, smem[wid], i0, n_msgs, lane);
}

template <bool kFused>
__device__ __noinline__ void decode_one_gz(BatchPtrs B, DevConfig C, uint32_t i, uint32_t fo_raw,
                                           const uint8_t* srow, uint8_t* shead, uint32_t row_bytes, uint32_t run_idx, DecodeOut* out) {
    decode_one_impl<kFused, true>(B, C, i, fo_raw, srow, shead, row_bytes, run_idx, out);
}
template <bool kFused, bool kGz>
__device__ __forceinline__ bool decode_one_impl(const BatchPtrs& B, const DevConfig& C, uint32_t i, uint32_t fo_raw,
                                                const uint8_t* srow, uint8_t* shead, uint32_t row_bytes, uint32_t run_idx, DecodeOut* out) {
    const uint32_t fo = fo_raw & 0x7fffffffu;
    // bit 31 of a frame offset says "not baidu_std": which of the other handlers cut it is read off its magic
    int proto = B2_PROTOCOL_BAIDU_STD;
    if (fo_raw >> 31) { const uint32_t mg = load_le32(srow); proto = mg == kMagicSTRM ? 2 : mg == kMagicHULU ? 3 : mg == kMagicSOFA ? 4 : 12; }
    const uint8_t* gframe = B.bytes + fo;
    const uint32_t my_run = kFused ? run_idx : B.frame_run[i];
    if (B.runs[my_run].flags & B2_RUN_RPC_DUMP) {
        // a record of an rpc_dump file: RpcDumpMeta + the sampled request; a baidu_std sample becomes the request frame rpc_replay would send
        // (the frame itself is written by pack_one: status B2_MSG_REPLAY)
        b2_msg_desc d;
        d.run_idx = my_run; d.frame_off = fo; d.body_size = load_be32(gframe + 4); d.meta_size = load_be32(gframe + 8);
        d.correlation_id = 0; d.log_id = 0; d.attachment_size = 0; d.compress_type = 0; d.checksum_type = 0; d.error_code = 0;
        d.has_bits = 0; d.protocol = 0; d.content_type = 0; d.method_idx = -1; d.status = B2_MSG_BAD_META; d.resp_off = 0; d.resp_len = 0;
        MsgAux a; a.msg_off = a.msg_len = a.att_len = a.att_off = a.cks_off = a.cks_len = 0; a.svc_off = a.svc_len = a.mth_off = a.mth_len = 0; a.pad = 0; a.err_kind = kErrNone;
        DumpMetaOut dm; uint32_t slot_len = 0;
        if (decode_dump_meta(gframe + 12, d.meta_size, dm)) {
            d.protocol = (uint8_t)dm.protocol_type; d.compress_type = dm.compress_type; d.attachment_size = dm.attachment_size; d.has_bits = (uint16_t)dm.has;
            const uint32_t first = B.run_status[my_run].first_msg;
            d.correlation_id = (long long)(B.runs[my_run].socket_id + (unsigned long long)(i - first));
            if (dm.protocol_type != B2_PROTOCOL_BAIDU_STD) d.status = B2_MSG_UNSUPPORTED;           // rpc_replay sends it on another protocol's channel
            else {
                d.status = B2_MSG_REPLAY;
                const uint32_t req = d.body_size - d.meta_size;
                const uint32_t att = dm.attachment_size > 0 ? (uint32_t)dm.attachment_size : 0u;      // (rpc_replay.cpp:184-188)
                a.svc_off = 12 + dm.service_name.off; a.svc_len = dm.service_name.len; a.mth_off = 12 + dm.method_name.off; a.mth_len = dm.method_name.len;
                a.att_len = att; a.msg_len = req;
                d.resp_len = 12 + replay_meta_len(a.svc_len, a.mth_len, dm.compress_type, d.correlation_id, att) + req;
                slot_len = (d.resp_len + 15u) & ~15u;
            }
        }
        B.msgs[i] = d;
        if (kFused) {
            out->fast = false; out->prefix = 0; out->rs = 0; out->slow = d.status == B2_MSG_REPLAY;
            if (out->slow) { B.aux[i] = a; B.slot[i] = fused_overflow_slot(B, C, slot_len); }
            return false;
        }
        B.aux[i] = a; B.slot[i] = slot_len;
        PackJob job; job.src_off = 0; job.bulk_len = 0; job.head_len = 0; job.pad = 0; job.fast = 0; job.slot_len = slot_len;
        B.jobs[i] = job;
        if (C.by_ref) B.refs[i] = make_uint4(0, 0, 0, 0);
        return false;
    }
    if (proto > 2) {
        // hulu_pbrpc / sofa_pbrpc / nshead: framed on the device, processed by the host (ProcessHuluRequest ... stay there): the descriptor
        // carries protocol, frame_off, meta_size and body_size (the bytes behind the 12 / 24 / 36-byte header)
        b2_msg_desc d;
        d.run_idx = my_run; d.frame_off = fo;
        if (proto == 3) { d.body_size = load_le32(srow + 4); d.meta_size = load_le32(srow + 8); }
        else if (proto == 4) { d.meta_size = load_le32(srow + 4); d.body_size = load_le32(srow + 16); }
        else { d.meta_size = 0; d.body_size = load_le32(srow + 32); }
        d.correlation_id = 0; d.log_id = 0; d.attachment_size = 0; d.compress_type = 0; d.checksum_type = 0; d.error_code = 0;
        d.has_bits = 0; d.protocol = (uint8_t)proto; d.content_type = 0; d.method_idx = -1; d.status = B2_MSG_FRAMED; d.resp_off = 0; d.resp_len = 0;
        B.msgs[i] = d;
        if (kFused) { out->fast = false; out->slow = false; out->prefix = 0; out->rs = 0; return false; }
        MsgAux a; a.msg_off = a.msg_len = a.att_len = a.att_off = a.cks_off = a.cks_len = 0; a.svc_off = a.svc_len = a.mth_off = a.mth_len = 0; a.pad = 0; a.err_kind = kErrNone;
        B.aux[i] = a; B.slot[i] = 0;
        PackJob job; job.src_off = 0; job.bulk_len = 0; job.head_len = 0; job.pad = 0; job.fast = 0; job.slot_len = 0;      // (pack_one returns at once: no reply)
        B.jobs[i] = job;
        if (C.by_ref) B.refs[i] = make_uint4(0, 0, 0, 0);
        return false;
    }
    // decode from the staged copy when header + meta + the first body bytes are inside it
    const uint32_t meta_size_peek = load_be32(srow + 8);
    // (the staged bytes must hold header, meta, the pb field header of the body and — when the reply is materialised — the <= 15 payload
    // bytes that travel in the head record; by-reference replies take none of the payload)
    const bool staged = (uint64_t)(fo_raw & 15u) + 12ull + meta_size_peek + (C.by_ref ? 8ull : 40ull) <= row_bytes;
    const uint8_t* frame = staged ? srow : gframe;
    b2_msg_desc d;
    d.frame_off = fo; d.body_size = load_be32(frame + 4); d.meta_size = load_be32(frame + 8);
    d.correlation_id = 0; d.log_id = 0; d.attachment_size = 0; d.compress_type = 0; d.checksum_type = 0; d.error_code = 0;
    d.has_bits = 0; d.protocol = (uint8_t)proto; d.content_type = 0; d.method_idx = -1; d.status = 0; d.resp_off = 0; d.resp_len = 0;
    d.run_idx = kFused ? run_idx : B.frame_run[i];
    MsgAux a; a.msg_off = a.msg_len = a.att_len = a.att_off = a.cks_off = a.cks_len = 0;
    a.svc_off = a.svc_len = a.mth_off = a.mth_len = 0; a.pad = 0; a.err_kind = kErrNone;
    uint32_t resp_len = 0, reserve = 0;               // reserve: slot bytes beyond resp_len a second outcome may need
    uint32_t ref_prefix = 0;                          // B2_RESP_BY_REF: bytes of the reply that are materialised (0 = the whole reply)
    const uint8_t* meta_p = frame + 12;
    const uint32_t req_size = d.body_size - d.meta_size;
    if (proto == B2_PROTOCOL_STREAMING_RPC) {
        StreamMetaOut sm;
        if (!decode_stream_meta(meta_p, d.meta_size, sm)) d.status = B2_MSG_BAD_STREAM_META;
        else {
            d.status = B2_MSG_STREAM_FRAME; d.correlation_id = sm.stream_id; d.log_id = sm.source_stream_id;
            d.compress_type = sm.frame_type; d.has_bits = (uint16_t)sm.has;
            d.attachment_size = (int32_t)(uint32_t)((uint64_t)sm.consumed_size & 0xffffffffu);
            d.checksum_type = (int32_t)(uint32_t)((uint64_t)sm.consumed_size >> 32);
            if (C.stream_handler == B2_STREAM_SNAPPY_UNCOMPRESS && (sm.has & B2_SHAS_FRAME_TYPE) && sm.frame_type == 3 /*FRAME_TYPE_DATA*/) {
                uint32_t ulen = 0, used = 0;
                bool ok = snappy_preamble(gframe + 12 + d.meta_size, req_size, ulen, used);
                if (ok && (uint64_t)ulen > 32ull * req_size + 64ull) ok = false;
                if (!ok) d.error_code = B2_EREQUEST;
                else { a.msg_off = kNone; a.msg_len = ulen; a.att_off = req_size; resp_len = ulen ? ulen : 1; }
            }
        }
    } else {
        RpcMetaOut m;
        if (!decode_rpc_meta_fast(meta_p, d.meta_size, m) && !decode_rpc_meta(meta_p, d.meta_size, m)) d.status = B2_MSG_BAD_META;
        else {
            d.correlation_id = m.correlation_id; d.log_id = m.log_id; d.attachment_size = m.attachment_size;
            d.compress_type = m.compress_type; d.checksum_type = m.checksum_type; d.content_type = (uint8_t)m.content_type;
            d.has_bits = (uint16_t)m.has;
            if (m.has & B2_HAS_CHECKSUM_VALUE) { a.cks_off = 12 + m.checksum_value.off; a.cks_len = m.checksum_value.len; }
            if (m.has & B2_HAS_REQUEST) {
                a.svc_off = 12 + m.service_name.off; a.svc_len = m.service_name.len;
                a.mth_off = 12 + m.method_name.off; a.mth_len = m.method_name.len;
            }
            const int64_t att = m.attachment_size;
            const DevMethod* mp = nullptr;
            if (B.runs[d.run_idx].flags & B2_RUN_CLIENT) {
                // ---- client-side socket: ProcessRpcResponse (baidu_rpc_protocol.cpp:911-1013), EchoResponse channel
                d.status = B2_MSG_RESPONSE;
                const uint32_t res_size = req_size;
                if (m.error_code != 0) d.error_code = m.error_code;                                   // :960-965
                else if ((m.has & B2_HAS_ATTACHMENT_SIZE) && att > (int64_t)res_size) d.error_code = B2_ERESPONSE;   // :971-976
                else {
                    int64_t bwo = (int64_t)res_size - ((m.has & B2_HAS_ATTACHMENT_SIZE) ? att : 0);
                    if (bwo > (int64_t)res_size) bwo = res_size;
                    const uint32_t body_len = (uint32_t)bwo;
                    if (m.content_type != B2_CONTENT_TYPE_PB) d.status = B2_MSG_UNSUPPORTED;
                    else if ((m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB) && body_len > kGzMaxIn) d.status = B2_MSG_UNSUPPORTED;
                    else {
                        bool ok = !(m.checksum_type == B2_CHECKSUM_TYPE_CRC32C && a.cks_len != 4);
                        if (ok && m.compress_type == B2_COMPRESS_TYPE_NONE) {
                            Span msg; msg.off = 0; msg.len = 0;
                            ok = decode_echo_request(gframe + 12 + d.meta_size, body_len, msg);
                            if (ok) { a.msg_off = 12 + d.meta_size + msg.off; a.msg_len = msg.len; a.att_off = body_len; d.resp_off = fo + a.msg_off; resp_len = msg.len; }
                        } else if (ok && m.compress_type == B2_COMPRESS_TYPE_SNAPPY) {
                            uint32_t ulen = 0, used = 0;
                            ok = snappy_preamble(gframe + 12 + d.meta_size, body_len, ulen, used);
                            if (ok && (uint64_t)ulen > 32ull * body_len + 64ull) ok = false;
                            if (ok) { d.status = B2_MSG_RESPONSE_UNZ; a.msg_off = kNone; a.msg_len = ulen; a.att_off = body_len; resp_len = ulen ? ulen : 1; }
                        } else if (ok && (m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB)) {
                            // GzipDecompress / ZlibDecompress (policy/gzip_compress.cpp:75-89): sized here, inflated by the pack stage
                            if (!kGz) return true;
                            bool big = false;
                            const uint32_t ulen = gz_input_stream<false>(gframe + 12 + d.meta_size, body_len, m.compress_type, nullptr, kGzMaxOut, &big);
                            if (big) { d.status = B2_MSG_UNSUPPORTED; }
                            else { d.status = B2_MSG_RESPONSE_UNZ; a.msg_off = kNone; a.msg_len = ulen; a.att_off = body_len; resp_len = ulen ? ulen : 1; }
                        } else ok = false;
                        if (!ok) { d.error_code = B2_EREQUEST; resp_len = 0; d.status = B2_MSG_RESPONSE; }  // :999-1007
                        if (d.status == B2_MSG_UNSUPPORTED) resp_len = 0;
                    }
                }
                d.resp_len = resp_len;
                B.msgs[i] = d; B.aux[i] = a;
                const uint32_t csl = d.status == B2_MSG_RESPONSE_UNZ ? ((resp_len + 15u) & ~15u) : 0u;
                if (kFused) {
                    // (an EMPTY message under a CRC32C checksum still has its checksum to verify: pack_one does, so it must see the message)
                    out->fast = false; out->prefix = 0; out->rs = 0;
                    out->slow = resp_len > 0 || (d.status == B2_MSG_RESPONSE && d.error_code == 0 && d.checksum_type == B2_CHECKSUM_TYPE_CRC32C);
                    B.slot[i] = csl ? fused_overflow_slot(B, C, csl) : 0u;
                    return false;
                }
                B.slot[i] = csl;
                PackJob cj; cj.src_off = 0; cj.bulk_len = 0; cj.head_len = 0; cj.pad = 0; cj.fast = 0; cj.slot_len = 0;
                B.jobs[i] = cj;
                if (C.by_ref) B.refs[i] = make_uint4(0, 0, 0, 0);            // (nothing is by reference on the client side; the entry is part of the output)
                return false;
            }
            if ((m.has & B2_HAS_ATTACHMENT_SIZE) && (int64_t)req_size < att) {
                a.err_kind = kErrAttachment; d.error_code = B2_EREQUEST;
            } else {
                bool no_service;
                const int mi = find_method(B.methods, C.n_methods, frame + a.svc_off, a.svc_len, frame + a.mth_off, a.mth_len, no_service);
                if (no_service) { a.err_kind = kErrNoService; d.error_code = B2_ENOSERVICE; }
                else if (mi < 0) { a.err_kind = kErrNoMethod; d.error_code = B2_ENOMETHOD; }
                else { d.method_idx = (int16_t)mi; mp = B.methods + mi; }
            }
            if (mp && mp->handler == B2_HANDLER_HOST) d.status = B2_MSG_HOST;
            else if (mp) {
                int64_t bwo = (int64_t)req_size - att;
                if (bwo > (int64_t)req_size) bwo = req_size;
                const uint32_t body_wo_att = (uint32_t)bwo;
                const uint32_t in_att_len = att > 0 ? (uint32_t)att : 0;
                if (m.content_type != B2_CONTENT_TYPE_PB) d.status = B2_MSG_UNSUPPORTED;
                else if (mp->response_compress_type != B2_COMPRESS_TYPE_NONE && mp->response_compress_type != B2_COMPRESS_TYPE_SNAPPY) d.status = B2_MSG_UNSUPPORTED;
                else if ((m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB) && body_wo_att > kGzMaxIn) d.status = B2_MSG_UNSUPPORTED;
                else if (m.compress_type == B2_COMPRESS_TYPE_SNAPPY || m.compress_type == B2_COMPRESS_TYPE_GZIP || m.compress_type == B2_COMPRESS_TYPE_ZLIB) {
                    // SnappyDecompress (policy/snappy_compress.cpp:51-70) happens in the pack stage; here only the
                    // announced length is read to reserve the reply slot.  A stream cannot expand more than ~22x
                    // (a 3-byte copy yields <= 64 bytes), so an announced length beyond 32x + 64 must fail.
                    // GzipDecompress / ZlibDecompress (policy/gzip_compress.cpp:75-89) announce nothing: a sizing pass walks the stream
                    uint32_t ulen = 0, used = 0;
                    bool ok = !(m.checksum_type == B2_CHECKSUM_TYPE_CRC32C && a.cks_len != 4), big = false;
                    if (m.compress_type == B2_COMPRESS_TYPE_SNAPPY) {
                    if (ok) ok = snappy_preamble(gframe + 12 + d.meta_size, body_wo_att, ulen, used);
                    if (ok && (uint64_t)ulen > 32ull * body_wo_att + 64ull) ok = false;
                    } else if (ok) {
                        if (!kGz) return true;
                        ulen = gz_input_stream<false>(gframe + 12 + d.meta_size, body_wo_att, m.compress_type, nullptr, kGzMaxOut, &big);
                    }
                    if (big) d.status = B2_MSG_UNSUPPORTED;
                    else if (!ok) { a.err_kind = kErrParseRequest; d.error_code = B2_EREQUEST; }
                    else {
                        d.status = B2_MSG_ECHOED;
                        a.msg_off = kNone; a.msg_len = ulen;        // resolved after decompression
                        if (mp->echo_attachment) { a.att_len = in_att_len; a.att_off = 12 + d.meta_size + body_wo_att; }
                        const uint32_t cks_len = mp->response_checksum_type == B2_CHECKSUM_TYPE_CRC32C ? 4u : a.cks_len;
                        const uint32_t ml = response_meta_len(0, 0, mp->response_compress_type, m.correlation_id, a.att_len, mp->response_checksum_type, cks_len);
                        resp_len = 12 + ml + 8 + ulen + a.att_len;   // upper bound; the pack stage writes the real length
                        if (mp->response_compress_type == B2_COMPRESS_TYPE_SNAPPY) resp_len = 12 + ml + snappy_max_compressed_length(ulen + 8) + a.att_len;
                        a.pad = 0;
                    }
                }
                else if (m.compress_type != B2_COMPRESS_TYPE_NONE) { a.err_kind = kErrParseRequest; d.error_code = B2_EREQUEST; }
                else {
                    Span msg; msg.off = 0; msg.len = 0;
                    bool ok = true;
                    if (m.checksum_type == B2_CHECKSUM_TYPE_CRC32C && a.cks_len != 4) ok = false;   // reference CHECK-aborts; see DESIGN.md
                    if (ok) {
                        // canonical body "0a <len> <message>": recognised from the staged bytes without walking
                        const uint8_t* sb = meta_p + d.meta_size;
                        bool canon = false;
                        if (staged && body_wo_att >= 2 && sb[0] == 0x0a) {
                            Reader r; r.p = sb + 1; r.end = sb + (body_wo_att < 6 ? body_wo_att : 6);
                            uint64_t l;
                            if (rd_varint(r, l) && l <= 0x7fffffefull && (uint64_t)(r.p - sb) + l == body_wo_att) {
                                canon = true; msg.off = (uint32_t)(r.p - sb); msg.len = (uint32_t)l;
                            }
                        }
                        if (!canon) ok = decode_echo_request(gframe + 12 + d.meta_size, body_wo_att, msg);
                    }
                    if (!ok) { a.err_kind = kErrParseRequest; d.error_code = B2_EREQUEST; }
                    else {
                        d.status = B2_MSG_ECHOED;
                        a.msg_off = 12 + d.meta_size + msg.off; a.msg_len = msg.len;
                        if (mp->echo_attachment) { a.att_len = in_att_len; a.att_off = 12 + d.meta_size + body_wo_att; }
                        const uint32_t cks_len = mp->response_checksum_type == B2_CHECKSUM_TYPE_CRC32C ? 4u : a.cks_len;
                        const uint32_t ml = response_meta_len(0, 0, mp->response_compress_type, m.correlation_id, a.att_len,
                                                              mp->response_checksum_type, cks_len);
                        const uint32_t prefix = 12 + ml + 1 + varint_len(msg.len);
                        resp_len = prefix + msg.len + a.att_len;
                        a.pad = (fo + a.msg_off - prefix) & 15u;       // payload keeps its (mod 16) alignment
                        // B2_RESP_BY_REF: only the prefix is materialised (same conditions as the bandwidth path below)
                        // k_fused: the reply is assembled IN PLACE over the request's own bytes (prefix right in front of the payload), so
                        // it also has to fit there; CRC-carrying requests are verified by k_pack_slow
                        if ((C.by_ref || kFused) && mp->response_checksum_type == B2_CHECKSUM_TYPE_NONE && mp->response_compress_type == B2_COMPRESS_TYPE_NONE &&
                            (a.att_len == 0 || a.att_off == a.msg_off + a.msg_len) && prefix <= 64 &&
                            (!kFused || (prefix <= a.msg_off && m.checksum_type != B2_CHECKSUM_TYPE_CRC32C))) { a.pad = 0; ref_prefix = prefix; }
                        if (mp->response_compress_type == B2_COMPRESS_TYPE_SNAPPY) {
                            resp_len = 12 + ml + snappy_max_compressed_length(1 + varint_len(msg.len) + msg.len) + a.att_len; a.pad = 0;
                        }
                    }
                }
            }
            if (a.err_kind != kErrNone) {
                d.status = B2_MSG_ERROR_REPLIED;
                const uint32_t tl = error_text_len(C, B.methods, d, a, frame);
                resp_len = 12 + response_meta_len(d.error_code, tl, 0, m.correlation_id, 0, 0, a.cks_len);
            }
            // a CRC-verified request can still turn into an EREQUEST reply in k_pack: reserve for both
            if (d.status == B2_MSG_ECHOED && (m.checksum_type == B2_CHECKSUM_TYPE_CRC32C || m.compress_type != B2_COMPRESS_TYPE_NONE)) {
                b2_msg_desc e = d; MsgAux ea = a; e.error_code = B2_EREQUEST; ea.err_kind = kErrParseRequest;
                const uint32_t tl = error_text_len(C, B.methods, e, ea, frame);
                const uint32_t el = 12 + response_meta_len(B2_EREQUEST, tl, 0, m.correlation_id, 0, 0, a.cks_len);
                if (a.pad + (ref_prefix ? ref_prefix : resp_len) < el) reserve = el - a.pad;    // slot must hold either reply (error reply is packed at pad 0)
            }
        }
    }
    d.resp_len = resp_len;
    if (!kFused) { B.msgs[i] = d; B.aux[i] = a; }
    const uint32_t slot_len = resp_len ? ((a.pad + max(ref_prefix ? ref_prefix : resp_len, reserve) + 15u) & ~15u) : 0u;
    if (!kFused) B.slot[i] = slot_len;
    uint4 ref = make_uint4(0, 0, 0, 0);
    // ---- bandwidth path: pre-build the reply prefix, shifted to the slot alignment -------------
    PackJob job; job.src_off = 0; job.bulk_len = 0; job.head_len = 0; job.pad = (uint8_t)a.pad; job.fast = 0; job.slot_len = slot_len;
    if (d.status == B2_MSG_ECHOED && d.compress_type == B2_COMPRESS_TYPE_NONE &&
        B.methods[d.method_idx].response_checksum_type == B2_CHECKSUM_TYPE_NONE &&
        B.methods[d.method_idx].response_compress_type == B2_COMPRESS_TYPE_NONE &&
        (a.att_len == 0 || a.att_off == a.msg_off + a.msg_len)) {
        const uint32_t ml = response_meta_len(0, 0, 0, d.correlation_id, a.att_len, 0, a.cks_len);
        const uint32_t vl = varint_len(a.msg_len);
        const uint32_t prefix = 12 + ml + 1 + vl;
        if (prefix <= 64) {
            const uint32_t n = a.msg_len + a.att_len;
            const uint32_t gs = fo + a.msg_off;
            const uint32_t lead = ref_prefix ? 0u : min(n, (16u - (gs & 15u)) & 15u);
            const uint32_t hl = (a.pad + prefix + lead + 15u) & ~15u;
            uint8_t* h = shead;
            {   // zero the record first (six 16-byte stores) instead of byte loops for the pad and the tail
                uint4* hz = reinterpret_cast<uint4*>(h);
                #pragma unroll
                for (uint32_t k = 0; k < kHeadBytes / 16; k++) hz[k] = make_uint4(0, 0, 0, 0);
            }
            uint8_t* p = h + a.pad;
            p[0] = 'P'; p[1] = 'R'; p[2] = 'P'; p[3] = 'C';
            put_be32(p + 4, ml + 1 + vl + n); put_be32(p + 8, ml); p += 12;
            *p++ = 0x12; *p++ = 0x02; *p++ = 0x08; *p++ = 0x00; *p++ = 0x18; *p++ = 0x00;
            *p++ = 0x20; p = put_varint(p, (uint64_t)d.correlation_id);
            if (a.att_len) { *p++ = 0x28; p = put_varint(p, a.att_len); }
            *p++ = 0x50; *p++ = 0x00; *p++ = 0x58; *p++ = 0x00;
            *p++ = 0x62; p = put_varint(p, a.cks_len);
            for (uint32_t k = 0; k < a.cks_len; k++) *p++ = frame[a.cks_off + k];
            *p++ = 0x0a; p = put_varint(p, a.msg_len);
            for (uint32_t k = 0; k < lead; k++) *p++ = frame[a.msg_off + k];
            job.src_off = gs + lead; job.bulk_len = ref_prefix ? 0u : ((n - lead + 15u) & ~15u); job.head_len = (uint16_t)hl;
            if (ref_prefix) ref = make_uint4(prefix, gs, n, 0);
            // a CRC32C-carrying request takes the bandwidth path once k_pack_slow's verify pass has checked it (fast 2 -> 1)
            job.fast = d.checksum_type == B2_CHECKSUM_TYPE_CRC32C ? 2 : 1;
        }
    }
    if (kFused) {
        const bool fast = job.fast == 1 && ref_prefix != 0;
        if (fast) d.resp_off = fo + a.msg_off - ref_prefix;               // final: the reply sits right in front of its payload
        B.msgs[i] = d;
        out->fast = fast; out->prefix = ref_prefix; out->rs = d.resp_off; out->slow = !fast && resp_len > 0;
        if (out->slow) { B.aux[i] = a; B.slot[i] = slot_len ? fused_overflow_slot(B, C, slot_len) : 0u; }
        return false;
    }
    B.jobs[i] = job;
    if (C.by_ref) B.refs[i] = ref;
    return false;
}

// --- exclusive scan of slot sizes: 2 kernels ---------------------------------
constexpr int kScanBlock = 1024, kScanItems = 4;
__device__ __forceinline__ void scan_top_body(const BatchPtrs& B, uint32_t* s_warp, uint32_t* s_carry_p) {
    // serial-by-chunks exclusive scan of the block sums (<= a few thousand entries)
    const uint32_t n = B.totals[0];
    const uint32_t nb = (n + kScanBlock * kScanItems - 1) / (kScanBlock * kScanItems);
    if (threadIdx.x == 0) *s_carry_p = 0;
    __syncthreads();
    for (uint32_t base = 0; base < nb; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        uint32_t v = i < nb ? __ldcg(B.scan_tmp + i) : 0, x = v;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if ((threadIdx.x & 31) >= d) x += y; }
        if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = x;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = s_warp[threadIdx.x], ws = w;
            #pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, ws, d); if (threadIdx.x >= d) ws += y; }
            s_warp[threadIdx.x] = ws - w;
        }
        __syncthreads();
        const uint32_t excl = *s_carry_p + s_warp[threadIdx.x >> 5] + x - v;
        if (i < nb) B.scan_tmp[i] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) *s_carry_p = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) { B.totals[1] = *s_carry_p; if (*s_carry_p > B.max_resp) B.totals[2] |= 2u; }
}
__global__ void __launch_bounds__(kScanBlock) k_scan_blocks(BatchPtrs B) {
    __shared__ uint32_t s_warp[32];
    const uint32_t n = B.totals[0];
    for (uint32_t blk = blockIdx.x; blk * kScanBlock * kScanItems < n; blk += gridDim.x) {
    const uint32_t base = blk * kScanBlock * kScanItems + threadIdx.x * kScanItems;
    uint32_t v[kScanItems], sum = 0;
    #pragma unroll
    for (int j = 0; j < kScanItems; j++) { v[j] = base + j < n ? B.slot[base + j] : 0; sum += v[j]; }
    uint32_t x = sum;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if ((threadIdx.x & 31) >= d) x += y; }
    if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t w = s_warp[threadIdx.x], ws = w;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, ws, d); if (threadIdx.x >= d) ws += y; }
        s_warp[threadIdx.x] = ws - w;
        if (threadIdx.x == 31) B.scan_tmp[blk] = ws;
    }
    __syncthreads();
    uint32_t excl = s_warp[threadIdx.x >> 5] + x - sum;
    #pragma unroll
    for (int j = 0; j < kScanItems; j++) { if (base + j < n) B.slot[base + j] = excl; excl += v[j]; }
    __syncthreads();
    }
    // the last CTA to finish scans the block sums (was a separate launch)
    __shared__ uint32_t s_ticket, s_carry;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(B.totals + 5, 1u);
    __syncthreads();
    if (s_ticket == gridDim.x - 1) { __threadfence(); scan_top_body(B, s_warp, &s_carry); }
}
// --- finalize: per-run response span + counters (prologue of the last pack kernel) ----------------
__device__ __forceinline__ void finalize_runs(const BatchPtrs& B, const DevConfig& C) {
    const uint32_t n_msgs = B.totals[0];
    if (C.fused && blockIdx.x == 0 && threadIdx.x == 0) {          // span of the resp region in use: the batch-shaped part (+ the overflow area)
        const uint32_t ovf = B.totals[9];
        B.totals[1] = ovf ? C.ovf_base + ovf : C.ovf_base;
    }
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < B.n_runs; r += gridDim.x * blockDim.x) {
        b2_run_status st = B.run_status[r];
        auto off_of = [&](uint32_t i) -> uint32_t {
            if (i >= n_msgs) return B.totals[1];
            return B.slot[i] + B.scan_tmp[i / (kScanBlock * kScanItems)];
        };
        if (C.fused) { st.resp_off = B.runs[r].offset; st.resp_bytes = st.consumed; }      // replies sit at their requests' offsets
        else {
        st.resp_off = off_of(st.first_msg);
        st.resp_bytes = off_of(st.first_msg + st.n_msgs) - st.resp_off;
        }
        B.run_status[r] = st;
        atomicAdd(B.counters + 0, (unsigned long long)st.consumed);
        atomicAdd(B.counters + 1, (unsigned long long)st.n_msgs);
        atomicAdd(B.counters + 2, (unsigned long long)st.resp_bytes);
        if (st.parse_error != B2_PARSE_ERROR_NOT_ENOUGH_DATA) atomicAdd(B.counters + 4, 1ull);
        if (r == 0) atomicAdd(B.counters + 5, 1ull);
    }
}

// Snappy raw-format decoder as a warp-level primitive: butil::snappy::RawUncompress
// (src/butil/third_party/snappy/snappy.cc:716-787 DecompressAllTags, :1145-1215 SnappyArrayWriter,
// format_description.txt).  The tag stream is inherently serial; every lane follows it (the tag
// bytes are broadcast loads) and the bytes of each element are moved by the whole warp.  A copy may
// overlap its own output (offset < length, RLE): byte i comes from out[op - offset + i % offset],
// which was written by an earlier element, so the lanes are independent.  Returns true iff the
// stream is well formed, consumed exactly, and produced exactly the announced length.
__device__ __forceinline__ bool snappy_preamble(const uint8_t* in, uint32_t n, uint32_t& ulen, uint32_t& used) {
    uint32_t v = 0, shift = 0, ip = 0;              // SnappyDecompressor::ReadUncompressedLength, snappy.cc:690-711
    for (;;) {
        if (shift >= 32) return false;
        if (ip >= n) return false;
        const uint32_t c = in[ip++];
        v |= (c & 0x7f) << shift;
        if (c < 128) break;
        shift += 7;
    }
    ulen = v; used = ip;
    return true;
}
__device__ __forceinline__ void warp_copy(uint8_t* dst, const uint8_t* src, uint32_t n, uint32_t lane);
// `ring` (optional): kSnapRing bytes of shared memory owned by this warp, mirroring the most recent output
// (ring[p & (kSnapRing-1)] == out[p] for p in [op - kSnapRing, op)).  A copy whose offset fits in it reads its
// source from shared memory (a back-reference to bytes the warp has just stored would otherwise pay an L2 round
// trip per element: stores do not allocate in L1).  The tag stream itself is read 32 bytes at a time, one byte
// per lane, and walked with shuffles, so a run of short elements costs one global load.
constexpr uint32_t kSnapRing = 4096;
__device__ __forceinline__ uint32_t ring_ld(uint32_t ring_s, uint32_t p) {
    uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(ring_s + (p & (kSnapRing - 1))) : "memory"); return v;
}
__device__ __forceinline__ void ring_st(uint32_t ring_s, uint32_t p, uint32_t v) {
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(ring_s + (p & (kSnapRing - 1))), "r"(v) : "memory");
}
__device__ __noinline__ bool warp_snappy_decode(const uint8_t* in, uint32_t n, uint8_t* out, uint32_t cap, uint32_t lane,
                                                uint32_t& produced, uint8_t* ring = nullptr) {
    uint32_t ulen, ip;
    produced = 0;
    if (!snappy_preamble(in, n, ulen, ip)) return false;
    if (ulen > cap) return false;
    const bool use_ring = ring != nullptr;
    const uint32_t ring_s = use_ring ? (uint32_t)__cvta_generic_to_shared(ring) : 0u;
    uint32_t op = 0;
    // look-ahead window [wbase, wbase + 32): lane L holds bytes wbase+L .. wbase+L+4 (w_lo = first four, w_b4 = the fifth)
    uint32_t wbase = 0, wbyte = 0, w_lo = 0, w_b4 = 0;
    auto refill = [&](uint32_t at) {
        wbase = at;
        wbyte = (wbase + lane < n) ? in[wbase + lane] : 0u;
        const uint32_t b1 = __shfl_down_sync(0xffffffffu, wbyte, 1), b2 = __shfl_down_sync(0xffffffffu, wbyte, 2);
        const uint32_t b3 = __shfl_down_sync(0xffffffffu, wbyte, 3);
        w_b4 = __shfl_down_sync(0xffffffffu, wbyte, 4);
        w_lo = wbyte | (b1 << 8) | (b2 << 16) | (b3 << 24);
    };
    refill(ip);
    while (ip < n) {
        if (ip + 5 > wbase + 32) refill(ip);                          // a whole tag (<= 5 bytes) is inside, on lanes <= 27
        const uint32_t t = __shfl_sync(0xffffffffu, w_lo, ip - wbase);            // tag + three operand bytes
        const uint32_t c = t & 0xffu;
        ip++;
        if ((c & 3u) == 0) {                                         // literal
            uint32_t len = (c >> 2) + 1;
            if (len >= 61) {
                const uint32_t ll = len - 60;
                if (n - ip < ll) return false;
                const uint32_t v = (t >> 8) | (__shfl_sync(0xffffffffu, w_b4, ip - 1 - wbase) << 24);
                len = (ll == 4 ? v : (v & ((1u << (8 * ll)) - 1u))) + 1; ip += ll;
                if (len == 0) return false;                          // 2^32 wrap: cannot fit
            }
            if (len > n - ip) return false;                          // premature end of input
            if (len > ulen - op) return false;                       // SnappyArrayWriter::Append: no room
            if (ip + len <= wbase + 32) {                            // the literal's bytes are already in the window
                const uint32_t b = __shfl_sync(0xffffffffu, wbyte, (ip - wbase + lane) & 31);
                if (lane < len) { out[op + lane] = (uint8_t)b; if (use_ring) ring_st(ring_s, op + lane, b); }
            } else {
                warp_copy(out + op, in + ip, len, lane);
                if (use_ring) {                                      // keep the mirror: the last min(len, ring) bytes
                    const uint32_t keep = min(len, kSnapRing), skip = len - keep;
                    for (uint32_t i = lane; i < keep; i += 32) ring_st(ring_s, op + skip + i, in[ip + skip + i]);
                }
            }
            ip += len; op += len;
        } else {                                                     // copy
            uint32_t len, offset;
            if ((c & 3u) == 1) {
                if (n - ip < 1) return false;
                len = ((c >> 2) & 7u) + 4; offset = ((c >> 5) << 8) | ((t >> 8) & 0xffu); ip += 1;
            } else if ((c & 3u) == 2) {
                if (n - ip < 2) return false;
                len = (c >> 2) + 1; offset = (t >> 8) & 0xffffu; ip += 2;
            } else {
                if (n - ip < 4) return false;
                len = (c >> 2) + 1;
                offset = (t >> 8) | (__shfl_sync(0xffffffffu, w_b4, ip - 1 - wbase) << 24); ip += 4;
            }
            if (offset == 0 || offset > op) return false;            // AppendFromSelf: op - base <= offset - 1
            if (len > ulen - op) return false;
            // byte i of the element comes from source byte i mod offset (an overlapping copy repeats its period)
            const uint32_t sp = op - offset;
            uint32_t i0 = lane, i1 = lane + 32;                      // len <= 64: at most two bytes per lane
            uint32_t s0, s1;
            if (offset >= len) { s0 = i0; s1 = i1; }
            else if (offset >= 32) { s0 = i0 >= offset ? i0 - offset : i0; s1 = i1 >= offset ? i1 - offset : i1; }   // i < 64 <= 2 * offset
            else { s0 = i0 % offset; s1 = i1 % offset; }
            if (use_ring && offset <= kSnapRing - 64) {              // sources [op-offset, op) stay mirrored through this element's writes
                uint32_t b0 = 0, b1 = 0;
                if (i0 < len) b0 = ring_ld(ring_s, sp + s0);
                if (i1 < len) b1 = ring_ld(ring_s, sp + s1);
                if (i0 < len) { out[op + i0] = (uint8_t)b0; ring_st(ring_s, op + i0, b0); }
                if (i1 < len) { out[op + i1] = (uint8_t)b1; ring_st(ring_s, op + i1, b1); }
            } else {
                const uint8_t* from = out + sp;
                uint32_t b0 = 0, b1 = 0;
                if (i0 < len) b0 = from[s0];
                if (i1 < len) b1 = from[s1];
                if (i0 < len) { out[op + i0] = (uint8_t)b0; if (use_ring) ring_st(ring_s, op + i0, b0); }
                if (i1 < len) { out[op + i1] = (uint8_t)b1; if (use_ring) ring_st(ring_s, op + i1, b1); }
            }
            op += len;
        }
        __syncwarp();                                                // later elements read what this one wrote
    }
    produced = op;
    return op == ulen;
}

// Snappy raw-format ENCODER, bit-exact with butil::snappy::RawCompress (snappy.cc:875-956 Compress,
// :329-468 CompressFragment, :156-233 EmitLiteral/EmitCopy, snappy-internal.h:86-120 FindMatchLength):
// same hash (load32 * 0x1e35a7bd >> shift), same table size rule (256..16384 entries, >= fragment
// size), same skip heuristic (skip++ >> 5), same 15-byte input margin, same emit rules, 64 KiB
// fragments with a zeroed table each.  The probe chain is serial by construction (every table write
// feeds later probes): lane 0 walks it; match extension and literal/tag emission use the warp.
constexpr uint32_t kSnappyWarps = 8192;
constexpr uint32_t kSnappyBlock = 65536, kSnappyMaxTable = 16384;

__device__ __forceinline__ uint32_t ld32u(const uint8_t* p) {      // UNALIGNED_LOAD32
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
// number of leading bytes in which s1[] and s2[] agree, s2 bounded by s2_limit (FindMatchLength)
__device__ __forceinline__ uint32_t warp_find_match_length(const uint8_t* s1, const uint8_t* s2, const uint8_t* s2_limit, uint32_t lane) {
    const uint32_t maxn = (uint32_t)(s2_limit - s2);
    for (uint32_t base = 0; base < maxn; base += 32) {
        const uint32_t i = base + lane;
        const bool diff = i >= maxn || s1[i] != s2[i];
        const uint32_t m = __ballot_sync(0xffffffffu, diff);
        if (m) return base + (__ffs(m) - 1);
    }
    return maxn;
}
// tag bytes of a literal of `len` (EmitLiteral); returns their count
__device__ __forceinline__ uint32_t snappy_literal_tag(uint8_t* op, uint32_t len, bool write) {
    uint32_t n = len - 1;
    if (n < 60) { if (write) op[0] = (uint8_t)(n << 2); return 1; }
    uint32_t count = 0, v = n;
    while (v > 0) { if (write) op[1 + count] = (uint8_t)(v & 0xff); v >>= 8; count++; }
    if (write) op[0] = (uint8_t)((59 + count) << 2);
    return 1 + count;
}
// EmitCopy: tags for a copy of `len` at `offset`; returns their byte count
__device__ __forceinline__ uint32_t snappy_copy_tags(uint8_t* op, uint32_t offset, uint32_t len, bool write) {
    uint32_t w = 0;
    auto less64 = [&](uint32_t l) {
        if (l < 12 && offset < 2048) {
            if (write) { op[w] = (uint8_t)(1 + ((l - 4) << 2) + ((offset >> 8) << 5)); op[w + 1] = (uint8_t)(offset & 0xff); }
            w += 2;
        } else {
            if (write) { op[w] = (uint8_t)(2 + ((l - 1) << 2)); op[w + 1] = (uint8_t)(offset & 0xff); op[w + 2] = (uint8_t)(offset >> 8); }
            w += 3;
        }
    };
    while (len >= 68) { less64(64); len -= 64; }
    if (len > 64) { less64(60); len -= 60; }
    less64(len);
    return w;
}
__device__ __forceinline__ void warp_copy(uint8_t* dst, const uint8_t* src, uint32_t n, uint32_t lane);

// one fragment (<= 64 KiB); returns the compressed size.  `table` is this warp's hash table.
__device__ __noinline__ uint32_t warp_snappy_compress_fragment(const uint8_t* input, uint32_t input_size, uint8_t* out,
                                                               uint16_t* table, uint32_t lane) {
    uint32_t table_size = 256;
    while (table_size < kSnappyMaxTable && table_size < input_size) table_size <<= 1;
    for (uint32_t i = lane; i < table_size / 2; i += 32) reinterpret_cast<uint32_t*>(table)[i] = 0;
    __syncwarp();
    const int shift = 32 - (31 - __clz(table_size));
    uint32_t op = 0, ip = 0, next_emit = 0;
    const uint32_t ip_end = input_size;
    if (input_size >= 15) {
        const uint32_t ip_limit = input_size - 15;
        uint32_t next_hash = 0;
        ip = 1;
        if (lane == 0) next_hash = (ld32u(input + ip) * 0x1e35a7bdu) >> shift;
        for (;;) {
            // Step 1 (lane 0): scan forward for a 4-byte match
            uint32_t found = 0, candidate = 0;
            if (lane == 0) {
                uint32_t skip = 32, next_ip = ip;
                for (;;) {
                    ip = next_ip;
                    const uint32_t hash = next_hash;
                    const uint32_t step = skip++ >> 5;
                    next_ip = ip + step;
                    if (next_ip > ip_limit) { found = 0; break; }
                    next_hash = (ld32u(input + next_ip) * 0x1e35a7bdu) >> shift;
                    candidate = table[hash];
                    table[hash] = (uint16_t)ip;
                    if (ld32u(input + ip) == ld32u(input + candidate)) { found = 1; break; }
                }
            }
            found = __shfl_sync(0xffffffffu, found, 0);
            if (!found) break;                                   // goto emit_remainder
            ip = __shfl_sync(0xffffffffu, ip, 0); candidate = __shfl_sync(0xffffffffu, candidate, 0);
            // Step 2: the literal [next_emit, ip)
            {
                const uint32_t len = ip - next_emit;
                const uint32_t tl = snappy_literal_tag(out + op, len, lane == 0);
                warp_copy(out + op + tl, input + next_emit, len, lane);
                op += tl + len;
            }
            // Step 3: copies, as long as the position right after a copy matches again
            bool remainder = false;
            for (;;) {
                const uint32_t base_ip = ip;
                const uint32_t matched = 4 + warp_find_match_length(input + candidate + 4, input + ip + 4, input + ip_end, lane);
                ip += matched;
                op += snappy_copy_tags(out + op, base_ip - candidate, matched, lane == 0);
                next_emit = ip;
                if (ip >= ip_limit) { remainder = true; break; }
                uint32_t again = 0;
                if (lane == 0) {
                    const uint32_t prev_hash = (ld32u(input + ip - 1) * 0x1e35a7bdu) >> shift;
                    table[prev_hash] = (uint16_t)(ip - 1);
                    const uint32_t cur = ld32u(input + ip);
                    const uint32_t cur_hash = (cur * 0x1e35a7bdu) >> shift;
                    candidate = table[cur_hash];
                    const uint32_t cand_bytes = ld32u(input + candidate);
                    table[cur_hash] = (uint16_t)ip;
                    again = cur == cand_bytes;
                }
                again = __shfl_sync(0xffffffffu, again, 0);
                candidate = __shfl_sync(0xffffffffu, candidate, 0);
                if (!again) break;
            }
            if (remainder) break;
            if (lane == 0) next_hash = (ld32u(input + ip + 1) * 0x1e35a7bdu) >> shift;
            ++ip;
        }
    }
    // emit_remainder
    if (next_emit < ip_end) {
        const uint32_t len = ip_end - next_emit;
        const uint32_t tl = snappy_literal_tag(out + op, len, lane == 0);
        warp_copy(out + op + tl, input + next_emit, len, lane);
        op += tl + len;
    }
    __syncwarp();
    return op;
}
// whole buffer: varint32 length + fragments; returns the compressed size
__device__ __forceinline__ uint32_t warp_snappy_compress(const uint8_t* in, uint32_t n, uint8_t* out, uint16_t* table, uint32_t lane) {
    uint32_t op = 0;
    { uint32_t v = n; while (v >= 0x80) { if (lane == 0) out[op] = (uint8_t)(v | 0x80); v >>= 7; op++; } if (lane == 0) out[op] = (uint8_t)v; op++; }
    for (uint32_t pos = 0; pos < n; pos += kSnappyBlock) {
        const uint32_t len = min(kSnappyBlock, n - pos);
        op += warp_snappy_compress_fragment(in + pos, len, out + op, table, lane);
    }
    return op;
}

#ifndef B2_PACK_MIN_BLOCKS
#define B2_PACK_MIN_BLOCKS 6
#endif
// --- k_pack: one warp per message --------------------------------------------
__device__ __constant__ uint32_t c_crc_table[256];   // CRC-32C byte table (poly 0x82f63b78 reflected)

__device__ __forceinline__ uint32_t crc32c_bytes_serial(uint32_t l, const uint8_t* p, uint32_t n) {
    for (uint32_t i = 0; i < n; i++) l = c_crc_table[(l ^ p[i]) & 0xff] ^ (l >> 8);
    return l;
}

// CRC-32C as a warp-level primitive (butil::crc32c::Extend, src/butil/crc32c.cc:379-454, without
// the 0xffffffff pre/post inversion: this works on the raw register `l`).
// The CRC register is linear over GF(2): update(l, A||B) = ADV_|B|(update(l, A)) ^ update(0, B),
// where ADV_k advances the register over k zero bytes.  Lane i takes every 32nd aligned 16-byte
// block (one coalesced 512-byte row per warp load): R_i = ADV_512(R_i) ^ S16(block), S16 = the
// slice-by-16 table sum of the block's bytes.  The blocks are front-padded with virtual zero
// blocks (no-ops on a zero register) so that the last block sits in lane 31, the incoming
// register is XORed into the first four message bytes, a 5-level shuffle tree with
// ADV_16..ADV_256 folds the 32 lanes, and the <= 15 trailing bytes finish serially.
// Tables (built on the host): hot = T[16][256] (T[k][b] = byte b followed by k zero bytes) then
// A512[4][256]; tree = ADV_{16<<t}[4][256], t = 0..4.  `hot` may live in shared memory.
constexpr uint32_t kCrcHotWords = 20 * 256, kCrcTreeWords = 5 * 4 * 256;
struct CrcTabs { const uint32_t* hot; const uint32_t* tree; uint8_t* ring = nullptr; };   // + this warp's snappy ring (or null)
__device__ __forceinline__ uint32_t crc_adv4(const uint32_t* T, uint32_t x) {      // 4x256 byte-sliced operator
    return T[x & 0xff] ^ T[256 + ((x >> 8) & 0xff)] ^ T[512 + ((x >> 16) & 0xff)] ^ T[768 + (x >> 24)];
}
__device__ __forceinline__ uint32_t crc_s16(const uint32_t* T, const uint4& v) {
    uint32_t r = 0;
    #pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t w = j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w;
        r ^= T[(15 - 4 * j) * 256 + (w & 0xff)] ^ T[(14 - 4 * j) * 256 + ((w >> 8) & 0xff)] ^
             T[(13 - 4 * j) * 256 + ((w >> 16) & 0xff)] ^ T[(12 - 4 * j) * 256 + (w >> 24)];
    }
    return r;
}
__device__ __forceinline__ uint32_t warp_crc32c_update(uint32_t l, const uint8_t* p, uint32_t n, uint32_t lane, const CrcTabs& ct) {
    const uint32_t lead = (uint32_t)((uintptr_t)p & 15u);
    if (lead + n < 48) return crc32c_bytes_serial(l, p, n);          // (uniform across the warp)
    const uint4* a0 = reinterpret_cast<const uint4*>(p - lead);
    const uint32_t W = (lead + n) >> 4, tailn = (lead + n) & 15u;    // whole 16-byte blocks from a0
    const uint32_t off = (32u - (W & 31u)) & 31u, rows = (W + off) >> 5;
    // the incoming register lands on message bytes 0..3 = virtual bytes lead..lead+3, i.e. words k0, k0+1 of blocks 0/1
    const uint32_t k0 = lead >> 2, sh = 8 * (lead & 3u);
    const uint32_t x_lo = l << sh, x_hi = sh ? l >> (32 - sh) : 0u;
    uint32_t R = 0;
    for (uint32_t r0 = 0; r0 < rows; r0 += 4) {
        // four rows (2 KB of the message) are requested before the first is folded in: the loop is a chain of table look-ups, the loads
        // must not sit inside it
        uint4 pre[4];
        #pragma unroll
        for (int u = 0; u < 4; u++) {
            const int32_t v = (int32_t)((r0 + u) * 32 + lane) - (int32_t)off;
            pre[u] = make_uint4(0, 0, 0, 0);
            if (r0 + u < rows && v >= 0) pre[u] = __ldg(a0 + v);
        }
        #pragma unroll
        for (int u = 0; u < 4; u++) {
            if (r0 + u >= rows) break;
            const int32_t v = (int32_t)((r0 + u) * 32 + lane) - (int32_t)off;
            uint4 blk = pre[u];
            if (v >= 0 && v <= 1) {                                  // zero the bytes in front of the message, fold the register in
                uint32_t w[4] = { blk.x, blk.y, blk.z, blk.w };
                #pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t gw = 4u * (uint32_t)v + k;        // word index over blocks 0 and 1
                    if (gw < k0) w[k] = 0;
                    else if (gw == k0) w[k] = (w[k] & (0xffffffffu << sh)) ^ x_lo;
                    else if (gw == k0 + 1) w[k] ^= x_hi;
                }
                blk = make_uint4(w[0], w[1], w[2], w[3]);
            }
            R = crc_adv4(ct.hot + 16 * 256, R) ^ crc_s16(ct.hot, blk);
        }
    }
    #pragma unroll
    for (int t = 0; t < 5; t++) {
        const uint32_t d = 1u << t;
        const uint32_t left = __shfl_up_sync(0xffffffffu, R, d);
        if ((lane & (2 * d - 1)) == 2 * d - 1) R = crc_adv4(ct.tree + t * 1024, left) ^ R;
    }
    R = __shfl_sync(0xffffffffu, R, 31);
    if (tailn == 0) return R;
    // the <= 15 trailing bytes, in parallel: update(R, tail) = update(R, tailn zero bytes) ^ update(0, tail);
    // a byte followed by k zero bytes is one lookup in T[k] (the slice tables), the register's byte j acts as data byte j
    const uint8_t* tp = reinterpret_cast<const uint8_t*>(a0 + W);
    uint32_t c = 0;
    if (lane < tailn) c = ct.hot[(tailn - 1 - lane) * 256 + tp[lane]];
    else if (lane >= 16 && lane < 20) {
        const uint32_t j = lane - 16, rb = (R >> (8 * j)) & 0xffu;
        if (j < tailn) c = ct.hot[(tailn - 1 - j) * 256 + rb];
    }
    if (lane == 20 && tailn < 4) c = R >> (8 * tailn);               // register bytes the short tail did not consume
    #pragma unroll
    for (int d = 16; d >= 1; d >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, d);
    return c;
}
// stage the hot tables into shared memory (all threads of the block cooperate)
__device__ __forceinline__ void crc_tabs_to_smem(uint32_t* s_hot, const uint32_t* g_hot) {
    for (uint32_t i = threadIdx.x; i < kCrcHotWords; i += blockDim.x) s_hot[i] = g_hot[i];
    __syncthreads();
}

// byte j of the base-128 varint of v (n bytes long)
__device__ __forceinline__ uint8_t varint_byte(uint64_t v, uint32_t j, uint32_t n) {
    return (uint8_t)(((v >> (7 * j)) & 0x7f) | (j + 1 < n ? 0x80 : 0));
}

// serial emitters used by the (rare) error-reply path
__device__ __forceinline__ uint8_t* put_str(uint8_t* p, const char* s, uint32_t n) { for (uint32_t i = 0; i < n; i++) p[i] = (uint8_t)s[i]; return p + n; }
__device__ __forceinline__ uint8_t* put_bytes(uint8_t* p, const uint8_t* s, uint32_t n) { for (uint32_t i = 0; i < n; i++) p[i] = s[i]; return p + n; }

__device__ __noinline__ uint32_t pack_error_reply(uint8_t* out, const DevConfig& C, const DevMethod* ms, const b2_msg_desc& d,
                                                  const MsgAux& a, const uint8_t* frame) {
    const uint32_t tl = error_text_len(C, ms, d, a, frame);
    const uint32_t req_size = d.body_size - d.meta_size;
    const uint32_t ml = response_meta_len(d.error_code, tl, 0, d.correlation_id, 0, 0, a.cks_len);
    uint8_t* p = out;
    p = put_str(p, "PRPC", 4); p = put_be32(p, ml); p = put_be32(p, ml);
    const uint32_t rm = 1 + varint_len((uint64_t)(int64_t)d.error_code) + 1 + varint_len(tl) + tl;
    *p++ = 0x12; p = put_varint(p, rm);
    *p++ = 0x08; p = put_varint(p, (uint64_t)(int64_t)d.error_code);
    *p++ = 0x12; p = put_varint(p, tl);
    if (C.identity_len) { *p++ = '['; p = put_str(p, C.identity, C.identity_len); *p++ = ']'; }
    *p++ = '['; *p++ = 'E'; p = put_dec(p, (uint32_t)d.error_code); *p++ = ']';
    switch (a.err_kind) {
    case kErrAttachment:
        p = put_str(p, "attachment_size=", 16); p = put_dec_i32(p, d.attachment_size);
        p = put_str(p, " is larger than request_size=", 29); p = put_dec(p, req_size); break;
    case kErrNoService:
        p = put_str(p, "Fail to find service=", 21); p = put_bytes(p, frame + a.svc_off, strnlen_dev(frame + a.svc_off, a.svc_len)); break;
    case kErrNoMethod:
        p = put_str(p, "Fail to find method=", 20); p = put_bytes(p, frame + a.svc_off, strnlen_dev(frame + a.svc_off, a.svc_len));
        *p++ = '/'; p = put_bytes(p, frame + a.mth_off, strnlen_dev(frame + a.mth_off, a.mth_len)); break;
    case kErrParseRequest: {
        const DevMethod& m = ms[d.method_idx];
        p = put_str(p, "Fail to parse request=", 22); p = put_str(p, m.request_type, m.request_type_len);
        p = put_str(p, ", ContentType=", 14); p = put_str(p, "pb", 2);
        p = put_str(p, ", CompressType=", 15);
        { const int32_t t = d.compress_type; p = put_str(p, t == 0 ? "none" : t == 1 ? "snappy" : t == 2 ? "gzip" : t == 3 ? "zlib" : "unknown", cstr_len_compress(t)); }
        p = put_str(p, ", ChecksumType=", 15);
        { const int32_t t = d.checksum_type; p = put_str(p, t == 0 ? "none" : t == 1 ? "crc32c" : "unknown", cstr_len_checksum(t)); }
        p = put_str(p, ", request_size=", 15); p = put_dec(p, req_size); break; }
    }
    *p++ = 0x18; *p++ = 0x00;                                  // compress_type = 0
    *p++ = 0x20; p = put_varint(p, (uint64_t)d.correlation_id);
    *p++ = 0x50; *p++ = 0x00;                                  // content_type = PB
    *p++ = 0x58; *p++ = 0x00;                                  // checksum_type = 0
    *p++ = 0x62; p = put_varint(p, a.cks_len); p = put_bytes(p, frame + a.cks_off, a.cks_len);   // request's checksum_value travels back
    return (uint32_t)(p - out);
}

// copy n bytes src -> dst with the whole warp; fast path when both share (mod 16) alignment
__device__ __forceinline__ void warp_copy(uint8_t* dst, const uint8_t* src, uint32_t n, uint32_t lane) {
    if ((((uintptr_t)dst ^ (uintptr_t)src) & 15u) == 0) {
        const uint32_t head = min(n, (uint32_t)((16u - ((uintptr_t)dst & 15u)) & 15u));
        if (lane < head) dst[lane] = src[lane];
        const uint32_t nv = (n - head) >> 4;
        const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
        uint4* d4 = reinterpret_cast<uint4*>(dst + head);
        uint32_t i = lane;
        for (; i + 96 < nv; i += 128) {                        // 4 independent 16 B loads in flight per lane
            const uint4 a = __ldg(s4 + i), b = __ldg(s4 + i + 32), c = __ldg(s4 + i + 64), d = __ldg(s4 + i + 96);
            d4[i] = a; d4[i + 32] = b; d4[i + 64] = c; d4[i + 96] = d;
        }
        for (; i + 32 < nv; i += 64) {                        // 2 loads in flight per lane (1 KB payloads)
            const uint4 a = __ldg(s4 + i), b = __ldg(s4 + i + 32);
            d4[i] = a; d4[i + 32] = b;
        }
        for (; i < nv; i += 32) d4[i] = __ldg(s4 + i);
        const uint32_t done = head + (nv << 4);
        if (lane < n - done) dst[done + lane] = src[done + lane];
    } else {
        uint32_t i = lane;
        for (; i + 224 < n; i += 256) {                        // 8 independent byte loads in flight per lane
            uint8_t v[8];
            #pragma unroll
            for (int k = 0; k < 8; k++) v[k] = src[i + 32 * k];
            #pragma unroll
            for (int k = 0; k < 8; k++) dst[i + 32 * k] = v[k];
        }
        for (; i < n; i += 32) dst[i] = src[i];
    }
}

// Lane-parallel reply prefix: lane j produces byte j (+32, +64 ...) of
//   "PRPC" be32(body) be32(meta) | 12 02 08 00 | 18 00 | 20 cid | [28 att] | 50 00 | 58 ck | 62 len cks | 0a len
// == PackRpcHeader + the RpcMeta of SendRpcResponse (baidu_rpc_protocol.cpp:75-81,339-349) + the
// EchoResponse field header.  `out` may point to shared or global memory.
__device__ __forceinline__ void write_echo_prefix(uint8_t* out, uint32_t lane, int64_t correlation_id, uint32_t att_len,
                                                  int32_t r_cks_type, uint32_t cks_len, uint32_t crc_be, const uint8_t* req_cks,
                                                  uint32_t msg_len, uint32_t ml, uint32_t vl, uint32_t prefix,
                                                  int32_t compress_type = 0, uint32_t compressed_body = 0) {
    const uint32_t cid_n = varint_len((uint64_t)correlation_id);
    const uint32_t att_n = att_len ? 1 + varint_len(att_len) : 0;
    const uint32_t o_cid = 12 + 6;                 // after 12 02 08 00 18 00
    const uint32_t o_att = o_cid + 1 + cid_n;
    const uint32_t o_ct = o_att + att_n;           // 50 00 58 xx 62
    const uint32_t o_ckl = o_ct + 5;               // varint(cks_len)
    const uint32_t ckl_n = varint_len(cks_len);
    const uint32_t o_ckv = o_ckl + ckl_n;
    const uint32_t o_pb = o_ckv + cks_len;         // == 12 + ml
    // compressed reply: the body is the compressed EchoResponse (no pb field header here, prefix == 12 + ml)
    const uint32_t total_body = compress_type ? ml + compressed_body + att_len : ml + 1 + vl + msg_len + att_len;
    for (uint32_t j = lane; j < prefix; j += 32) {
        uint8_t b;
        if (j < 4) b = (uint8_t)(kMagicPRPC >> (8 * j));
        else if (j < 8) b = (uint8_t)(total_body >> (8 * (7 - j)));
        else if (j < 12) b = (uint8_t)(ml >> (8 * (11 - j)));
        else if (j < o_cid) { const uint32_t k = j - 12; b = (k == 0) ? 0x12 : (k == 1) ? 0x02 : (k == 2) ? 0x08 : (k == 4) ? 0x18 : (k == 5) ? (uint8_t)compress_type : 0x00; }
        else if (j == o_cid) b = 0x20;
        else if (j < o_att) b = varint_byte((uint64_t)correlation_id, j - o_cid - 1, cid_n);
        else if (j < o_ct) b = (j == o_att) ? 0x28 : varint_byte(att_len, j - o_att - 1, att_n - 1);
        else if (j < o_ckl) { const uint32_t k = j - o_ct; b = (k == 0) ? 0x50 : (k == 2) ? 0x58 : (k == 3) ? (uint8_t)r_cks_type : (k == 4) ? 0x62 : 0x00; }
        else if (j < o_ckv) b = varint_byte(cks_len, j - o_ckl, ckl_n);
        else if (j < o_pb) b = (r_cks_type == B2_CHECKSUM_TYPE_CRC32C) ? (uint8_t)(crc_be >> (8 * (3 - (j - o_ckv)))) : req_cks[j - o_ckv];
        else if (j == o_pb) b = 0x0a;
        else b = varint_byte(msg_len, j - o_pb - 1, vl);
        out[j] = b;
    }
}

struct CrcTabs;
__device__ __forceinline__ void pack_one(const BatchPtrs& B, const DevConfig& C, uint32_t i, uint32_t lane, const CrcTabs& ct);

// persistent: a fixed grid (multiple of the SM count); every warp strides over the messages
__global__ void __launch_bounds__(256, B2_PACK_MIN_BLOCKS) k_pack(BatchPtrs B, DevConfig C) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t n_msgs = B.totals[0];
    if (B.totals[2] & 3u) return;
    finalize_runs(B, C);
    __shared__ uint32_t s_hot[kCrcHotWords];
    crc_tabs_to_smem(s_hot, B.crc_adv);
    CrcTabs ct; ct.hot = s_hot; ct.tree = B.crc_adv + kCrcHotWords;
    const uint32_t n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_msgs; i += n_warps) pack_one(B, C, i, lane, ct);
}

__device__ __forceinline__ void pack_one(const BatchPtrs& B, const DevConfig& C, uint32_t i, uint32_t lane, const CrcTabs& ct) {
    const uint32_t bi = i / (kScanBlock * kScanItems);
    const uint32_t slot_off = C.fused ? B.slot[i] : B.slot[i] + B.scan_tmp[bi];
    const b2_msg_desc d = B.msgs[i];
    __syncwarp();                                                   // (lane 0 stores resp_off / resp_len / status into msgs[i] further down: every lane has its copy first)
    // nothing to produce — except for a client-side response that parsed to an empty message and carries a CRC32C checksum: Crc32cVerify comes
    // before the parse in DeserializeRpcMessage, a wrong checksum fails the call whatever the message holds
    const bool empty_to_verify = d.status == B2_MSG_RESPONSE && d.error_code == 0 && d.checksum_type == B2_CHECKSUM_TYPE_CRC32C;
    if (d.resp_len == 0 && !empty_to_verify) { if (lane == 0 && d.status != B2_MSG_RESPONSE) B.msgs[i].resp_off = slot_off; return; }
    const MsgAux a = B.aux[i];
    const uint8_t* frame = B.bytes + d.frame_off;
    if (d.status == B2_MSG_REPLAY) {
        // PackRpcRequest replaying a sampled request (baidu_rpc_protocol.cpp:1067-1075 + :1080-1131): header, RpcMeta{request{service_name,
        // method_name}, compress_type, correlation_id, [attachment_size], content_type}, then the sampled bytes (body + attachment) as they were
        uint8_t* out = B.resp + slot_off;
        const uint32_t ml = replay_meta_len(a.svc_len, a.mth_len, d.compress_type, d.correlation_id, a.att_len);
        if (lane == 0) {
            uint8_t* p = out;
            p[0] = 'P'; p[1] = 'R'; p[2] = 'P'; p[3] = 'C'; put_be32(p + 4, ml + a.msg_len); put_be32(p + 8, ml); p += 12;
            const uint32_t rl = 1 + varint_len(a.svc_len) + a.svc_len + 1 + varint_len(a.mth_len) + a.mth_len;
            *p++ = 0x0a; p = put_varint(p, rl);
            *p++ = 0x0a; p = put_varint(p, a.svc_len); for (uint32_t k = 0; k < a.svc_len; k++) *p++ = frame[a.svc_off + k];
            *p++ = 0x12; p = put_varint(p, a.mth_len); for (uint32_t k = 0; k < a.mth_len; k++) *p++ = frame[a.mth_off + k];
            *p++ = 0x18; p = put_varint(p, (uint64_t)(long long)d.compress_type);
            *p++ = 0x20; p = put_varint(p, (uint64_t)d.correlation_id);
            if (a.att_len) { *p++ = 0x28; p = put_varint(p, a.att_len); }
            *p++ = 0x50; *p++ = 0x00;
            B.msgs[i].resp_off = slot_off;
        }
        warp_copy(out + 12 + ml, frame + 12 + d.meta_size, a.msg_len, lane);
        return;
    }
    if (d.status == B2_MSG_STREAM_FRAME) {
        // the application-level SnappyDecompress of a streaming DATA frame's payload
        uint32_t produced = 0;
        const bool ok = warp_snappy_decode(frame + 12 + d.meta_size, a.att_off, B.resp + slot_off, a.msg_len, lane, produced, ct.ring);
        if (lane == 0) {
            if (ok) { B.msgs[i].resp_off = slot_off; B.msgs[i].resp_len = produced; }
            else { B.msgs[i].resp_off = slot_off; B.msgs[i].resp_len = 0; B.msgs[i].error_code = B2_EREQUEST; }
        }
        return;
    }
    if (d.status == B2_MSG_RESPONSE || d.status == B2_MSG_RESPONSE_UNZ) {
        // client side: DeserializeRpcMessage of the response body = checksum verify, then (snappy ->) parse
        bool ok = true;
        const uint8_t* body = frame + 12 + d.meta_size; const uint32_t body_len = a.att_off;
        if (d.checksum_type == B2_CHECKSUM_TYPE_CRC32C) {
            const uint32_t crc = warp_crc32c_update(0xffffffffu, body, body_len, lane, ct) ^ 0xffffffffu;
            ok = crc == crc32c_unmask(load_be32(frame + a.cks_off));
        }
        uint32_t off = d.resp_off, len = d.resp_len;
        if (ok && d.status == B2_MSG_RESPONSE_UNZ) {
            uint32_t produced = 0;
            if (d.compress_type == B2_COMPRESS_TYPE_SNAPPY) ok = warp_snappy_decode(body, body_len, B.resp + slot_off, a.msg_len, lane, produced, ct.ring);
            else {
                if (lane == 0) { bool big; produced = gz_input_stream<true>(body, body_len, d.compress_type, B.resp + slot_off, a.msg_len, &big); }
                produced = __shfl_sync(0xffffffffu, produced, 0);
            }
            Span msg; msg.off = 0; msg.len = 0;
            if (ok) ok = decode_echo_request(B.resp + slot_off, produced, msg);
            off = slot_off + msg.off; len = msg.len;
        }
        if (lane == 0) {
            if (ok) { B.msgs[i].resp_off = off; B.msgs[i].resp_len = len; }
            else { B.msgs[i].status = B2_MSG_RESPONSE; B.msgs[i].error_code = B2_EREQUEST; B.msgs[i].resp_off = 0; B.msgs[i].resp_len = 0; }
        }
        return;
    }
    const DevMethod* mp = d.method_idx >= 0 ? B.methods + d.method_idx : nullptr;
    uint16_t status = d.status;
    if (status == B2_MSG_ECHOED && d.checksum_type == B2_CHECKSUM_TYPE_CRC32C) {
        // Crc32cVerify (policy/crc32c_checksum.cpp:44-61) over body_wo_att
        const uint32_t req_size = d.body_size - d.meta_size;
        int64_t bwo = (int64_t)req_size - (int64_t)d.attachment_size; if (bwo > (int64_t)req_size) bwo = req_size;
        const uint32_t crc = warp_crc32c_update(0xffffffffu, frame + 12 + d.meta_size, (uint32_t)bwo, lane, ct) ^ 0xffffffffu;
        if (crc != crc32c_unmask(load_be32(frame + a.cks_off))) status = B2_MSG_ERROR_REPLIED;
    }
    const uint8_t* msg_src = frame + a.msg_off;
    uint32_t msg_len = a.msg_len;
    if (status == B2_MSG_ECHOED && d.compress_type == B2_COMPRESS_TYPE_SNAPPY) {
        // SnappyDecompress (policy/snappy_compress.cpp:51-70) into the scratch slot, then ParseFromZeroCopyStream
        const uint32_t req_size = d.body_size - d.meta_size;
        int64_t bwo = (int64_t)req_size - (int64_t)d.attachment_size; if (bwo > (int64_t)req_size) bwo = req_size;
        uint8_t* scratch = B.unz + slot_off;
        uint32_t produced = 0;
        bool ok = warp_snappy_decode(frame + 12 + d.meta_size, (uint32_t)bwo, scratch, a.msg_len, lane, produced, ct.ring);
        Span msg; msg.off = 0; msg.len = 0;
        if (ok) ok = decode_echo_request(scratch, produced, msg);
        if (!ok) status = B2_MSG_ERROR_REPLIED;
        else { msg_src = scratch + msg.off; msg_len = msg.len; }
    }
    if (status == B2_MSG_ECHOED && (d.compress_type == B2_COMPRESS_TYPE_GZIP || d.compress_type == B2_COMPRESS_TYPE_ZLIB)) {
        // GzipDecompress / ZlibDecompress (policy/gzip_compress.cpp:75-89): lane 0 walks the DEFLATE stream into the scratch slot; the parser
        // gets what the GzipInputStream would have handed it (a corrupt stream is end-of-input to it)
        const uint32_t req_size = d.body_size - d.meta_size;
        int64_t bwo = (int64_t)req_size - (int64_t)d.attachment_size; if (bwo > (int64_t)req_size) bwo = req_size;
        uint8_t* scratch = B.unz + slot_off;
        uint32_t produced = 0;
        if (lane == 0) { bool big; produced = gz_input_stream<true>(frame + 12 + d.meta_size, (uint32_t)bwo, d.compress_type, scratch, a.msg_len, &big); }
        produced = __shfl_sync(0xffffffffu, produced, 0);
        Span msg; msg.off = 0; msg.len = 0;
        if (!decode_echo_request(scratch, produced, msg)) status = B2_MSG_ERROR_REPLIED;
        else { msg_src = scratch + msg.off; msg_len = msg.len; }
    }
    if (status == B2_MSG_ERROR_REPLIED) {
        uint32_t n = 0;
        if (lane == 0) {
            b2_msg_desc e = d; MsgAux ea = a;
            if (d.status == B2_MSG_ECHOED) { e.error_code = B2_EREQUEST; ea.err_kind = kErrParseRequest; }
            n = pack_error_reply(B.resp + slot_off, C, B.methods, e, ea, frame);
            B.msgs[i].resp_off = slot_off; B.msgs[i].resp_len = n;
            if (C.by_ref) B.refs[i] = make_uint4(0, 0, 0, 0);          // the whole (error) reply is materialised
            if (d.status == B2_MSG_ECHOED) { B.msgs[i].status = B2_MSG_ERROR_REPLIED; B.msgs[i].error_code = B2_EREQUEST; }
        }
        return;
    }
    // ---- OK echo reply: SendRpcResponse with append_body -----------------------------------
    const int32_t r_cks_type = mp->response_checksum_type;
    const int32_t r_compress = mp->response_compress_type;
    const uint32_t cks_len = r_cks_type == B2_CHECKSUM_TYPE_CRC32C ? 4u : a.cks_len;
    const uint32_t ml = response_meta_len(0, 0, r_compress, d.correlation_id, a.att_len, r_cks_type, cks_len);
    const uint32_t vl = varint_len(msg_len);
    uint8_t* out = B.resp + slot_off + a.pad;
    if (C.by_ref && B.refs[i].x != 0) {
        // B2_RESP_BY_REF (a CRC-verified request served by the latency path): the slot holds the prefix only
        const uint32_t prefix = 12 + ml + 1 + vl;
        write_echo_prefix(out, lane, d.correlation_id, a.att_len, r_cks_type, cks_len, 0, frame + a.cks_off, msg_len, ml, vl, prefix);
        if (lane == 0) B.msgs[i].resp_off = slot_off;
        return;
    }
    if (r_compress == B2_COMPRESS_TYPE_SNAPPY) {
        // SnappyCompress (policy/snappy_compress.cpp:28-49): serialize the EchoResponse, then compress it
        uint8_t* pb = B.unz + (size_t)B.max_resp + slot_off;
        const uint32_t pb_len = 1 + vl + msg_len;
        if (lane == 0) { pb[0] = 0x0a; put_varint(pb + 1, msg_len); }
        warp_copy(pb + 1 + vl, msg_src, msg_len, lane);
        __syncwarp();
        const uint32_t warp_id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
        uint16_t* table = B.snappy_tab + (size_t)(warp_id % kSnappyWarps) * kSnappyMaxTable;
        const uint32_t prefix = 12 + ml;
        const uint32_t clen = warp_snappy_compress(pb, pb_len, out + prefix, table, lane);
        __syncwarp();
        uint32_t crc_be = 0;
        if (r_cks_type == B2_CHECKSUM_TYPE_CRC32C)
            crc_be = crc32c_mask(warp_crc32c_update(0xffffffffu, out + prefix, clen, lane, ct) ^ 0xffffffffu);
        write_echo_prefix(out, lane, d.correlation_id, a.att_len, r_cks_type, cks_len, crc_be, frame + a.cks_off, msg_len, ml, vl, prefix,
                          r_compress, clen);
        if (a.att_len) warp_copy(out + prefix + clen, frame + a.att_off, a.att_len, lane);
        if (lane == 0) { B.msgs[i].resp_off = slot_off + a.pad; B.msgs[i].resp_len = prefix + clen + a.att_len; }
        return;
    }
    const uint32_t prefix = 12 + ml + 1 + vl;
    const uint32_t resp_len = prefix + msg_len + a.att_len;
    uint32_t crc_be = 0;
    if (r_cks_type == B2_CHECKSUM_TYPE_CRC32C) {
        // Crc32cCompute (policy/crc32c_checksum.cpp:28-42) over the serialized EchoResponse
        uint32_t l = 0xffffffffu;
        uint8_t hdr[6]; hdr[0] = 0x0a; uint8_t* e = put_varint(hdr + 1, msg_len);
        l = crc32c_bytes_serial(l, hdr, (uint32_t)(e - hdr));
        l = warp_crc32c_update(l, msg_src, msg_len, lane, ct);
        crc_be = crc32c_mask(l ^ 0xffffffffu);
    }
    write_echo_prefix(out, lane, d.correlation_id, a.att_len, r_cks_type, cks_len, crc_be, frame + a.cks_off, msg_len, ml, vl, prefix);
    // payload: message bytes (+ attachment when it directly follows them, the normal layout)
    if (a.att_len && d.compress_type == B2_COMPRESS_TYPE_NONE && a.att_off == a.msg_off + a.msg_len) {
        warp_copy(out + prefix, msg_src, msg_len + a.att_len, lane);
    } else {
        warp_copy(out + prefix, msg_src, msg_len, lane);
        if (a.att_len) warp_copy(out + prefix + msg_len, frame + a.att_off, a.att_len, lane);
    }
    if (lane == 0) { B.msgs[i].resp_off = slot_off + a.pad; B.msgs[i].resp_len = resp_len; }
}


// --- k_pack_tma: the bandwidth path -------------------------------------------
// OK echo replies without CRC work are staged through shared memory with the bulk
// async-copy engine (TMA, cp.async.bulk): every warp owns two staging buffers; per
// round it takes kPackGroup consecutive messages, pulls their metadata with one
// coalesced load, issues one bulk load per payload (all in flight together, completion
// on an mbarrier), writes the reply prefixes into the same staging image while the
// payloads fly, then pushes every reply frame out with one bulk store.  Because the slot
// layout keeps (dst mod 16) == (src mod 16), the 16-byte aligned interior of payload and
// frame moves with TMA and only <= 15 head/tail bytes per side move with byte accesses.
// Everything else (error replies, CRC32C, replies larger than a staging buffer, split
// attachments) goes through pack_one.
#ifndef B2_PACK_WARPS
#define B2_PACK_WARPS 8
#endif
constexpr uint32_t kPackWarps = B2_PACK_WARPS;
#ifndef B2_PACK_GROUP
#define B2_PACK_GROUP 8
#endif
#ifndef B2_STAGE_BYTES
#define B2_STAGE_BYTES 9216
#endif
constexpr uint32_t kPackGroup = B2_PACK_GROUP;    // messages per warp round (one lane each), power of two: replies of 1 KB and more
constexpr uint32_t kPackGroupSmall = 32;          // ... and when the average request is small (more messages per barrier round)
constexpr uint32_t kStageBytes = B2_STAGE_BYTES;  // per buffer, two buffers per warp
struct PackWarpSmem {
    alignas(128) uint8_t stage[2][kStageBytes];
    alignas(8) unsigned long long mbar[2];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void* sdst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
// L2 prefetch of a byte range (16-byte aligned address and size): the DRAM reads start now, the later bulk load finds the lines in L2
__device__ __forceinline__ void bulk_prefetch_l2(const void* gsrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// Pure data movement: per message two TMA bulk loads (the pre-built head record and the
// 16-byte aligned remainder of the payload) into one staging slot and one TMA bulk store of
// the whole slot.  Lane l of a warp owns message base+l of the round; two staging buffers per
// warp keep one round's stores draining while the next round's loads are in flight.
template <uint32_t kGroup>
__global__ void __launch_bounds__(kPackWarps * 32, 1) k_pack_tma(BatchPtrs B, DevConfig C) {
    extern __shared__ __align__(128) uint8_t pack_smem_raw[];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    PackWarpSmem& S = reinterpret_cast<PackWarpSmem*>(pack_smem_raw)[wid];
    const uint32_t n_msgs = B.totals[0];
    if (B.totals[2] & 3u) return;
    if (lane == 0) {
        mbar_init(&S.mbar[0], 1); mbar_init(&S.mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const uint32_t stride = gridDim.x * kPackWarps * kGroup;
    uint32_t it = 0, phase0 = 0, phase1 = 0;        // mbarrier phases advance only in rounds that arm them
    PackJob job; job.fast = 0; job.slot_len = 0; job.head_len = 0; job.bulk_len = 0; job.src_off = 0; job.pad = 0;
    uint32_t slot_off = 0;
    uint32_t base = (blockIdx.x * kPackWarps + wid) * kGroup;
    auto fetch = [&](uint32_t bse, PackJob& j, uint32_t& so) {
        const uint32_t i = bse + lane;
        j.fast = 0; j.slot_len = 0;
        if (lane < kGroup && i < n_msgs) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(B.jobs + i));
            j = *reinterpret_cast<const PackJob*>(&v);
            so = B.slot[i] + B.scan_tmp[i / (kScanBlock * kScanItems)];
        }
    };
    // one staging round: arm the buffer's mbarrier, run `issue` (bulk loads), wait for the bytes
    auto begin_round = [&](uint32_t b) { bulk_wait_read<1>(); __syncwarp(); };   // stores that last read buffer b drained
    auto wait_round = [&](uint32_t b) { mbar_wait(&S.mbar[b], (b ? phase1 : phase0) & 1u); if (b) phase1++; else phase0++; };
    if (base < n_msgs) fetch(base, job, slot_off);
    for (; base < n_msgs; base += stride) {
        // software pipeline: request the next group's jobs now, use them next iteration
        PackJob njob; uint32_t nslot = 0;
        njob.fast = 0; njob.slot_len = 0; njob.head_len = 0; njob.bulk_len = 0; njob.src_off = 0; njob.pad = 0;
        if (base + stride < n_msgs) fetch(base + stride, njob, nslot);
        uint32_t pending = __ballot_sync(0xffffffffu, job.fast != 0);      // (jobs that are not fast belong to k_pack_slow)
        while (pending) {
            const uint32_t b = it & 1; it++;
            uint8_t* stage = S.stage[b];
            const uint32_t first = __ffs(pending) - 1;
            const uint32_t first_len = __shfl_sync(0xffffffffu, job.slot_len, first);
            if (first_len > kStageBytes) {
                // ---- a reply larger than a staging buffer: the warp streams it in chunks.  The slot image is
                // [head record | payload bulk]; chunk boundaries are multiples of 16, so every piece is a legal
                // bulk copy.  Lane 0 drives; two buffers alternate so a chunk's store overlaps the next load.
                const uint32_t hl = __shfl_sync(0xffffffffu, (uint32_t)job.head_len, first);
                const uint32_t so = __shfl_sync(0xffffffffu, slot_off, first);
                const uint32_t src = __shfl_sync(0xffffffffu, job.src_off, first);
                const uint32_t pad = __shfl_sync(0xffffffffu, (uint32_t)job.pad, first);
                const uint8_t* head = B.heads + (size_t)(base + first) * kHeadBytes;
                uint32_t bb = b;
                for (uint32_t c0 = 0; c0 < first_len; c0 += kStageBytes) {
                    const uint32_t c1 = min(c0 + kStageBytes, first_len);
                    if (c0) { bb = it & 1; it++; }
                    uint8_t* st = S.stage[bb];
                    begin_round(bb);
                    if (lane == 0) {
                        mbar_arrive_expect_tx(&S.mbar[bb], c1 - c0);
                        uint32_t at = c0;
                        if (at < hl) { const uint32_t e = min(hl, c1); bulk_g2s(st, head + at, e - at, &S.mbar[bb]); at = e; }
                        if (at < c1) bulk_g2s(st + (at - c0), B.bytes + src + (at - hl), c1 - at, &S.mbar[bb]);
                    }
                    wait_round(bb);
                    if (lane == 0) bulk_s2g(B.resp + so + c0, st, c1 - c0);
                    bulk_commit();
                }
                if (lane == 0) B.msgs[base + first].resp_off = so + pad;
                pending &= ~(1u << first);
                continue;
            }
            // ---- staging layout: the pending jobs, in lane order, as long as they fit the buffer
            const bool mine = (pending >> lane) & 1u;
            uint32_t need = mine ? job.slot_len : 0, incl = need;
            #pragma unroll
            for (int d = 1; d < (int)kGroup; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (uint32_t)d) incl += y; }
            const bool take = mine && incl <= kStageBytes;
            const uint32_t soff = incl - need;
            uint32_t tx = take ? (uint32_t)job.head_len + job.bulk_len : 0;
            #pragma unroll
            for (int d = 1; d < (int)kGroup; d <<= 1) tx += __shfl_xor_sync(0xffffffffu, tx, d);
            tx = __shfl_sync(0xffffffffu, tx, 0);
            begin_round(b);
            if (lane == 0) mbar_arrive_expect_tx(&S.mbar[b], tx);
            __syncwarp();
            if (take) {
                bulk_g2s(stage + soff, B.heads + (size_t)(base + lane) * kHeadBytes, job.head_len, &S.mbar[b]);
                if (job.bulk_len) bulk_g2s(stage + soff + job.head_len, B.bytes + job.src_off, job.bulk_len, &S.mbar[b]);
            }
            wait_round(b);
            const uint32_t took = __ballot_sync(0xffffffffu, take);
            if (kGroup > 8) {
                // small replies: the slots of consecutive messages are adjacent in resp, and so are their images in the staging
                // buffer when the taken lanes form one unbroken range — then ONE bulk store moves the whole round
                const uint32_t lo = __ffs(took) - 1, span = took >> lo;
                const bool contiguous = took && (span & (span + 1)) == 0;          // took == 0..0 1..1 0..0
                uint32_t total = take ? job.slot_len : 0;
                #pragma unroll
                for (int d = 1; d < 32; d <<= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
                // (adjacency in resp also needs every taken message's slot to follow its left neighbour's: true for consecutive messages)
                if (contiguous) { if (lane == lo) bulk_s2g(B.resp + slot_off, stage + soff, total); }
                else if (take) bulk_s2g(B.resp + slot_off, stage + soff, job.slot_len);
                if (take) B.msgs[base + lane].resp_off = slot_off + job.pad;
            } else if (take) {
                bulk_s2g(B.resp + slot_off, stage + soff, job.slot_len);
                B.msgs[base + lane].resp_off = slot_off + job.pad;
            }
            bulk_commit();
            pending &= ~took;
        }
        job = njob; slot_off = nslot;
    }
    bulk_wait<0>();
}


// --- k_fused: decode + echo + pack in ONE pass over the bytes ------------------------------------------------------------
// One warp per live tile (the frames that START in the tile, as k_resolve verified them).  The tile's byte range is pulled
// into shared memory with one TMA bulk load; the warp finds the frame starts (the offsets k_tile_walk kept, or a walk over
// the shared-memory copy), decodes one message per lane straight from shared memory, and writes each OK echo's reply prefix
// IN PLACE, right in front of the payload it answers: the reply to the request at batch offset o lives at the same offset
// of the resp region (a reply is never longer than its request there: same payload, shorter meta), so the patched image
// of the whole tile goes back out with ONE TMA bulk store — no head records, no slot scan, no per-message copies, every
// byte read once and written once.  Replies that cannot be built that way (errors, CRC-carrying or compressed bodies,
// client-side and stream outputs) get a slot in the overflow area behind the batch-shaped part of resp and are served by
// k_pack_slow.  A tile larger than the staging buffer (big frames) decodes from 160-byte rows and streams its range through
// the buffer in chunks, patching the prefixes that fall into each chunk.
#ifndef B2_FUSED_BUF
#define B2_FUSED_BUF 10240
#endif
// (16 x ~13.5 KB leave ~12 KB of the SM's shared memory to k_resolve of the next batch, which runs beside this kernel)
#ifndef B2_FUSED_WARPS
#define B2_FUSED_WARPS 16      // measured: 16 warps x 128 registers 115 us per 256 MiB batch; 20 x 96 the same (spills), 21 x 96 does not launch
#endif
constexpr uint32_t kFusedWarps = B2_FUSED_WARPS, kFusedBuf = B2_FUSED_BUF, kFusedRowStride = 176;
// The plain echo request exactly as PackRpcRequest emits it (baidu_rpc_protocol.cpp:1045-1133) — known fields once each, ascending,
// one-byte tags and lengths, compress / content / checksum type 0, no attachment, no checksum bytes, body "0a <len> <message>" —
// decoded, looked up and ANSWERED in ~300 instructions: descriptor to HBM, reply prefix written right in front of the payload
// (pfx_out == nullptr: in place inside the staged tile) or into pfx_out.  Returns false on ANY deviation: the caller then runs
// decode_one<true>, which alone defines the semantics; for what it accepts the result is identical (tests/test_gpu_parity.py,
// tools/fuzz_parity.py run both).
__device__ __forceinline__ bool fused_fast_echo(const BatchPtrs& B, const DevMethod* ms, uint32_t n_ms, uint32_t i, uint32_t fo, uint32_t run_idx,
                                                uint8_t* f, uint32_t avail, uint8_t* pfx_out, DecodeOut& o) {
    if (ld32_any(f) != kMagicPRPC) return false;
    const uint32_t body = __byte_perm(ld32_any(f + 4), 0, 0x0123), meta = __byte_perm(ld32_any(f + 8), 0, 0x0123);
    if (meta < 8 || (uint64_t)12 + meta + 8 > avail || meta > body) return false;
    const uint8_t* m = f + 12; const uint8_t* te = m + meta;
    if (m[0] != 0x0a) return false;
    const uint32_t L = m[1];
    if (L >= 128 || L < 4 || 2 + L > meta) return false;
    const uint8_t* q = m + 2; const uint8_t* e = q + L;
    if (q[0] != 0x0a) return false;
    const uint32_t sl = q[1];
    if (sl >= 128 || sl + 4 > L) return false;
    const uint8_t* svc = q + 2; q = svc + sl;
    if (q[0] != 0x12) return false;
    const uint32_t ml = q[1];
    if (ml >= 128 || (uint32_t)(e - q) < 2 + ml) return false;
    const uint8_t* mth = q + 2; q = mth + ml;
    uint32_t has = B2_HAS_REQUEST; uint64_t v = 0; long long log_id = 0;
    if (q < e) {
        if (*q != 0x18) return false;
        Reader r; r.p = q + 1; r.end = e;
        if (!rd_varint(r, v) || r.p != e) return false;
        log_id = (long long)v; has |= B2_HAS_LOG_ID;
    }
    const uint8_t* t = e;
    if (t + 2 <= te && t[0] == 0x18) { if (t[1] != 0) return false; has |= B2_HAS_COMPRESS_TYPE; t += 2; }
    long long cid = 0;
    if (t < te && t[0] == 0x20) { Reader r; r.p = t + 1; r.end = te; if (!rd_varint(r, v)) return false; cid = (long long)v; has |= B2_HAS_CORRELATION_ID; t = r.p; }
    if (t + 2 <= te && t[0] == 0x50) { if (t[1] != 0) return false; has |= B2_HAS_CONTENT_TYPE; t += 2; }
    if (t + 2 <= te && t[0] == 0x58) { if (t[1] != 0) return false; has |= B2_HAS_CHECKSUM_TYPE; t += 2; }
    if (t + 2 <= te && t[0] == 0x62) { if (t[1] != 0) return false; has |= B2_HAS_CHECKSUM_VALUE; t += 2; }
    if (t != te) return false;
    // Server::FindMethodPropertyByFullName on a service name that carries its package (the jprotobuf short form goes the generic way)
    bool has_dot = false;
    for (uint32_t k = 0; k < sl && !has_dot; k += 4) {
        uint32_t eq = __vcmpeq4(ld32_any(svc + k), 0x2e2e2e2eu);
        if (sl - k < 4) eq &= (1u << (8 * (sl - k))) - 1u;
        has_dot = eq != 0;
    }
    if (!has_dot) return false;
    int idx = -1;
    for (uint32_t k = 0; k < n_ms; k++) {
        const DevMethod& d = ms[k];
        if (d.full_method_len == sl + 1 + ml && d.full_method[sl] == '.' && bytes_eq(svc, d.full_method, sl) && bytes_eq(mth, d.full_method + sl + 1, ml)) { idx = (int)k; break; }
    }
    if (idx < 0) return false;
    const DevMethod& M = ms[idx];
    if (M.handler != B2_HANDLER_ECHO || M.response_checksum_type != B2_CHECKSUM_TYPE_NONE || M.response_compress_type != B2_COMPRESS_TYPE_NONE) return false;
    // EchoRequest{message}: "0a <len> <bytes>" filling the body exactly
    const uint32_t req_size = body - meta;
    if (req_size < 2 || te[0] != 0x0a) return false;
    Reader r; r.p = te + 1; r.end = te + (req_size < 6 ? req_size : 6);
    if (!rd_varint(r, v)) return false;
    const uint32_t hdr = (uint32_t)(r.p - te);
    if (v > 0x7fffffefull || (uint64_t)hdr + v != req_size) return false;
    const uint32_t msg_len = (uint32_t)v, msg_off = 12 + meta + hdr;
    // SendRpcResponse: 12 02 08 00 | 18 00 | 20 cid | 50 00 | 58 00 | 62 00, then the EchoResponse field header
    const uint32_t cidn = varint_len((uint64_t)cid), mlr = 13 + cidn, vl = varint_len(msg_len), prefix = 12 + mlr + 1 + vl;
    if (prefix > msg_off) return false;
    uint8_t* p = pfx_out ? pfx_out : f + msg_off - prefix;
    p[0] = 'P'; p[1] = 'R'; p[2] = 'P'; p[3] = 'C';
    put_be32(p + 4, mlr + 1 + vl + msg_len); put_be32(p + 8, mlr); p += 12;
    p[0] = 0x12; p[1] = 0x02; p[2] = 0x08; p[3] = 0x00; p[4] = 0x18; p[5] = 0x00; p[6] = 0x20; p += 7;
    p = put_varint(p, (uint64_t)cid);
    p[0] = 0x50; p[1] = 0x00; p[2] = 0x58; p[3] = 0x00; p[4] = 0x62; p[5] = 0x00; p[6] = 0x0a; p += 7;
    put_varint(p, msg_len);
    b2_msg_desc d;
    d.run_idx = run_idx; d.frame_off = fo; d.body_size = body; d.meta_size = meta; d.correlation_id = cid; d.log_id = log_id;
    d.attachment_size = 0; d.compress_type = 0; d.checksum_type = 0; d.error_code = 0; d.has_bits = (uint16_t)has; d.protocol = B2_PROTOCOL_BAIDU_STD;
    d.content_type = 0; d.method_idx = (int16_t)idx; d.status = B2_MSG_ECHOED; d.resp_off = fo + msg_off - prefix; d.resp_len = prefix + msg_len;
    B.msgs[i] = d;
    o.fast = true; o.slow = false; o.prefix = prefix; o.rs = d.resp_off;
    return true;
}

struct FusedWarpSmem {
    alignas(128) uint8_t buf[kFusedBuf];
    uint32_t foff[32];
    alignas(8) unsigned long long mbar;
};
// (the reply prefix of a message the GENERIC decoder answers is staged in HBM — B.heads, 96 bytes per message — not in shared
// memory: the exact-shape path writes its prefix in place and needs no staging, and shared memory buys resident warps)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// resp[a, b) <- the shared-memory image whose byte 0 is batch offset `img_off`; 16-byte aligned interior by TMA, edges by bytes
__device__ __forceinline__ void fused_store(uint8_t* resp, const uint8_t* img, uint32_t img_off, uint32_t a, uint32_t b, uint32_t lane) {
    if (a >= b) return;
    const uint32_t a0 = (a + 15u) & ~15u, b0 = b & ~15u;
    if (a0 >= b0) { for (uint32_t k = a + lane; k < b; k += 32) resp[k] = img[k - img_off]; return; }
    if (lane == 0) bulk_s2g(resp + a0, img + (a0 - img_off), b0 - a0);
    if (lane < a0 - a) resp[a + lane] = img[a + lane - img_off];
    if (lane >= 16 && lane - 16 < b - b0) resp[b0 + lane - 16] = img[b0 + lane - 16 - img_off];
}

#ifndef B2_FUSED_REGS
#define B2_FUSED_REGS 128
#endif
#ifndef B2_FUSED_PREFETCH
#define B2_FUSED_PREFETCH 1
#endif
static_assert(B2_FUSED_REGS * B2_FUSED_WARPS * 32 <= 65536, "k_fused: registers x threads must fit the SM's register file");
__global__ void __maxnreg__(B2_FUSED_REGS) k_fused(BatchPtrs B, DevConfig C) {
    extern __shared__ __align__(128) uint8_t fused_raw[];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    FusedWarpSmem& S = reinterpret_cast<FusedWarpSmem*>(fused_raw)[wid];
    if (B.totals[2] & 1u) return;
    // the method table of a typical server (one or two methods) is read from shared memory by every message
    __shared__ __align__(16) DevMethod s_methods[2];
    {
        const uint32_t nw = min(C.n_methods, 2u) * (uint32_t)(sizeof(DevMethod) / 4);
        const uint32_t* src = reinterpret_cast<const uint32_t*>(B.methods); uint32_t* dst = reinterpret_cast<uint32_t*>(s_methods);
        for (uint32_t k = threadIdx.x; k < nw; k += blockDim.x) dst[k] = src[k];
    }
    __syncthreads();
    const DevMethod* ms = C.n_methods <= 2 ? s_methods : B.methods;
    if (lane == 0) { mbar_init(&S.mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncwarp();
    uint32_t phase = 0;
    const uint32_t n_warps = gridDim.x * kFusedWarps;
    // the records of the NEXT tile are requested before the current one is worked on (they would otherwise cost a DRAM round trip per tile)
    uint32_t t = blockIdx.x * kFusedWarps + wid;
    uint4 rec_raw = make_uint4(0, 0, 0, 0), ti = make_uint4(0, 0, 0, 0); uint32_t tbase = 0;
    if (t < B.n_tiles) { rec_raw = *reinterpret_cast<const uint4*>(B.tiles + t); ti = __ldg(B.tile_info + t); tbase = B.tile_base[t]; }
    for (; t < B.n_tiles; t += n_warps) {
        const uint4 rec_cur = rec_raw, ti_cur = ti; const uint32_t tbase_cur = tbase;
        const uint32_t tn = t + n_warps;
        if (tn < B.n_tiles) { rec_raw = *reinterpret_cast<const uint4*>(B.tiles + tn); ti = __ldg(B.tile_info + tn); tbase = B.tile_base[tn]; }
        TileRec rec; *reinterpret_cast<uint4*>(&rec) = rec_cur;
        const uint32_t count = rec.count;
        if (!rec.live || count == 0) continue;
        const uint4 ti_nx = ti;                                      // (the NEXT tile's run record, loaded above)
        const uint4 ti = ti_cur;
        const uint32_t r = ti.w & 0xffffffu, run_off = ti.x, run_len = ti.y;
        const bool client = ((ti.w >> 24) & B2_RUN_CLIENT) != 0, dump = ((ti.w >> 24) & B2_RUN_RPC_DUMP) != 0;
        const uint32_t first = B.run_status[r].first_msg + tbase_cur;
        const uint32_t hi = run_off + rec.exit;
        const bool spec_ok = !(rec.kind & kKindRewalked) && count <= C.spec_k;
        const uint32_t* spec = B.tile_spec + (size_t)t * C.spec_k;
        uint32_t sub_lo = run_off + rec.entry, wpos = rec.entry; int wpf = rec.pf_in;
        for (uint32_t done = 0; done < count; done += 32) {
            const uint32_t cnt = min(32u, count - done);
            // ---- frame starts of this round of <= 32 messages, and where the round's bytes end
            uint32_t fo_raw = 0, sub_hi;
            if (spec_ok) {
                if (lane < cnt) fo_raw = __ldg(spec + done + lane);
                sub_hi = done + cnt < count ? (__ldg(spec + done + cnt) & 0x7fffffffu) : hi;
            } else {
                if (lane == 0) {                                        // a tile k_resolve re-walked (or a dense one): the chain again, true preferred index
                    for (uint32_t k = 0; k < cnt; k++) {
                        const Step sp = cut_input_message(B.bytes + run_off, run_len, wpos, wpf, C.max_body_size, client, run_mask(C.proto_mask, ti.w >> 24));
                        S.foff[k] = (run_off + sp.frame_pos) | ((uint32_t)(sp.index != 1) << 31);
                        wpos = sp.new_pos; wpf = sp.pf;
                    }
                }
                wpos = __shfl_sync(0xffffffffu, wpos, 0); wpf = __shfl_sync(0xffffffffu, wpf, 0);
                __syncwarp();
                if (lane < cnt) fo_raw = S.foff[lane];
                sub_hi = done + cnt < count ? run_off + wpos : hi;
            }
            const uint32_t lo16 = sub_lo & ~15u, hi16 = (sub_hi + 15u) & ~15u, span = hi16 - lo16;
            const uint32_t i = first + done + lane;
            const uint32_t fo = fo_raw & 0x7fffffffu;
            DecodeOut o; o.fast = false; o.slow = false; o.prefix = 0; o.rs = 0;
            const bool fits = span <= kFusedBuf;
            if (fits) {
                // ---- the whole round in one buffer: load, decode in place, patch, store
                if (lane == 0) { bulk_wait_read<0>(); mbar_arrive_expect_tx(&S.mbar, span); bulk_g2s(S.buf, B.bytes + lo16, span, &S.mbar); }
#if B2_FUSED_PREFETCH
                // while this tile is on its way: ask for the NEXT tile's bytes (its record arrived meanwhile) to be brought into L2, so that a
                // warp has two tiles' worth of DRAM reads in flight with one staging buffer
                if (lane == 0 && done == 0 && tn < B.n_tiles) {
                    TileRec nx; *reinterpret_cast<uint4*>(&nx) = rec_raw;
                    if (nx.live && nx.count) {
                        const uint32_t plo = (ti_nx.x + nx.entry) & ~15u, phi = (ti_nx.x + nx.exit + 15u) & ~15u;
                        if (phi > plo) bulk_prefetch_l2(B.bytes + plo, min(phi - plo, 2u * kFusedBuf));
                    }
                }
#endif
                __syncwarp();
                mbar_wait(&S.mbar, phase & 1u); phase++;
                bool in_place = false;
                if (lane < cnt && i < B.max_msgs) {
                    uint8_t* f = S.buf + (fo - lo16);
                    in_place = !client && !dump && !(fo_raw >> 31) && fused_fast_echo(B, ms, C.n_methods, i, fo, r, f, hi16 - fo, nullptr, o);
                    if (!in_place) decode_one<true>(B, C, i, fo_raw, f, B.heads + (size_t)i * kHeadBytes, 0xffffffffu, r, &o);
                }
                if (in_place) o.prefix = 0;                                 // (already written where it belongs)
            } else {
                // ---- big frames: decode from 160-byte rows staged in the (idle) buffer
                if (lane == 0) bulk_wait_read<0>();
                __syncwarp();
                const uint32_t sub = lane & 15, half = lane >> 4;
                for (uint32_t m2 = 0; m2 < cnt; m2 += 2) {
                    const uint32_t m = m2 + half;
                    const uint32_t f = __shfl_sync(0xffffffffu, fo, m & 31);
                    if (m < cnt && sub < kRowVecs) {
                        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(S.buf + m * kFusedRowStride + sub * 16);
                        const uint4* src = reinterpret_cast<const uint4*>(B.bytes + (f & ~15u)) + sub;
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
                if (lane < cnt && i < B.max_msgs) {
                    uint8_t* f = S.buf + lane * kFusedRowStride + (fo & 15u);
                    if (client || dump || (fo_raw >> 31) || !fused_fast_echo(B, ms, C.n_methods, i, fo, r, f, kRowBytes - (fo & 15u), B.heads + (size_t)i * kHeadBytes, o))
                        decode_one<true>(B, C, i, fo_raw, f, B.heads + (size_t)i * kHeadBytes, kRowBytes, r, &o);
                }
                __syncwarp();
            }
            // ---- everything that is not an in-place echo goes to k_pack_slow
            const uint32_t slow_mask = __ballot_sync(0xffffffffu, o.slow);
            if (slow_mask) {
                uint32_t sbase = 0;
                if (lane == 0) sbase = atomicAdd(B.totals + 3, (uint32_t)__popc(slow_mask));
                sbase = __shfl_sync(0xffffffffu, sbase, 0);
                if (o.slow) B.slow_idx[sbase + __popc(slow_mask & ((1u << lane) - 1u))] = i;
            }
            if (fits) {
                if (o.fast && o.prefix) { uint8_t* dst = S.buf + (o.rs - lo16); const uint8_t* src = B.heads + (size_t)i * kHeadBytes; for (uint32_t k = 0; k < o.prefix; k++) dst[k] = src[k]; }
                fence_proxy_async();
                __syncwarp();
                fused_store(B.resp, S.buf, lo16, sub_lo, sub_hi, lane);
                if (lane == 0) bulk_commit();
                __syncwarp();                                           // (the edge bytes were read from the buffer by other lanes)
            } else {
                // ---- stream [sub_lo, sub_hi) through the buffer, patching the prefixes that fall into each chunk
                for (uint32_t c0 = lo16; c0 < hi16; c0 += kFusedBuf) {
                    const uint32_t c1 = min(c0 + kFusedBuf, hi16);
                    if (lane == 0) { bulk_wait_read<0>(); mbar_arrive_expect_tx(&S.mbar, c1 - c0); bulk_g2s(S.buf, B.bytes + c0, c1 - c0, &S.mbar); }
                    __syncwarp();
                    mbar_wait(&S.mbar, phase & 1u); phase++;
                    if (o.fast) {
                        const uint32_t p0 = max(o.rs, c0), p1 = min(o.rs + o.prefix, c1);
                        const uint8_t* pf = B.heads + (size_t)i * kHeadBytes;
                        for (uint32_t k = p0; k < p1; k++) S.buf[k - c0] = pf[k - o.rs];
                    }
                    fence_proxy_async();
                    __syncwarp();
                    fused_store(B.resp, S.buf, c0, max(sub_lo, c0), min(sub_hi, c1), lane);
                    if (lane == 0) bulk_commit();
                    __syncwarp();
                }
            }
            sub_lo = sub_hi;
        }
    }
    if (lane == 0) bulk_wait<0>();
}


// --- k_pack_requests: the client mirror -------------------------------------------------------------
// PackRpcRequest + SerializeRpcRequest (baidu_rpc_protocol.cpp:1015-1133) and PackStreamMessage
// (streaming_rpc_protocol.cpp:42-58): one warp per frame.  The meta length does not depend on the body, so the
// body is produced in place first (serialized / snappy-compressed, CRC over what was produced), then lane 0
// writes header and meta in front of it.
struct ReqDesc {                     // == b2_request
    uint32_t kind, flags; int32_t method_idx, timeout_ms; long long correlation_id, log_id;
    int32_t compress_type, checksum_type, frame_type; uint32_t payload_off, payload_len, attachment_off, attachment_len, reserved;
};
__global__ void __launch_bounds__(256) k_pack_requests(const uint8_t* bytes, const ReqDesc* reqs, uint32_t n, const DevMethod* methods, uint32_t n_methods,
                                                       uint8_t* out, const uint32_t* out_offs, uint32_t* out_lens, uint8_t* scratch,
                                                       uint16_t* snappy_tab, const uint32_t* crc_adv) {
    __shared__ uint32_t s_hot[kCrcHotWords];
    crc_tabs_to_smem(s_hot, crc_adv);
    CrcTabs ct; ct.hot = s_hot; ct.tree = crc_adv + kCrcHotWords;
    const uint32_t lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5, warp_id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    for (uint32_t i = warp_id; i < n; i += n_warps) {
        const ReqDesc R = reqs[i];
        uint8_t* o = out + out_offs[i];
        const uint8_t* payload = bytes + R.payload_off;
        if (R.kind == 1) {                                           // ---- PackStreamMessage
            uint8_t meta[40]; uint8_t* m = meta;
            *m++ = 0x08; m = put_varint(m, (uint64_t)R.correlation_id);
            if (R.flags & 1u) { *m++ = 0x10; m = put_varint(m, (uint64_t)R.log_id); }
            *m++ = 0x18; m = put_varint(m, (uint64_t)(long long)R.frame_type);
            if (R.flags & 2u) { *m++ = 0x20; *m++ = (R.flags & 4u) ? 1 : 0; }
            const uint32_t ml = (uint32_t)(m - meta);
            if (lane == 0) {
                o[0] = 'S'; o[1] = 'T'; o[2] = 'R'; o[3] = 'M'; put_be32(o + 4, ml + R.payload_len); put_be32(o + 8, ml);
                for (uint32_t k = 0; k < ml; k++) o[12 + k] = meta[k];
            }
            warp_copy(o + 12 + ml, payload, R.payload_len, lane);
            if (lane == 0) out_lens[i] = 12 + ml + R.payload_len;
            continue;
        }
        if (R.method_idx < 0 || (uint32_t)R.method_idx >= n_methods ||
            (R.compress_type != B2_COMPRESS_TYPE_NONE && R.compress_type != B2_COMPRESS_TYPE_SNAPPY)) { if (lane == 0) out_lens[i] = 0; continue; }
        const DevMethod& M = methods[R.method_idx];
        const uint32_t mth_len = M.full_method_len - M.service_full_len - 1;
        const uint8_t* mth = reinterpret_cast<const uint8_t*>(M.full_method) + M.service_full_len + 1;
        // RpcRequestMeta: service_name(1) method_name(2) [log_id(3)] [timeout_ms(8)]
        uint32_t rl = 1 + varint_len(M.service_full_len) + M.service_full_len + 1 + varint_len(mth_len) + mth_len;
        if (R.flags & 1u) rl += 1 + varint_len((uint64_t)R.log_id);
        const bool has_to = (R.flags & 2u) && R.timeout_ms > 0;
        if (has_to) rl += 1 + varint_len((uint64_t)(long long)R.timeout_ms);
        const uint32_t cks_len = R.checksum_type == B2_CHECKSUM_TYPE_CRC32C ? 4u : 0u;
        // RpcMeta: request(1) compress_type(3) correlation_id(4) [attachment_size(5)] content_type(10) checksum_type(11) checksum_value(12)
        uint32_t ml = 1 + varint_len(rl) + rl + 1 + varint_len((uint64_t)(long long)R.compress_type) + 1 + varint_len((uint64_t)R.correlation_id);
        if (R.attachment_len) ml += 1 + varint_len(R.attachment_len);
        ml += 2 + 1 + varint_len((uint64_t)(long long)R.checksum_type) + 1 + 1 + cks_len;
        uint8_t* body = o + 12 + ml;
        const uint32_t vl = varint_len(R.payload_len), pb_len = 1 + vl + R.payload_len;
        uint32_t body_len;
        if (R.compress_type == B2_COMPRESS_TYPE_SNAPPY) {
            uint8_t* pb = scratch + out_offs[i];                     // the serialized EchoRequest, then compressed into place
            if (lane == 0) { pb[0] = 0x0a; put_varint(pb + 1, R.payload_len); }
            warp_copy(pb + 1 + vl, payload, R.payload_len, lane);
            __syncwarp();
            body_len = warp_snappy_compress(pb, pb_len, body, snappy_tab + (size_t)(warp_id % kSnappyWarps) * kSnappyMaxTable, lane);
        } else {
            if (lane == 0) { body[0] = 0x0a; put_varint(body + 1, R.payload_len); }
            warp_copy(body + 1 + vl, payload, R.payload_len, lane);
            body_len = pb_len;
        }
        __syncwarp();
        uint32_t crc_be = 0;
        if (cks_len) {                                               // Crc32cCompute (policy/crc32c_checksum.cpp:28-42) over the body
            uint32_t l = 0xffffffffu;
            if (R.compress_type == B2_COMPRESS_TYPE_SNAPPY) { __threadfence_block(); l = warp_crc32c_update(l, body, body_len, lane, ct); }
            else {                                                   // from the sources: field header, then the message bytes
                uint8_t hdr[6]; hdr[0] = 0x0a; uint8_t* e = put_varint(hdr + 1, R.payload_len);
                l = crc32c_bytes_serial(l, hdr, (uint32_t)(e - hdr));
                l = warp_crc32c_update(l, payload, R.payload_len, lane, ct);
            }
            crc_be = crc32c_mask(l ^ 0xffffffffu);
        }
        if (R.attachment_len) warp_copy(body + body_len, bytes + R.attachment_off, R.attachment_len, lane);
        if (lane == 0) {
            uint8_t* p = o;
            p[0] = 'P'; p[1] = 'R'; p[2] = 'P'; p[3] = 'C'; put_be32(p + 4, ml + body_len + R.attachment_len); put_be32(p + 8, ml); p += 12;
            *p++ = 0x0a; p = put_varint(p, rl);
            *p++ = 0x0a; p = put_varint(p, M.service_full_len); for (uint32_t k = 0; k < M.service_full_len; k++) *p++ = (uint8_t)M.service_full[k];
            *p++ = 0x12; p = put_varint(p, mth_len); for (uint32_t k = 0; k < mth_len; k++) *p++ = mth[k];
            if (R.flags & 1u) { *p++ = 0x18; p = put_varint(p, (uint64_t)R.log_id); }
            if (has_to) { *p++ = 0x40; p = put_varint(p, (uint64_t)(long long)R.timeout_ms); }
            *p++ = 0x18; p = put_varint(p, (uint64_t)(long long)R.compress_type);
            *p++ = 0x20; p = put_varint(p, (uint64_t)R.correlation_id);
            if (R.attachment_len) { *p++ = 0x28; p = put_varint(p, R.attachment_len); }
            *p++ = 0x50; *p++ = 0x00;
            *p++ = 0x58; p = put_varint(p, (uint64_t)(long long)R.checksum_type);
            *p++ = 0x62; *p++ = (uint8_t)cks_len;
            if (cks_len) p = put_be32(p, crc_be);
            out_lens[i] = 12 + ml + body_len + R.attachment_len;
        }
    }
}

// --- k_emit_iov: B2_RESP_IOVEC -------------------------------------------------------------------------------------------------
// The gather list of the write, with host addresses: what IOBuf::cut_multiple_into_file_descriptor (butil/iobuf.cpp:954-992) builds from
// the block references of queued replies.  Thread per message, after the pack kernels fixed every resp_off.
__global__ void __launch_bounds__(256) k_emit_iov(BatchPtrs B, ulonglong2* iov, unsigned long long resp_base, unsigned long long bytes_base) {
    if (B.totals[2] & 3u) return;
    const uint32_t n = B.totals[0];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const b2_msg_desc* d = B.msgs + i;
        const uint32_t status = d->status;
        ulonglong2 a = make_ulonglong2(resp_base, 0ull), b = a;
        if (status == B2_MSG_ECHOED || status == B2_MSG_ERROR_REPLIED) {
            const uint4 rf = status == B2_MSG_ECHOED ? B.refs[i] : make_uint4(0, 0, 0, 0);
            a = make_ulonglong2(resp_base + d->resp_off, rf.z ? rf.x : d->resp_len);
            if (rf.z) b = make_ulonglong2(bytes_base + rf.y, rf.z);
        } else atomicAdd(&B.run_status[d->run_idx].n_unanswered, 1u);
        iov[2 * (size_t)i] = a; iov[2 * (size_t)i + 1] = b;
    }
}

// --- k_pack_responses: SendRpcResponse (policy/baidu_rpc_protocol.cpp:273-460) for replies the host produced ------------------------
// one warp per reply: body (copied, or snappy-compressed into place), CRC32C over it, then lane 0 writes header + RpcMeta
struct ReplyDesc {                   // == b2_reply
    uint32_t flags; int32_t error_code; long long correlation_id; int32_t compress_type, checksum_type, content_type;
    uint32_t error_text_off, error_text_len, body_off, body_len, attachment_off, attachment_len, checksum_value_off, checksum_value_len,
             extra_streams_off, n_extra_streams, user_fields_off, n_user_fields, reserved;
    long long stream_id;
};
__device__ __forceinline__ uint32_t reply_user_fields_len(const uint8_t* uf, uint32_t n) {     // sum over entries of tag + len + entry
    uint32_t total = 0;
    for (uint32_t k = 0; k < n; k++) {
        const uint32_t kl = load_le32(uf), vl = load_le32(uf + 4);
        const uint32_t el = 1 + varint_len(kl) + kl + 1 + varint_len(vl) + vl;
        total += 1 + varint_len(el) + el; uf += 8 + kl + vl;
    }
    return total;
}
__global__ void __launch_bounds__(256) k_pack_responses(const uint8_t* bytes, const ReplyDesc* reps, uint32_t n, uint8_t* out, const uint32_t* out_offs,
                                                        uint32_t* out_lens, uint8_t* scratch, uint16_t* snappy_tab, const uint32_t* crc_adv) {
    __shared__ uint32_t s_hot[kCrcHotWords];
    crc_tabs_to_smem(s_hot, crc_adv);
    CrcTabs ct; ct.hot = s_hot; ct.tree = crc_adv + kCrcHotWords;
    const uint32_t lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5, warp_id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    for (uint32_t i = warp_id; i < n; i += n_warps) {
        const ReplyDesc R = reps[i];
        uint8_t* o = out + out_offs[i];
        const int32_t err = R.error_code == -1 ? B2_EINTERNAL : R.error_code;                  // :333-337
        const bool append_body = err == 0;                                                       // :316-330
        if (append_body && R.compress_type != B2_COMPRESS_TYPE_NONE && R.compress_type != B2_COMPRESS_TYPE_SNAPPY) { if (lane == 0) out_lens[i] = 0; continue; }
        const bool own_cks = append_body && R.checksum_type == B2_CHECKSUM_TYPE_CRC32C;
        const uint32_t cks_len = own_cks ? 4u : R.checksum_value_len;
        const uint32_t att_len = append_body ? R.attachment_len : 0u;
        // RpcResponseMeta: error_code(1) [error_text(2)]
        uint32_t rl = 1 + varint_len((uint64_t)(long long)err);
        if (R.error_text_len) rl += 1 + varint_len(R.error_text_len) + R.error_text_len;
        // StreamSettings: stream_id(1) need_feedback(2) writable(3) extra_stream_ids(4)*
        uint32_t sl = 0;
        const long long* extra = reinterpret_cast<const long long*>(bytes + R.extra_streams_off);
        if (R.flags & B2_RSP_HAS_STREAM) {
            sl = 1 + varint_len((uint64_t)R.stream_id) + 2 + 2;
            for (uint32_t k = 0; k < R.n_extra_streams; k++) sl += 1 + varint_len((uint64_t)extra[k]);
        }
        const uint32_t ufl = R.n_user_fields ? reply_user_fields_len(bytes + R.user_fields_off, R.n_user_fields) : 0u;
        uint32_t ml = 1 + varint_len(rl) + rl + 1 + varint_len((uint64_t)(long long)R.compress_type) + 1 + varint_len((uint64_t)R.correlation_id);
        if (att_len) ml += 1 + varint_len(att_len);
        if (R.flags & B2_RSP_HAS_STREAM) ml += 1 + varint_len(sl) + sl;
        ml += ufl;
        ml += 1 + varint_len((uint64_t)(long long)R.content_type) + 1 + varint_len((uint64_t)(long long)R.checksum_type) + 1 + varint_len(cks_len) + cks_len;
        uint8_t* body = o + 12 + ml;
        uint32_t body_len = 0;
        if (append_body) {
            if (R.compress_type == B2_COMPRESS_TYPE_SNAPPY)
                body_len = warp_snappy_compress(bytes + R.body_off, R.body_len, body, snappy_tab + (size_t)(warp_id % kSnappyWarps) * kSnappyMaxTable, lane);
            else { warp_copy(body, bytes + R.body_off, R.body_len, lane); body_len = R.body_len; }
        }
        __syncwarp();
        uint32_t crc_be = 0;
        if (own_cks) {                                                                           // Crc32cCompute over what goes on the wire
            const uint8_t* src = R.compress_type == B2_COMPRESS_TYPE_SNAPPY ? body : bytes + R.body_off;
            if (R.compress_type == B2_COMPRESS_TYPE_SNAPPY) __threadfence_block();
            crc_be = crc32c_mask(warp_crc32c_update(0xffffffffu, src, body_len, lane, ct) ^ 0xffffffffu);
        }
        if (att_len) warp_copy(body + body_len, bytes + R.attachment_off, att_len, lane);
        if (lane == 0) {
            uint8_t* p = o;
            p[0] = 'P'; p[1] = 'R'; p[2] = 'P'; p[3] = 'C'; put_be32(p + 4, ml + body_len + att_len); put_be32(p + 8, ml); p += 12;
            *p++ = 0x12; p = put_varint(p, rl);
            *p++ = 0x08; p = put_varint(p, (uint64_t)(long long)err);
            if (R.error_text_len) { *p++ = 0x12; p = put_varint(p, R.error_text_len); for (uint32_t k = 0; k < R.error_text_len; k++) *p++ = bytes[R.error_text_off + k]; }
            *p++ = 0x18; p = put_varint(p, (uint64_t)(long long)R.compress_type);
            *p++ = 0x20; p = put_varint(p, (uint64_t)R.correlation_id);
            if (att_len) { *p++ = 0x28; p = put_varint(p, att_len); }
            if (R.flags & B2_RSP_HAS_STREAM) {
                *p++ = 0x42; p = put_varint(p, sl);
                *p++ = 0x08; p = put_varint(p, (uint64_t)R.stream_id);
                *p++ = 0x10; *p++ = (R.flags & B2_RSP_STREAM_NEED_FEEDBACK) ? 1 : 0;
                *p++ = 0x18; *p++ = (R.flags & B2_RSP_STREAM_WRITABLE) ? 1 : 0;
                for (uint32_t k = 0; k < R.n_extra_streams; k++) { *p++ = 0x20; p = put_varint(p, (uint64_t)extra[k]); }
            }
            const uint8_t* uf = bytes + R.user_fields_off;
            for (uint32_t k = 0; k < R.n_user_fields; k++) {                                     // map<string,string> user_fields = 9: entry {key = 1, value = 2}
                const uint32_t kl = load_le32(uf), vl = load_le32(uf + 4);
                const uint32_t el = 1 + varint_len(kl) + kl + 1 + varint_len(vl) + vl;
                *p++ = 0x4a; p = put_varint(p, el);
                *p++ = 0x0a; p = put_varint(p, kl); for (uint32_t q = 0; q < kl; q++) *p++ = uf[8 + q];
                *p++ = 0x12; p = put_varint(p, vl); for (uint32_t q = 0; q < vl; q++) *p++ = uf[8 + kl + q];
                uf += 8 + kl + vl;
            }
            *p++ = 0x50; p = put_varint(p, (uint64_t)(long long)R.content_type);
            *p++ = 0x58; p = put_varint(p, (uint64_t)(long long)R.checksum_type);
            *p++ = 0x62; p = put_varint(p, cks_len);
            if (own_cks) p = put_be32(p, crc_be);
            else for (uint32_t k = 0; k < cks_len; k++) *p++ = bytes[R.checksum_value_off + k];
            out_lens[i] = 12 + ml + body_len + att_len;
        }
    }
}

// --- k_pack_slow: everything that is not a plain OK echo ----------------------
// error replies, CRC32C verify/compute, snappy requests, split attachments: warp per message,
// high occupancy (these are latency-bound), skipping the messages k_pack_tma moves.
#ifndef B2_SLOW_MIN_BLOCKS
#define B2_SLOW_MIN_BLOCKS 3
#endif
// kLite: no shared memory at all (CRC tables read through L1, no snappy ring) — the variant launched behind k_fused, where slow messages
// are rare by construction and the kernel must be able to start on SMs whose shared memory the next batch's k_fused already holds
template <bool kLite>
__global__ void __launch_bounds__(256, B2_SLOW_MIN_BLOCKS) k_pack_slow(BatchPtrs B, DevConfig C) {
    const uint32_t lane = threadIdx.x & 31;
    if (B.totals[2] & 3u) return;
    finalize_runs(B, C);                               // (was a separate launch)
    const uint32_t n_verify = C.verify_done ? 0u : B.totals[7];
    if (B.totals[3] == 0 && n_verify == 0) return;
    __shared__ uint32_t s_hot[kLite ? 1 : kCrcHotWords];
    extern __shared__ __align__(16) uint8_t s_rings[];           // kSnapRing bytes per warp
    CrcTabs ct; ct.tree = B.crc_adv + kCrcHotWords;
    if (kLite) { ct.hot = B.crc_adv; ct.ring = nullptr; }
    else { crc_tabs_to_smem(s_hot, B.crc_adv); ct.hot = s_hot; ct.ring = s_rings + (threadIdx.x >> 5) * kSnapRing; }
    // the slow messages were listed by k_decode; warps pull them one at a time (sizes vary from an error
    // text to a 256 KiB snappy stream, so the queue is dynamic: totals[6] is the ticket)
    // verify pass: Crc32cVerify (policy/crc32c_checksum.cpp:44-61) of the plain echoes whose reply k_pack_tma moves;
    // a request that fails is answered here (EREQUEST) and taken off the bandwidth path
    for (; !C.verify_done;) {
        uint32_t k = 0;
        if (lane == 0) k = atomicAdd(B.totals + 8, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= n_verify) break;
        const uint32_t i = B.slow_idx[B.max_msgs - 1 - k];
        const uint32_t fo = B.msgs[i].frame_off, meta_size = B.msgs[i].meta_size;
        const uint32_t req_size = B.msgs[i].body_size - meta_size;
        int64_t bwo = (int64_t)req_size - (int64_t)B.msgs[i].attachment_size; if (bwo > (int64_t)req_size) bwo = req_size;
        const uint8_t* frame = B.bytes + fo;
        const uint32_t crc = warp_crc32c_update(0xffffffffu, frame + 12 + meta_size, (uint32_t)bwo, lane, ct) ^ 0xffffffffu;
        const bool good = crc == crc32c_unmask(load_be32(frame + B.aux[i].cks_off));
        if (good) { if (lane == 0) B.jobs[i].fast = 1; }
        else { if (lane == 0) B.jobs[i].fast = 0; __syncwarp(); pack_one(B, C, i, lane, ct); }
    }
    const uint32_t n_slow = B.totals[3];
    for (;;) {
        uint32_t k = 0;
        if (lane == 0) k = atomicAdd(B.totals + 6, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= n_slow) break;
        const uint32_t i = B.slow_idx[k];
        const bool deferred = C.fused && B.msgs[i].status == kDeferred;
        __syncwarp();                                               // (every lane has read the status before lane 0 rewrites the descriptor)
        if (deferred) {                                             // parked by k_fused: the out-of-line decode (sizing pass included), then the pack
            if (lane == 0) {
                const uint32_t fo_raw = B.msgs[i].frame_off; DecodeOut o;
                decode_one_gz<true>(B, C, i, fo_raw, B.bytes + (fo_raw & 0x7fffffffu), B.heads + (size_t)i * kHeadBytes, 0xffffffffu, B.msgs[i].run_idx, &o);
            }
            __threadfence_block();
            __syncwarp();
        }
        pack_one(B, C, i, lane, ct);
    }
}


// --- k_crc_verify: Crc32cVerify (policy/crc32c_checksum.cpp:44-61) of every CRC-carrying plain echo, as a kernel of its own -----------
// The verify pass is a chain of shared-memory table look-ups per message: what it needs is many resident warps and loads issued ahead of
// the chain, not the 80 registers of the general slow path.  48 warps per SM, one message per warp at a time; a request that passes is
// released to the bandwidth path (jobs[i].fast = 1), one that fails joins k_pack_slow's list and is answered EREQUEST there.
__global__ void __launch_bounds__(256, 6) k_crc_verify(BatchPtrs B, DevConfig C) {
    if (B.totals[2] & 3u) return;
    const uint32_t n_verify = B.totals[7];
    if (n_verify == 0) return;
    __shared__ uint32_t s_hot[kCrcHotWords];
    crc_tabs_to_smem(s_hot, B.crc_adv);
    CrcTabs ct; ct.hot = s_hot; ct.tree = B.crc_adv + kCrcHotWords; ct.ring = nullptr;
    const uint32_t lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_verify; k += n_warps) {
        const uint32_t i = B.slow_idx[B.max_msgs - 1 - k];
        const uint32_t fo = B.msgs[i].frame_off, meta_size = B.msgs[i].meta_size;
        const uint32_t req_size = B.msgs[i].body_size - meta_size;
        int64_t bwo = (int64_t)req_size - (int64_t)B.msgs[i].attachment_size; if (bwo > (int64_t)req_size) bwo = req_size;
        const uint8_t* frame = B.bytes + fo;
        const uint32_t crc = warp_crc32c_update(0xffffffffu, frame + 12 + meta_size, (uint32_t)bwo, lane, ct) ^ 0xffffffffu;
        const bool good = crc == crc32c_unmask(load_be32(frame + B.aux[i].cks_off));
        if (lane == 0) {
            if (good) B.jobs[i].fast = 1;
            else { B.jobs[i].fast = 0; B.slow_idx[atomicAdd(B.totals + 3, 1u)] = i; }
        }
    }
}

// --- k_small: the whole path in ONE launch for latency-sized batches ------------------------------
// A batch of <= 128 KB / 512 runs / 1024 messages (what a set of synchronous clients has in flight)
// does not need the tile machinery: one CTA walks every run's frame chain (thread per run, true
// preferred index, no speculation), scans, decodes (same decode_round as k_decode), scans the reply
// slots and packs (register copies), with __syncthreads() where the big pipeline has kernel
// boundaries.  Ten launches become one; results are identical by construction (same device functions).
constexpr uint32_t kSmallThreads = 512, kSmallWarps = kSmallThreads / 32;
struct SmallSmem {
    DecodeWarpSmem dec[kSmallWarps];
    uint32_t run_count[kSmallThreads];
    uint32_t scan[1024 + 1];
    uint32_t s_hot[kCrcHotWords];
    uint32_t warp_tot[kSmallWarps];
    uint32_t n_msgs, resp_total;
};
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* warp_tot, uint32_t& total) {
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= (uint32_t)d) x += y; }
    __syncthreads();
    if (lane == 31) warp_tot[wid] = x;
    __syncthreads();
    uint32_t base = 0, tot = 0;
    for (uint32_t w = 0; w < kSmallWarps; w++) { const uint32_t t = warp_tot[w]; if (w < wid) base += t; tot += t; }
    total = tot;
    return base + x - v;
}
__device__ __forceinline__ void small_body(const BatchPtrs& B, const DevConfig& C, SmallSmem& S) {
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    CrcTabs ct; ct.hot = S.s_hot; ct.tree = B.crc_adv + kCrcHotWords;
    // ---- cut loop: thread per run (ProcessNewMessage over the whole run)
    uint32_t my_count = 0; b2_run_status st; st.consumed = 0; st.parse_error = B2_PARSE_ERROR_NOT_ENOUGH_DATA; st.n_msgs = 0;
    st.first_msg = 0; st.preferred_proto = -1; st.n_unanswered = 0; st.resp_off = 0; st.resp_bytes = 0;
    b2_run run; run.offset = 0; run.length = 0; run.preferred_proto = -1; run.flags = 0; run.socket_id = 0;
    if (tid < B.n_runs) {
        run = B.runs[tid];
        uint32_t pos = 0; int pf = run.preferred_proto;
        for (;;) {
            const Step sp = cut_input_message(B.bytes + run.offset, run.length, pos, pf, C.max_body_size, (run.flags & B2_RUN_CLIENT) != 0, run_mask(C.proto_mask, run.flags));
            pos = sp.new_pos; pf = sp.pf;
            if (sp.err != B2_PARSE_OK) { st.parse_error = (uint32_t)sp.err; break; }
            my_count++;
        }
        st.consumed = pos; st.preferred_proto = pf; st.n_msgs = my_count;
    }
    uint32_t total = 0;
    const uint32_t first = block_excl_scan(my_count, S.warp_tot, total);
    if (tid == 0) { S.n_msgs = total; B.totals[0] = total; if (total > B.max_msgs) B.totals[2] |= 1u; }
    __syncthreads();
    if (total > B.max_msgs) return;
    // ---- frame table: the same walk again, now writing offsets
    if (tid < B.n_runs) {
        st.first_msg = first;
        uint32_t pos = 0, k = 0; int pf = run.preferred_proto;
        for (;;) {
            const Step sp = cut_input_message(B.bytes + run.offset, run.length, pos, pf, C.max_body_size, (run.flags & B2_RUN_CLIENT) != 0, run_mask(C.proto_mask, run.flags));
            if (sp.err != B2_PARSE_OK) break;
            B.frame_off[first + k] = (run.offset + sp.frame_pos) | ((uint32_t)(sp.index != 1) << 31);
            B.frame_run[first + k] = tid; if (C.pull) B.frame_row[first + k] = kNone; k++;
            pos = sp.new_pos; pf = sp.pf;
        }
        B.run_status[tid] = st;
    }
    __syncthreads();
    // ---- decode
    for (uint32_t i0 = wid * 32; i0 < total; i0 += kSmallWarps * 32) decode_round(B, C, S.dec[wid], i0, total, lane);
    __syncthreads();
    // ---- reply slots: exclusive scan (<= 1024 messages: two per thread)
    {
        const uint32_t a0 = 2 * tid, a1 = 2 * tid + 1;
        const uint32_t v0 = a0 < total ? B.slot[a0] : 0, v1 = a1 < total ? B.slot[a1] : 0;
        uint32_t tot = 0;
        const uint32_t ex = block_excl_scan(v0 + v1, S.warp_tot, tot);
        if (a0 < total) B.slot[a0] = ex;
        if (a1 < total) B.slot[a1] = ex + v0;
        if (tid == 0) { B.scan_tmp[0] = 0; B.totals[1] = tot; S.resp_total = tot; if (tot > B.max_resp) B.totals[2] |= 2u; }
    }
    __syncthreads();
    if (S.resp_total > B.max_resp) return;
    // ---- pack: warp per message
    for (uint32_t i = wid; i < total; i += kSmallWarps) {
        const PackJob job = B.jobs[i];
        if (job.fast != 1) { pack_one(B, C, i, lane, ct); continue; }   // (2 = CRC to verify: pack_one does it)
        const uint32_t so = B.slot[i];
        // slot image = head record + 16-byte aligned rest of the payload (see k_pack_tma); plain 16 B copies here
        const uint4* hs = reinterpret_cast<const uint4*>(B.heads + (size_t)i * kHeadBytes);
        uint4* dst = reinterpret_cast<uint4*>(B.resp + so);
        for (uint32_t k = lane; k < job.head_len / 16u; k += 32) dst[k] = hs[k];
        const uint4* ps = reinterpret_cast<const uint4*>(B.bytes + job.src_off);
        uint4* pd = reinterpret_cast<uint4*>(B.resp + so + job.head_len);
        for (uint32_t k = lane; k < job.bulk_len / 16u; k += 32) pd[k] = __ldg(ps + k);
        if (lane == 0) B.msgs[i].resp_off = so + job.pad;
    }
    __syncthreads();
    // ---- per-run reply span + counters
    if (tid < B.n_runs) {
        auto off_of = [&](uint32_t i) -> uint32_t { return i >= total ? S.resp_total : B.slot[i]; };
        st.resp_off = off_of(st.first_msg);
        st.resp_bytes = off_of(st.first_msg + st.n_msgs) - st.resp_off;
        B.run_status[tid] = st;
        atomicAdd(B.counters + 0, (unsigned long long)st.consumed);
        atomicAdd(B.counters + 1, (unsigned long long)st.n_msgs);
        atomicAdd(B.counters + 2, (unsigned long long)st.resp_bytes);
        if (st.parse_error != B2_PARSE_ERROR_NOT_ENOUGH_DATA) atomicAdd(B.counters + 4, 1ull);
        if (tid == 0) atomicAdd(B.counters + 5, 1ull);
    }
}

__global__ void __launch_bounds__(kSmallThreads, 1) k_small(BatchPtrs B, DevConfig C) {
    extern __shared__ __align__(128) uint8_t small_raw[];
    SmallSmem& S = *reinterpret_cast<SmallSmem*>(small_raw);
    crc_tabs_to_smem(S.s_hot, B.crc_adv);
    small_body(B, C, S);
}

// --- k_ring: the persistent latency kernel ----------------------------------------------------------------------
// One resident CTA per context polls a submit ring in pinned + mapped host memory (the doorbell is a plain host store,
// there is no launch and no cudaMemcpy per batch): when slot (ticket % kRingSlots) carries `ticket`, the CTA pulls the
// slot's runs and the batch bytes out of host memory with coalesced 16-byte loads into HBM, runs small_body (the same
// device code as k_small) and pushes the compact result block straight into the slot's pinned output area with posted
// PCIe writes, then releases `done = ticket` system-wide.  It leaves on `stop` or after idle_ns without work (so that
// device-wide synchronisation points — cudaFree, cudaDeviceSynchronize — are never held for long); the host relaunches
// it with the next submission.
constexpr uint32_t kRingSlots = 8;
struct RingSlotHdr {                 // in mapped host memory, one per slot; the host fills everything, then stores `submit` last
    volatile uint32_t submit;        // ticket of the submission this slot carries
    uint32_t n_runs, nbytes, small_msgs;
    uint32_t small_resp, off_rs, off_msgs, off_refs;
    uint32_t off_resp, total, by_ref, reserved;
    unsigned long long bytes_dev;    // device-visible address of the batch bytes (the caller's pinned block, or the slot's staging area)
    unsigned long long pad0;
    volatile uint32_t done;          // device: ticket, after the output block is visible
    uint32_t pad1[3];
    unsigned long long stamps[6];    // device %globaltimer (ns): doorbell seen, header read, bytes pulled, body done, results pushed, (spare)
};                                   // 128 bytes
struct RingDev {
    uint8_t* slots;                  // mapped host memory: kRingSlots x slot_stride
    uint32_t slot_stride, off_runs, off_in, off_out;     // layout of one slot: [RingSlotHdr | runs | staged input | output block]
    volatile uint32_t* ctl;          // mapped host memory: [0] stop  [1] running  [2] batches served
    uint32_t* next_ticket;           // device memory: ticket the kernel waits for next (survives relaunches)
    unsigned long long idle_ns;
    uint8_t* d_bytes; uint8_t* d_meta; uint8_t* d_small;   // device staging: batch bytes, runs, compact output block
};
__device__ __forceinline__ uint32_t ld_sys_u32(const volatile uint32_t* p) {
    uint32_t v; asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_sys_u32(volatile uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

__global__ void __launch_bounds__(kSmallThreads, 1) k_ring(RingDev R, BatchPtrs B0, DevConfig C) {
    extern __shared__ __align__(128) uint8_t small_raw[];
    SmallSmem& S = *reinterpret_cast<SmallSmem*>(small_raw);
    __shared__ uint32_t s_go;
    __shared__ RingSlotHdr s_hdr;
    const uint32_t tid = threadIdx.x;
    crc_tabs_to_smem(S.s_hot, B0.crc_adv);
    uint32_t ticket = *R.next_ticket;
    for (;;) {
        uint8_t* slot = R.slots + (size_t)(ticket % kRingSlots) * R.slot_stride;
        RingSlotHdr* hdr = reinterpret_cast<RingSlotHdr*>(slot);
        if (tid == 0) {
            const unsigned long long t0 = globaltimer_ns();
            uint32_t go = 0;
            for (;;) {
                if (ld_sys_u32(&hdr->submit) == ticket) { go = 1; break; }
                if (ld_sys_u32(R.ctl + 0)) break;
                if (globaltimer_ns() - t0 > R.idle_ns) {
                    // leave: announce it first, then look once more so that a submission racing with the exit is not lost
                    st_sys_u32(R.ctl + 1, 0); __threadfence_system();
                    if (ld_sys_u32(&hdr->submit) == ticket) { st_sys_u32(R.ctl + 1, 1); go = 1; }
                    break;
                }
            }
            s_go = go;
        }
        __syncthreads();
        if (!s_go) break;
        unsigned long long t_seen = 0, t_hdr = 0, t_pull = 0, t_body = 0;
        if (tid == 0) t_seen = globaltimer_ns();
        // the slot header (the host's stores are ordered before `submit` by its release fence)
        if (tid < sizeof(RingSlotHdr) / 4) reinterpret_cast<uint32_t*>(&s_hdr)[tid] = ld_sys_u32(reinterpret_cast<const volatile uint32_t*>(slot) + tid);
        __syncthreads();
        const uint32_t n_runs = s_hdr.n_runs, nbytes = s_hdr.nbytes;
        if (tid == 0) t_hdr = globaltimer_ns();
        {   // pull: runs (24 B each) + per-run tile base placeholder, then the batch bytes, 16 bytes per thread per trip
            const uint4* src = reinterpret_cast<const uint4*>(slot + R.off_runs);
            uint4* dst = reinterpret_cast<uint4*>(R.d_meta);
            for (uint32_t k = tid; k < (n_runs * 24u + 15u) / 16u; k += kSmallThreads) dst[k] = src[k];
            const uint4* bs = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(s_hdr.bytes_dev));
            uint4* bd = reinterpret_cast<uint4*>(R.d_bytes);
            const uint32_t nv = (nbytes + 15u) / 16u;
            uint32_t k = tid;
            for (; k + 3 * kSmallThreads < nv; k += 4 * kSmallThreads) {              // four loads in flight per thread
                const uint4 a = bs[k], b = bs[k + kSmallThreads], c = bs[k + 2 * kSmallThreads], d = bs[k + 3 * kSmallThreads];
                bd[k] = a; bd[k + kSmallThreads] = b; bd[k + 2 * kSmallThreads] = c; bd[k + 3 * kSmallThreads] = d;
            }
            for (; k < nv; k += kSmallThreads) bd[k] = bs[k];
        }
        BatchPtrs B = B0;
        B.bytes = R.d_bytes; B.runs = reinterpret_cast<const b2_run*>(R.d_meta); B.n_runs = n_runs;
        B.totals = reinterpret_cast<uint32_t*>(R.d_small);
        B.run_status = reinterpret_cast<b2_run_status*>(R.d_small + s_hdr.off_rs);
        B.msgs = reinterpret_cast<b2_msg_desc*>(R.d_small + s_hdr.off_msgs);
        B.refs = reinterpret_cast<uint4*>(R.d_small + s_hdr.off_refs);
        B.resp = R.d_small + s_hdr.off_resp;
        B.max_msgs = s_hdr.small_msgs; B.max_resp = s_hdr.small_resp;
        DevConfig Cb = C; Cb.by_ref = s_hdr.by_ref; Cb.pull = 0;
        if (tid < 16) B.totals[tid] = 0;
        __threadfence();
        __syncthreads();
        if (tid == 0) t_pull = globaltimer_ns();
        small_body(B, Cb, S);
        __threadfence();
        __syncthreads();
        if (tid == 0) t_body = globaltimer_ns();
        {   // push the compact block [totals | run_status | msgs | refs | resp] into the slot's output area
            const uint32_t used = (B.totals[2] & 3u) ? 64u : s_hdr.off_resp + ((B.totals[1] + 15u) & ~15u);
            const uint4* src = reinterpret_cast<const uint4*>(R.d_small);
            uint4* dst = reinterpret_cast<uint4*>(slot + R.off_out);
            for (uint32_t k = tid; k < (used + 15u) / 16u; k += kSmallThreads) dst[k] = __ldcg(src + k);
        }
        if (tid == 0) { hdr->stamps[0] = t_seen; hdr->stamps[1] = t_hdr; hdr->stamps[2] = t_pull; hdr->stamps[3] = t_body; hdr->stamps[4] = globaltimer_ns(); }
        __threadfence_system();
        __syncthreads();
        if (tid == 0) { st_sys_u32(&hdr->done, ticket); st_sys_u32(R.ctl + 2, ticket + 1); }
        ticket++;
    }
    if (tid == 0) *R.next_ticket = ticket;
}

// b2_h2_decompress_requests: the output slots of the messages to inflate (B2_H2_UNZ_OK, out_len = the sizing bound), back to back in
// message order: an exclusive scan of the bounds by one block, each thread a contiguous run of messages.  A message whose slot would
// end past out_cap is B2_H2_UNZ_NO_ROOM, and so is every later one with a non-empty bound (the running sum keeps its bound).
constexpr uint32_t kUnzScanBlock = 1024;
__global__ void __launch_bounds__(kUnzScanBlock) k_h2_unz_offsets(b2_h2_unz_result* res, uint32_t n, uint32_t out_cap) {
    __shared__ unsigned long long s[kUnzScanBlock];
    const uint32_t t = threadIdx.x, per = (n + kUnzScanBlock - 1) / kUnzScanBlock, b = min(t * per, n), e = min(b + per, n);
    unsigned long long sum = 0;
    for (uint32_t i = b; i < e; i++) if (res[i].status == B2_H2_UNZ_OK) sum += res[i].out_len;
    s[t] = sum;
    __syncthreads();
    for (uint32_t d = 1; d < kUnzScanBlock; d <<= 1) {
        const unsigned long long v = t >= d ? s[t - d] : 0ull;
        __syncthreads();
        s[t] += v;
        __syncthreads();
    }
    unsigned long long off = s[t] - sum;
    for (uint32_t i = b; i < e; i++) {
        if (res[i].status != B2_H2_UNZ_OK) continue;
        const uint32_t bound = res[i].out_len;
        if (off + bound > out_cap) { res[i].status = B2_H2_UNZ_NO_ROOM; res[i].out_len = 0; }
        else res[i].out_off = (uint32_t)off;
        off += bound;
    }
}

#endif  // __CUDACC__
}  // namespace b2
