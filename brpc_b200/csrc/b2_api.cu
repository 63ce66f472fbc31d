// b2_api.cu — the C ABI (include/b2rpc.h) over the sm_100a kernels.
// Host code is plain C++ + the CUDA runtime; nothing here computes on the CPU:
// without a CUDA device every entry point fails with B2_E_NO_DEVICE.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdio.h>
#include <time.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>
#include "b2_kernels.cuh"
#include "b2_h2.cuh"

using namespace b2;

static thread_local char g_err[512] = "";
static void set_err(const char* fmt, const char* a = "", const char* b = "") { snprintf(g_err, sizeof g_err, fmt, a, b); }

#define CU(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) { set_err("%s: %s", #call, cudaGetErrorString(e_)); return B2_E_CUDA; } \
    } while (0)

namespace {
constexpr int kMaxStages = 16;
constexpr uint32_t kSmallBytes = 128 << 10;        // batches up to this size take the latency path
constexpr uint32_t kSmallRuns = 512, kSmallMsgs = 1024;   // == kSmallThreads, 2 * kSmallThreads of k_small
constexpr size_t kSmallBlock = 64 + kSmallRuns * 32 + kSmallMsgs * (64 + 16) + (kSmallBytes + kSmallMsgs * 80 + 4096);
struct Stage { const char* name; cudaEvent_t ev; };
}

struct b2_ctx {
    b2_options opt;
    DevConfig cfg;
    std::vector<DevMethod> methods;
    // device
    uint8_t* d_bytes = nullptr; b2_run* d_runs = nullptr; uint32_t* d_run_tile_base = nullptr;
    TileRec* d_tiles = nullptr; uint32_t* d_tile_base = nullptr; uint32_t* d_tile_scratch = nullptr; uint32_t* d_tile_spec = nullptr; b2_run_status* d_run_status = nullptr;
    uint32_t* d_frame_off = nullptr; uint32_t* d_frame_run = nullptr; b2_msg_desc* d_msgs = nullptr; MsgAux* d_aux = nullptr; PackJob* d_jobs = nullptr; uint32_t* d_slow_idx = nullptr; uint8_t* d_heads = nullptr;
    uint32_t* d_slot = nullptr; uint32_t* d_scan_tmp = nullptr; uint8_t* d_resp = nullptr; uint8_t* d_unz = nullptr; uint16_t* d_snappy_tab = nullptr; HpackState* d_hpack = nullptr; H2Conn* d_h2 = nullptr; H2Stream* d_h2_streams = nullptr; uint8_t* d_h2_slots = nullptr; uint32_t h2_max_conns = B2_H2_MAX_CONNS, h2_pending = B2_H2_MAX_PENDING, h2_stream_bytes = B2_H2_STREAM_BYTES; uint64_t h2_last_in = 0, h2_last_out = 0, h2_last_unz = 0;   // sizes of the last h2 batch (and of its inflated messages) still on the device
    uint8_t* d_h2_unz = nullptr;                                  // b2_h2_decompress_requests output (max_resp_bytes, allocated on first use)
    uint32_t* d_frame_row = nullptr; uint4* d_rows = nullptr;
    // persistent latency kernel (b2_ring_*): pinned + mapped submit ring, its own stream
    uint8_t* ring_slots = nullptr; volatile uint32_t* ring_ctl = nullptr; uint32_t* d_ring_ticket = nullptr; cudaStream_t ring_stream = nullptr;
    uint32_t ring_next = 1, ring_stride = 0, ring_off_runs = 0, ring_off_in = 0, ring_off_out = 0; bool ring_collected[8] = { true, true, true, true, true, true, true, true };
    const void* ring_bytes[8] = {}; const void* ring_pin_base = nullptr; unsigned long long ring_pin_dev = 0; uint64_t ring_launches = 0;
    ulonglong2* d_iov = nullptr; b2_iovec* h_iov = nullptr; const void* host_bytes = nullptr;      // B2_RESP_IOVEC
    uint4* d_refs = nullptr; b2_resp_ref* h_refs = nullptr; int input_mode = B2_INPUT_COPY, resp_mode = B2_RESP_COPY; const uint8_t* pull_bytes = nullptr; uint32_t small_off_refs = 0;
    uint32_t* d_crc_adv = nullptr; unsigned long long* d_counters = nullptr; uint32_t* d_totals = nullptr; DevMethod* d_methods = nullptr;
    size_t meta_tile_off = 0; uint32_t max_tiles = 0; uint32_t n_sms = 148; bool use_tma_pack = true; uint32_t stage_mask = 7;  // debug: 1 front stages, 2 k_pack_tma, 4 k_pack_slow
    // pinned host mirrors
    b2_run_status* h_run_status = nullptr; b2_msg_desc* h_msgs = nullptr; uint8_t* h_resp = nullptr;
    uint32_t* h_totals = nullptr; uint32_t* h_run_tile_base = nullptr;
    // current batch
    uint32_t n_runs = 0, n_tiles = 0, nbytes = 0, max_run_tiles = 0; uint64_t covered = 0;
    bool uploaded = false, executed = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[kMaxStages + 1];
    const char* stage_names[kMaxStages];
    int n_stages = 0;
    float last_kernel_ms = 0.f; uint32_t last_launches = 0;
    cudaEvent_t ev_first = nullptr, ev_last = nullptr; bool first_pending = true;
    bool profile_stages = false; bool allow_small = true; bool use_fused = true; bool fused_last = false; bool slow_heavy = false;   // slow_heavy: the previous batch sent > 1/8 of its messages to k_pack_slow (CRC'd / compressed traffic): the classic pipeline serves that better
    bool adaptive_tile = false; bool dense = false; uint32_t avg_frame = 0;   // tile size follows the message size of the previous batch      // per-stage events only when a harness asks for stage times
    // small-batch (latency) mode: one compact H2D block, one compact output block, one D2H, one sync
    uint8_t* d_meta = nullptr; uint8_t* h_meta = nullptr;       // [runs | run_tile_base]
    uint8_t* d_small = nullptr; uint8_t* h_small = nullptr;     // [totals | run_status | msgs | resp]
    bool small = false, small_copy_queued = false, use_fused_small = true; uint32_t small_msgs = 0, small_resp = 0, small_off_rs = 0, small_off_msgs = 0, small_off_resp = 0, small_total = 0;
};

static uint32_t g_crc_tab_host[256];
static void crc_table_init() {
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0x82f63b78u : (c >> 1);
        g_crc_tab_host[i] = c;
    }
}

extern "C" const char* b2_last_error(void) { return g_err; }
extern "C" const char* b2_version(void) { return "brpc_b200 0.1 (sm_100a)"; }

// ---- pinned block pool (seam 3: butil::iobuf::blockmem_allocate / blockmem_deallocate, src/butil/iobuf.cpp:168-169; same role as
// rdma::block_pool, src/brpc/rdma/block_pool.h:74-105).  cudaHostAlloc / cudaFreeHost cost tens of microseconds and serialise
// with the device, so they are paid per SLAB, never per block: blocks of up to 8 KiB (IOBuf::DEFAULT_BLOCK_SIZE) are carved out
// of 4 MiB slabs and recycled through a free list; larger requests (socket read arenas, batch buffers) are rounded up to a power
// of two (+ 1 KiB of slack so 16-byte over-reads of a device kernel stay inside the mapping) and cached per size class when
// freed.  All memory is mapped (cudaHostAllocMapped | Portable): a kernel can read it in place (B2_INPUT_PULL).
namespace {
struct BlockPool {
    std::mutex mu;
    static constexpr size_t kSmall = 8192, kSlab = 4u << 20;
    std::vector<uint8_t*> slabs; std::vector<void*> small_free;
    std::unordered_map<void*, int> large_class;          // live + cached large blocks -> size class (log2)
    std::vector<void*> large_free[40];
    uint64_t n_host_alloc = 0;
    void* alloc(size_t size) {
        std::lock_guard<std::mutex> g(mu);
        if (size <= kSmall) {
            if (small_free.empty()) {
                uint8_t* slab = nullptr;
                if (cudaHostAlloc((void**)&slab, kSlab, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return nullptr;
                n_host_alloc++; slabs.push_back(slab);
                for (size_t o = 0; o + kSmall <= kSlab; o += kSmall) small_free.push_back(slab + o);
            }
            void* p = small_free.back(); small_free.pop_back(); return p;
        }
        int cls = 14; while (((size_t)1 << cls) < size) cls++;
        if (cls >= 40) return nullptr;
        if (!large_free[cls].empty()) { void* p = large_free[cls].back(); large_free[cls].pop_back(); return p; }
        void* p = nullptr;
        if (cudaHostAlloc(&p, ((size_t)1 << cls) + 1024, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return nullptr;
        n_host_alloc++; large_class[p] = cls;
        return p;
    }
    void free(void* p) {
        std::lock_guard<std::mutex> g(mu);
        auto it = large_class.find(p);
        if (it != large_class.end()) { large_free[it->second].push_back(p); return; }
        small_free.push_back(p);                           // (a slab block; slabs live until process exit)
    }
};
BlockPool& block_pool() { static BlockPool* p = new BlockPool; return *p; }
}
extern "C" void* b2_block_alloc(size_t size) {
    void* p = block_pool().alloc(size ? size : 1);
    if (!p) set_err("cudaHostAlloc failed");
    return p;
}
extern "C" void b2_block_free(void* p) { if (p) block_pool().free(p); }
extern "C" uint64_t b2_block_pool_host_allocs(void) { std::lock_guard<std::mutex> g(block_pool().mu); return block_pool().n_host_alloc; }

static void ring_halt(b2_ctx* c);
extern "C" void b2_ctx_destroy(b2_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->opt.device);
    ring_halt(c);
    if (c->ring_stream) cudaStreamDestroy(c->ring_stream);
    if (c->ring_slots) cudaFreeHost(c->ring_slots);
    if (c->ring_ctl) cudaFreeHost((void*)c->ring_ctl);
    cudaFree(c->d_ring_ticket);
    cudaFree(c->d_bytes); cudaFree(c->d_runs); cudaFree(c->d_run_tile_base); cudaFree(c->d_tiles); cudaFree(c->d_tile_base); cudaFree(c->d_tile_scratch); cudaFree(c->d_tile_spec);
    cudaFree(c->d_run_status); cudaFree(c->d_frame_off); cudaFree(c->d_frame_run); cudaFree(c->d_msgs); cudaFree(c->d_aux); cudaFree(c->d_jobs); cudaFree(c->d_slow_idx); cudaFree(c->d_heads); cudaFree(c->d_slot);
    cudaFree(c->d_scan_tmp); cudaFree(c->d_resp); cudaFree(c->d_unz); cudaFree(c->d_snappy_tab); cudaFree(c->d_refs); cudaFree(c->d_iov); cudaFreeHost(c->h_iov); cudaFree(c->d_frame_row); cudaFree(c->d_rows); cudaFreeHost(c->h_refs); cudaFree(c->d_hpack); cudaFree(c->d_h2); cudaFree(c->d_h2_streams); cudaFree(c->d_h2_slots); cudaFree(c->d_h2_unz); cudaFree(c->d_counters); cudaFree(c->d_totals); cudaFree(c->d_methods); cudaFree(c->d_crc_adv); cudaFree(c->d_meta); cudaFree(c->d_small); cudaFreeHost(c->h_meta); cudaFreeHost(c->h_small);
    cudaFreeHost(c->h_run_status); cudaFreeHost(c->h_msgs); cudaFreeHost(c->h_resp); cudaFreeHost(c->h_totals);
    cudaFreeHost(c->h_run_tile_base);
    for (int i = 0; i <= kMaxStages; i++) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int b2_ctx_create(const b2_options* o, b2_ctx** out) {
    if (!o || !out) { set_err("null argument"); return B2_E_INVAL; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_err("no CUDA device: brpc_b200 has no CPU path"); return B2_E_NO_DEVICE;
    }
    if (o->device < 0 || o->device >= ndev) { set_err("bad device ordinal"); return B2_E_INVAL; }
    if (o->max_batch_bytes == 0 || o->max_batch_bytes >= (1u << 31) || o->max_msgs == 0 || o->max_runs == 0) {
        set_err("capacities must be non-zero and max_batch_bytes < 2 GiB"); return B2_E_INVAL;
    }
    CU(cudaSetDevice(o->device));
    b2_ctx* c = new b2_ctx();
    { int v = 148; cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, o->device); c->n_sms = (uint32_t)v; }
    for (int i = 0; i <= kMaxStages; i++) c->ev[i] = nullptr;
    c->opt = *o;
    c->adaptive_tile = o->tile_bytes == 0;
    uint32_t tile = o->tile_bytes ? o->tile_bytes : 8192;
    if (tile < 512 || (tile & (tile - 1))) { delete c; set_err("tile_bytes must be a power of two >= 512"); return B2_E_INVAL; }
    c->opt.tile_bytes = tile;
    if (c->opt.max_resp_bytes == 0) {
        uint64_t r = (uint64_t)o->max_batch_bytes + (uint64_t)o->max_msgs * 64 + (1u << 20);
        c->opt.max_resp_bytes = r > 0xfffffff0ull ? 0xfffffff0u : (uint32_t)r;
    }
    memset(&c->cfg, 0, sizeof c->cfg);
    c->cfg.max_body_size = o->max_body_size ? o->max_body_size : (64ull << 20);
    c->cfg.proto_mask = kProtoMaskDefault;
    c->cfg.tile_bytes = tile;
    c->cfg.tile_shift = 0; while ((1u << c->cfg.tile_shift) < tile) c->cfg.tile_shift++;
    c->max_tiles = o->max_batch_bytes / tile + o->max_runs + 1;
    const uint32_t scan_blocks = o->max_msgs / (kScanBlock * kScanItems) + 2;
#define ALLOC(ptr, bytes) do { if (cudaMalloc((void**)&(ptr), (bytes)) != cudaSuccess) { set_err("cudaMalloc %s failed", #ptr); b2_ctx_destroy(c); return B2_E_NOMEM; } } while (0)
#define HALLOC(ptr, bytes) do { if (cudaHostAlloc((void**)&(ptr), (bytes), cudaHostAllocDefault) != cudaSuccess) { set_err("cudaHostAlloc %s failed", #ptr); b2_ctx_destroy(c); return B2_E_NOMEM; } } while (0)
    ALLOC(c->d_bytes, (size_t)o->max_batch_bytes + 1024);
    ALLOC(c->d_runs, sizeof(b2_run) * (size_t)o->max_runs);
    ALLOC(c->d_run_tile_base, 4 * ((size_t)o->max_runs + 1));
    ALLOC(c->d_tiles, sizeof(TileRec) * (size_t)c->max_tiles);
    ALLOC(c->d_tile_base, 4 * (size_t)c->max_tiles);
    ALLOC(c->d_tile_scratch, 12 * (size_t)c->max_tiles);
    {   // kSpecK offsets per tile; dense mode (tiles >= 2 KiB holding many small frames) keeps kSpecKDense
        size_t dense_tiles = (size_t)o->max_batch_bytes / 2048 + o->max_runs + 1; if (dense_tiles > c->max_tiles) dense_tiles = c->max_tiles;
        size_t words = (size_t)kSpecK * c->max_tiles; if ((size_t)kSpecKDense * dense_tiles > words) words = (size_t)kSpecKDense * dense_tiles;
        ALLOC(c->d_tile_spec, 4 * words);
    }
    ALLOC(c->d_run_status, sizeof(b2_run_status) * (size_t)o->max_runs);
    ALLOC(c->d_frame_off, 4 * (size_t)o->max_msgs);
    ALLOC(c->d_frame_run, 4 * (size_t)o->max_msgs);
    ALLOC(c->d_msgs, sizeof(b2_msg_desc) * (size_t)o->max_msgs);
    ALLOC(c->d_aux, sizeof(MsgAux) * (size_t)o->max_msgs);
    ALLOC(c->d_jobs, sizeof(PackJob) * (size_t)o->max_msgs);
    ALLOC(c->d_refs, sizeof(uint4) * (size_t)o->max_msgs);
    ALLOC(c->d_slow_idx, sizeof(uint32_t) * (size_t)o->max_msgs);
    ALLOC(c->d_heads, (size_t)kHeadBytes * (size_t)o->max_msgs);
    ALLOC(c->d_slot, 4 * ((size_t)o->max_msgs + 1));
    ALLOC(c->d_scan_tmp, 4 * (size_t)scan_blocks);
    ALLOC(c->d_resp, (size_t)c->opt.max_resp_bytes + 1024);
    ALLOC(c->d_unz, 2 * (size_t)c->opt.max_resp_bytes + 1024);
    ALLOC(c->d_snappy_tab, (size_t)kSnappyWarps * kSnappyMaxTable * 2);
    ALLOC(c->d_hpack, sizeof(HpackState) * (size_t)B2_HPACK_MAX_CONNS);
    CU(cudaMemset(c->d_hpack, 0, sizeof(HpackState) * (size_t)B2_HPACK_MAX_CONNS));
    ALLOC(c->d_counters, 8 * B2_N_COUNTERS);
    ALLOC(c->d_totals, 64);
    ALLOC(c->d_methods, sizeof(DevMethod) * 64);
    ALLOC(c->d_crc_adv, (kCrcHotWords + kCrcTreeWords) * 4);
    ALLOC(c->d_meta, (size_t)o->max_runs * 28 + 16 * (size_t)c->max_tiles + 64);
    ALLOC(c->d_small, kSmallBlock);
    HALLOC(c->h_meta, (size_t)o->max_runs * 28 + 16 * (size_t)c->max_tiles + 64);
    HALLOC(c->h_small, kSmallBlock);
    HALLOC(c->h_run_status, sizeof(b2_run_status) * (size_t)o->max_runs);
    HALLOC(c->h_msgs, sizeof(b2_msg_desc) * (size_t)o->max_msgs);
    HALLOC(c->h_refs, sizeof(b2_resp_ref) * (size_t)o->max_msgs);
    HALLOC(c->h_resp, (size_t)c->opt.max_resp_bytes);
    HALLOC(c->h_totals, 64);
    HALLOC(c->h_run_tile_base, 4 * ((size_t)o->max_runs + 1));
    CU(cudaMemset(c->d_counters, 0, 8 * B2_N_COUNTERS));
    CU(cudaMemset(c->d_bytes, 0, (size_t)o->max_batch_bytes + 1024));
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (int i = 0; i <= kMaxStages; i++) CU(cudaEventCreate(&c->ev[i]));
    CU(cudaEventCreate(&c->ev_first)); CU(cudaEventCreate(&c->ev_last));
    crc_table_init();
    CU(cudaMemcpyToSymbol(c_crc_table, g_crc_tab_host, sizeof g_crc_tab_host));
    {   // warp-CRC tables: T[k][b] = byte b followed by k zero bytes (k = 0..15), A512 = advance by 512 zero bytes,
        // tree t = advance by 16 << t zero bytes; the advance operators are stored byte-sliced (4 x 256)
        std::vector<uint32_t> tab(kCrcHotWords + kCrcTreeWords);
        auto adv = [&](uint32_t x, int bytes) { for (int k = 0; k < bytes; k++) x = g_crc_tab_host[x & 0xff] ^ (x >> 8); return x; };
        for (int k = 0; k < 16; k++) for (uint32_t b = 0; b < 256; b++) tab[k * 256 + b] = adv(g_crc_tab_host[b], k);
        for (int j = 0; j < 4; j++) for (uint32_t b = 0; b < 256; b++) tab[(16 + j) * 256 + b] = adv(b << (8 * j), 512);
        for (int t = 0; t < 5; t++) for (int j = 0; j < 4; j++) for (uint32_t b = 0; b < 256; b++)
            tab[kCrcHotWords + (t * 4 + j) * 256 + b] = adv(b << (8 * j), 16 << t);
        CU(cudaMemcpy(c->d_crc_adv, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
    }
    CU(cudaFuncSetAttribute(k_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CU(cudaFuncSetAttribute(k_pack_slow<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(8 * kSnapRing)));
    CU(cudaFuncSetAttribute(k_pack_tma<kPackGroup>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(PackWarpSmem) * kPackWarps)));
    CU(cudaFuncSetAttribute(k_pack_tma<kPackGroupSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(PackWarpSmem) * kPackWarps)));
    if (const char* e = getenv("B2_PACK")) c->use_tma_pack = strcmp(e, "reg") != 0;
    if (const char* e = getenv("B2_SMALL")) c->use_fused_small = strcmp(e, "off") != 0;
    if (const char* e = getenv("B2_FUSED")) c->use_fused = strcmp(e, "off") != 0;
    CU(cudaFuncSetAttribute(k_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(FusedWarpSmem) * kFusedWarps)));
    CU(cudaFuncSetAttribute(k_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmallSmem)));
    *out = c;
    return B2_OK;
}

extern "C" int b2_set_server_identity(b2_ctx* c, const char* ip_port) {
    if (!c) return B2_E_INVAL;
    const size_t n = ip_port ? strlen(ip_port) : 0;
    if (n >= sizeof c->cfg.identity) { set_err("identity too long"); return B2_E_INVAL; }
    memset(c->cfg.identity, 0, sizeof c->cfg.identity);
    if (n) memcpy(c->cfg.identity, ip_port, n);
    c->cfg.identity_len = (uint32_t)n;
    return B2_OK;
}

extern "C" int b2_set_modes(b2_ctx* c, int input_mode, int resp_mode) {
    if (!c || (input_mode != B2_INPUT_COPY && input_mode != B2_INPUT_PULL) || (resp_mode != B2_RESP_COPY && resp_mode != B2_RESP_BY_REF && resp_mode != B2_RESP_IOVEC)) { set_err("bad mode"); return B2_E_INVAL; }
    static_assert(sizeof(b2_resp_ref) == sizeof(uint4), "b2_resp_ref is 16 bytes");
    static_assert(sizeof(b2_iovec) == sizeof(ulonglong2) && sizeof(void*) == 8, "b2_iovec is a 16-byte struct iovec");
    if (resp_mode == B2_RESP_IOVEC && !c->d_iov) {
        CU(cudaSetDevice(c->opt.device));
        if (cudaMalloc((void**)&c->d_iov, 32 * (size_t)c->opt.max_msgs) != cudaSuccess || cudaHostAlloc((void**)&c->h_iov, 32 * (size_t)c->opt.max_msgs, cudaHostAllocDefault) != cudaSuccess) {
            cudaFree(c->d_iov); c->d_iov = nullptr; cudaGetLastError(); set_err("allocation of the iovec list failed"); return B2_E_NOMEM;
        }
    }
    if (input_mode == B2_INPUT_PULL && !c->d_rows) {
        // row stash of the pull walk: spec_k rows of 128 bytes per tile (tiles are >= 32 KiB in this mode unless the caller fixed them)
        CU(cudaSetDevice(c->opt.device));
        const uint32_t tile = c->adaptive_tile ? 32768u : c->opt.tile_bytes;
        const size_t tiles = (size_t)c->opt.max_batch_bytes / tile + c->opt.max_runs + 1;
        const size_t rows = tiles * (tile >= 2048 ? kSpecKDense : kSpecK);
        if (cudaMalloc((void**)&c->d_rows, rows * 128) != cudaSuccess || cudaMalloc((void**)&c->d_frame_row, 4 * (size_t)c->opt.max_msgs) != cudaSuccess) {
            cudaFree(c->d_rows); c->d_rows = nullptr; cudaGetLastError(); set_err("cudaMalloc of the pull-mode row stash failed"); return B2_E_NOMEM;
        }
    }
    ring_halt(c);
    c->input_mode = input_mode; c->resp_mode = resp_mode; c->cfg.by_ref = resp_mode != B2_RESP_COPY; c->cfg.pull = input_mode == B2_INPUT_PULL; c->cfg.pull_vecs = resp_mode != B2_RESP_COPY ? 6u : 8u;
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

extern "C" int b2_set_protocols(b2_ctx* c, uint32_t mask) {
    const uint32_t known = (1u << 1) | (1u << 2) | (1u << 3) | (1u << 4) | (1u << 12);
    if (!c || mask == 0 || (mask & ~known)) { set_err("unknown protocol in mask (baidu_std 1, streaming_rpc 2, hulu_pbrpc 3, sofa_pbrpc 4, nshead 12)"); return B2_E_INVAL; }
    ring_halt(c);
    c->cfg.proto_mask = mask;
    return B2_OK;
}

extern "C" int b2_set_stream_handler(b2_ctx* c, int kind) {
    if (!c || (kind != B2_STREAM_DESC_ONLY && kind != B2_STREAM_SNAPPY_UNCOMPRESS)) { set_err("bad stream handler"); return B2_E_INVAL; }
    c->cfg.stream_handler = (uint32_t)kind;
    return B2_OK;
}

extern "C" int b2_register_method(b2_ctx* c, const b2_method* m) {
    if (!c || !m || !m->service_full_name || !m->service_name || !m->method_name || !m->request_type_name) { set_err("null argument"); return B2_E_INVAL; }
    if (c->methods.size() >= 64) { set_err("method table full"); return B2_E_CAPACITY; }
    DevMethod d; memset(&d, 0, sizeof d);
    std::string full = std::string(m->service_full_name) + "." + m->method_name;
    if (full.size() >= sizeof d.full_method || strlen(m->service_name) >= sizeof d.service_short ||
        strlen(m->service_full_name) >= sizeof d.service_full || strlen(m->request_type_name) >= sizeof d.request_type) {
        set_err("method names too long"); return B2_E_INVAL;
    }
    memcpy(d.full_method, full.data(), full.size()); d.full_method_len = (uint32_t)full.size();
    d.service_short_len = (uint32_t)strlen(m->service_name); memcpy(d.service_short, m->service_name, d.service_short_len);
    d.service_full_len = (uint32_t)strlen(m->service_full_name); memcpy(d.service_full, m->service_full_name, d.service_full_len);
    d.request_type_len = (uint32_t)strlen(m->request_type_name); memcpy(d.request_type, m->request_type_name, d.request_type_len);
    d.handler = m->handler; d.echo_attachment = m->echo_attachment;
    d.response_checksum_type = m->response_checksum_type; d.response_compress_type = m->response_compress_type;
    ring_halt(c);                                  // (DevConfig is a launch argument of the resident kernel)
    c->methods.push_back(d);
    c->cfg.n_methods = (uint32_t)c->methods.size();
    CU(cudaSetDevice(c->opt.device));
    CU(cudaMemcpy(c->d_methods, c->methods.data(), sizeof(DevMethod) * c->methods.size(), cudaMemcpyHostToDevice));
    return (int)c->methods.size() - 1;
}

static BatchPtrs make_ptrs(b2_ctx* c) {
    BatchPtrs B;
    B.bytes = c->d_bytes; B.runs = c->d_runs; B.run_tile_base = c->d_run_tile_base; B.tiles = c->d_tiles;
    B.tile_base = c->d_tile_base; B.tile_scratch = c->d_tile_scratch; B.tile_spec = c->d_tile_spec; B.run_status = c->d_run_status; B.frame_off = c->d_frame_off; B.frame_run = c->d_frame_run; B.frame_row = c->d_frame_row; B.rows = c->d_rows; B.msgs = c->d_msgs;
    B.aux = c->d_aux; B.jobs = c->d_jobs; B.refs = c->d_refs; B.slow_idx = c->d_slow_idx; B.heads = c->d_heads; B.slot = c->d_slot; B.scan_tmp = c->d_scan_tmp; B.resp = c->d_resp; B.unz = c->d_unz; B.snappy_tab = c->d_snappy_tab; B.counters = c->d_counters;
    B.totals = c->d_totals; B.methods = c->d_methods; B.crc_adv = c->d_crc_adv;
    B.n_runs = c->n_runs; B.n_tiles = c->n_tiles; B.max_msgs = c->opt.max_msgs; B.max_resp = c->opt.max_resp_bytes;
    B.runs = reinterpret_cast<const b2_run*>(c->d_meta);
    B.run_tile_base = reinterpret_cast<const uint32_t*>(c->d_meta + (size_t)c->n_runs * sizeof(b2_run));
    B.tile_info = reinterpret_cast<const uint4*>(c->d_meta + c->meta_tile_off);
    if (c->input_mode == B2_INPUT_PULL) B.bytes = c->pull_bytes;          // the caller's pinned + mapped batch buffer, read in place
    if (c->small) {
        B.refs = reinterpret_cast<uint4*>(c->d_small + c->small_off_refs);
        B.totals = reinterpret_cast<uint32_t*>(c->d_small);
        B.run_status = reinterpret_cast<b2_run_status*>(c->d_small + c->small_off_rs);
        B.msgs = reinterpret_cast<b2_msg_desc*>(c->d_small + c->small_off_msgs);
        B.resp = c->d_small + c->small_off_resp;
        B.max_msgs = c->small_msgs; B.max_resp = c->small_resp;
    }
    return B;
}

extern "C" int b2_batch_upload(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs) {
    if (!c || (!bytes && nbytes) || (!runs && n_runs)) { set_err("null argument"); return B2_E_INVAL; }
    // (B2_INPUT_PULL: `bytes` is the caller's whole pinned arena and nothing is copied — what is bounded is the bytes the runs cover)
    if ((c->input_mode != B2_INPUT_PULL && nbytes > c->opt.max_batch_bytes) || nbytes >= (1u << 31) || n_runs > c->opt.max_runs) { set_err("batch exceeds ctx capacity"); return B2_E_CAPACITY; }
    uint64_t covered = 0; for (uint32_t r = 0; r < n_runs; r++) covered += runs[r].length;
    if (c->input_mode == B2_INPUT_PULL && covered > c->opt.max_batch_bytes) { set_err("runs exceed ctx capacity"); return B2_E_CAPACITY; }
    c->covered = covered;                           // (what the runs hold: with B2_INPUT_PULL nbytes spans the caller's whole arena)
    CU(cudaSetDevice(c->opt.device));
    if (c->adaptive_tile) {
        // like Socket::_avg_msg_size steering the read size (input_messenger.cpp:348-353): a tile should hold
        // 6-12 messages so the speculative entry search reads a small fraction of it
        uint32_t t = 8192;
        // (B2_INPUT_PULL: the speculative scan window of every tile crosses PCIe, so tiles are 4x larger)
        const uint32_t per_tile = c->input_mode == B2_INPUT_PULL ? 48u : 6u;
        if (c->input_mode == B2_INPUT_PULL && t < 32768) t = 32768;
        while (t < (1u << 20) && t < per_tile * c->avg_frame) t <<= 1;
        c->cfg.tile_bytes = t; c->cfg.tile_shift = 0; while ((1u << c->cfg.tile_shift) < t) c->cfg.tile_shift++;
    }
    const uint32_t shift = c->cfg.tile_shift, tile = c->cfg.tile_bytes;
    // small requests (the previous batches' average says a tile holds more than kSpecK frames): k_tile_walk keeps longer offset
    // lists so that k_frame_table still only copies (a measured 139 -> 29 us for 124-byte frames)
    c->dense = tile >= 2048 && c->avg_frame && (uint64_t)c->avg_frame * kSpecK < tile;
    c->cfg.spec_k = c->dense ? kSpecKDense : kSpecK;
    uint64_t nt = 0; uint32_t max_rt = 0;
    for (uint32_t r = 0; r < n_runs; r++) {
        if ((runs[r].offset & 15u) || (uint64_t)runs[r].offset + runs[r].length > nbytes) { set_err("run offset must be 16-aligned and inside the batch"); return B2_E_INVAL; }
        c->h_run_tile_base[r] = (uint32_t)nt;
        const uint32_t t = (uint32_t)(((uint64_t)runs[r].length + tile - 1) >> shift);
        nt += t; if (t > max_rt) max_rt = t;
    }
    c->h_run_tile_base[n_runs] = (uint32_t)nt;
    if (nt > c->max_tiles) { set_err("too many tiles"); return B2_E_CAPACITY; }
    c->n_runs = n_runs; c->n_tiles = (uint32_t)nt; c->nbytes = nbytes; c->max_run_tiles = max_rt; c->host_bytes = bytes;
    // runs + tile bases travel as one compact block (24 B * n is 4-byte aligned)
    const size_t tile_off = ((size_t)n_runs * sizeof(b2_run) + 4 * ((size_t)n_runs + 1) + 15) & ~(size_t)15;
    const size_t meta_bytes = tile_off + 16 * (size_t)nt;
    c->meta_tile_off = tile_off;
    if (n_runs) memcpy(c->h_meta, runs, (size_t)n_runs * sizeof(b2_run));
    memcpy(c->h_meta + (size_t)n_runs * sizeof(b2_run), c->h_run_tile_base, 4 * ((size_t)n_runs + 1));
    {   // per-tile record {run offset, run length, tile index in the run, run | flags << 24}: one load per tile thread
        uint32_t* ti = reinterpret_cast<uint32_t*>(c->h_meta + tile_off);
        for (uint32_t r = 0; r < n_runs; r++) {
            const uint32_t t0 = c->h_run_tile_base[r], t1 = c->h_run_tile_base[r + 1];
            for (uint32_t t = t0; t < t1; t++) { uint32_t* q = ti + 4 * (size_t)t; q[0] = runs[r].offset; q[1] = runs[r].length; q[2] = t - t0; q[3] = r | (runs[r].flags << 24); }
        }
    }
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    if (c->input_mode == B2_INPUT_PULL) {
        // no copy: the kernels read the caller's pinned block in place (it must stay untouched until collect)
        void* dp = nullptr;
        if (nbytes && cudaHostGetDevicePointer(&dp, const_cast<void*>(bytes), 0) != cudaSuccess) {
            cudaGetLastError(); set_err("B2_INPUT_PULL: bytes must be pinned + mapped memory from b2_block_alloc"); return B2_E_INVAL;
        }
        c->pull_bytes = static_cast<const uint8_t*>(dp);
    } else if (nbytes) CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_meta, c->h_meta, meta_bytes, cudaMemcpyHostToDevice, c->stream));
    // latency path: outputs of a small batch live in one compact block -> one D2H copy, one sync
    c->small = c->allow_small && nbytes <= kSmallBytes && n_runs <= kSmallRuns && n_runs > 0;
    if (c->small) {
        uint32_t mb = nbytes / 12 + 1; if (mb > kSmallMsgs) mb = kSmallMsgs;
        if (mb > c->opt.max_msgs) mb = c->opt.max_msgs;      // d_frame_off / d_aux / d_jobs / d_heads ... are sized by opt.max_msgs
        c->small_msgs = mb; c->small_resp = nbytes + mb * 80 + 2048;
        c->small_off_rs = 64; c->small_off_msgs = 64 + n_runs * 32; c->small_off_refs = c->small_off_msgs + mb * 64;
        c->small_off_resp = (c->small_off_refs + mb * 16 + 255u) & ~255u;
        c->small_total = c->small_off_resp + c->small_resp;
    }
    if (const char* e = getenv("B2_STAGE_MASK")) c->stage_mask = (uint32_t)atoi(e);   // timing experiments only (tools/overlap_probe.py)
    c->uploaded = true; c->executed = false;
    return B2_OK;
}

static int launch_pipeline(b2_ctx* c) {
    const BatchPtrs B = make_ptrs(c);
    DevConfig C = c->cfg;
    // the fused decode+pack kernel serves batches whose bytes and replies both live in HBM
    const bool fused = c->use_fused && !c->slow_heavy && !c->small && c->input_mode == B2_INPUT_COPY && c->resp_mode == B2_RESP_COPY && c->use_tma_pack &&
                       (((uint64_t)c->nbytes + 255) & ~255ull) + 4096 <= c->opt.max_resp_bytes;
    C.fused = fused ? 1u : 0u; C.ovf_base = (c->nbytes + 255u) & ~255u; c->fused_last = fused;
    cudaStream_t s = c->stream;
    int st = 0; uint32_t launches = 0;
    const bool prof = c->profile_stages;
    auto mark = [&](const char* name) { if (prof) { c->stage_names[st] = name; cudaEventRecord(c->ev[st + 1], s); st++; } };
    const uint32_t mask = c->stage_mask;
    if (mask & 1) CU(cudaMemsetAsync(B.totals, 0, 48, s));
    CU(cudaEventRecord(c->ev[0], s));
    if (c->n_runs == 0) { c->n_stages = 0; c->last_launches = 0; return B2_OK; }
    if (c->small && c->use_fused_small && !prof) {
        // latency path: the whole pipeline in one launch, one CTA
        k_small<<<1, kSmallThreads, sizeof(SmallSmem), s>>>(B, C);
        c->stage_names[0] = "fused_small"; cudaEventRecord(c->ev[1], s);
        c->n_stages = 1; c->last_launches = 1;
        CU(cudaGetLastError());
        return B2_OK;
    }
    const uint32_t sms = c->n_sms;
    if (mask & 1) {
    if (c->n_tiles) {
        k_tile_search<<<(c->n_tiles * 32 + 255) / 256, 256, 0, s>>>(B, C); launches++; mark("tile_search");
        if (C.pull) k_tile_walk_pull<<<(uint32_t)(((uint64_t)c->n_tiles * 8 + 127) / 128), 128, 0, s>>>(B, C);
        else k_tile_walk<<<(c->n_tiles + 127) / 128, 128, 0, s>>>(B, C);
        launches++; mark("tile_walk");
    }
    {
        size_t smem = (size_t)c->max_run_tiles * 12;
        if (smem > 200 * 1024) smem = 0;                 // some run does not fit: EVERY run of this launch uses the global scratch
        k_resolve<<<c->n_runs, 256, smem, s>>>(B, C, smem == 0 ? 1u : 0u); launches++; mark("resolve");
    }
    if (fused) {
        // one pass over the bytes: decode + echo + pack per live tile (k_frame_table / k_decode / k_scan / k_pack_tma are not needed)
        if (c->n_tiles) { k_fused<<<sms, kFusedWarps * 32, sizeof(FusedWarpSmem) * kFusedWarps, s>>>(B, C); launches++; mark("fused"); }
    } else {
    if (c->n_tiles) { k_frame_table<<<(uint32_t)(((uint64_t)c->n_tiles * C.spec_k + 255) / 256), 256, 0, s>>>(B, C); launches++; mark("frame_table"); }
    // message-count dependent kernels are persistent: fixed grids (multiples of the SM count)
    // stride over the device-side message count, so no host round trip sizes a launch
    k_decode<<<sms * B2_DECODE_MIN_BLOCKS, kDecodeWarps * 32, 0, s>>>(B, C); launches++; mark("decode");
    k_scan_blocks<<<sms, kScanBlock, 0, s>>>(B); launches++;
    mark("scan");
    }
    }
    if (fused) {
        if (mask & 4) { k_pack_slow<true><<<sms * B2_SLOW_MIN_BLOCKS, 256, 0, s>>>(B, C); launches++; mark("pack_slow"); }
    } else if (c->use_tma_pack) {
        // the verify pass decides which CRC-carrying echoes k_pack_tma may move; k_pack_slow answers the ones that fail
        if (mask & 4) {
            if (c->slow_heavy || c->cfg.by_ref) { C.verify_done = 1; k_crc_verify<<<sms * 6, 256, 0, s>>>(B, C); launches++; mark("crc_verify"); }
            k_pack_slow<false><<<sms * B2_SLOW_MIN_BLOCKS, 256, 8 * kSnapRing, s>>>(B, C); launches++; mark("pack_slow");
        }
        if (mask & 2) {
            // small requests: 32 messages per warp round instead of 8 (measured +30 % at 64 B payloads, -3 % at 1 KB)
            if ((c->avg_frame && c->avg_frame < 640) || c->cfg.by_ref) k_pack_tma<kPackGroupSmall><<<sms, kPackWarps * 32, sizeof(PackWarpSmem) * kPackWarps, s>>>(B, C);
            else k_pack_tma<kPackGroup><<<sms, kPackWarps * 32, sizeof(PackWarpSmem) * kPackWarps, s>>>(B, C);
            launches++; mark("pack");
        }
    } else { k_pack<<<sms * B2_PACK_MIN_BLOCKS, 256, 0, s>>>(B, C); launches++; mark("pack"); }
    if (c->resp_mode == B2_RESP_IOVEC && !c->small) {
        k_emit_iov<<<sms * 4, 256, 0, s>>>(B, c->d_iov, (unsigned long long)(uintptr_t)c->h_resp, (unsigned long long)(uintptr_t)c->host_bytes);
        launches++; mark("emit_iov");
    }
    if (!prof) { c->stage_names[0] = "pipeline"; cudaEventRecord(c->ev[1], s); st = 1; }
    c->n_stages = st; c->last_launches = launches;
    CU(cudaGetLastError());
    return B2_OK;
}

extern "C" int b2_batch_execute(b2_ctx* c, float* kernel_ms, uint32_t* n_launches) {
    if (!c || !c->uploaded) { set_err("no batch uploaded"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    c->profile_stages = true;
    int rc = launch_pipeline(c);
    c->profile_stages = false;
    if (rc != B2_OK) return rc;
    CU(cudaStreamSynchronize(c->stream));
    float ms = 0.f;
    if (c->n_stages) CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[c->n_stages]));
    c->last_kernel_ms = ms; c->executed = true;
    if (kernel_ms) *kernel_ms = ms;
    if (n_launches) *n_launches = c->last_launches;
    return B2_OK;
}

extern "C" int b2_batch_execute_many(b2_ctx* c, uint32_t steps, float* total_ms, uint32_t* n_launches) {
    if (!c || !c->uploaded || steps == 0) { set_err("no batch uploaded"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, c->stream));
    uint32_t launches = 0;
    for (uint32_t i = 0; i < steps; i++) {
        int rc = launch_pipeline(c);
        if (rc != B2_OK) return rc;
        launches += c->last_launches;
    }
    CU(cudaEventRecord(e1, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    c->executed = true;
    if (c->n_stages) { float t = 0.f; cudaEventElapsedTime(&t, c->ev[0], c->ev[c->n_stages]); c->last_kernel_ms = t; }
    if (total_ms) *total_ms = ms;
    if (n_launches) *n_launches = launches;
    return B2_OK;
}

extern "C" int b2_batch_launch(b2_ctx* c) {
    if (!c || !c->uploaded) { set_err("no batch uploaded"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    if (c->first_pending) { CU(cudaEventRecord(c->ev_first, c->stream)); c->first_pending = false; }
    int rc = launch_pipeline(c);
    if (rc != B2_OK) return rc;
    CU(cudaEventRecord(c->ev_last, c->stream));
    c->executed = true;
    return B2_OK;
}
extern "C" int b2_batch_wait(b2_ctx* c) {
    if (!c) return B2_E_INVAL;
    CU(cudaSetDevice(c->opt.device));
    CU(cudaStreamSynchronize(c->stream));
    c->first_pending = true;
    return B2_OK;
}
extern "C" int b2_elapsed_ms(b2_ctx* a, b2_ctx* b, float* ms) {
    if (!a || !b || !ms) return B2_E_INVAL;
    CU(cudaSetDevice(a->opt.device));
    CU(cudaEventElapsedTime(ms, a->ev_first, b->ev_last));
    return B2_OK;
}

// B2_RESP_IOVEC on the latency path (a handful of messages in one compact block): the list is built here from the refs that came back
static void refs_to_iov(b2_ctx* c, b2_batch_result* out, const void* host_bytes) {
    b2_run_status* rs = const_cast<b2_run_status*>(out->runs);
    for (uint32_t r = 0; r < out->n_runs; r++) rs[r].n_unanswered = 0;
    for (uint32_t i = 0; i < out->n_msgs; i++) {
        const b2_msg_desc& d = out->msgs[i];
        b2_iovec a = { const_cast<uint8_t*>(out->resp), 0 }, b = a;
        if (d.status == B2_MSG_ECHOED || d.status == B2_MSG_ERROR_REPLIED) {
            const b2_resp_ref rf = d.status == B2_MSG_ECHOED ? out->refs[i] : b2_resp_ref{0, 0, 0, 0};
            a.iov_base = const_cast<uint8_t*>(out->resp) + d.resp_off; a.iov_len = rf.src_len ? rf.prefix_len : d.resp_len;
            if (rf.src_len) { b.iov_base = const_cast<uint8_t*>(static_cast<const uint8_t*>(host_bytes)) + rf.src_off; b.iov_len = rf.src_len; }
        } else rs[d.run_idx].n_unanswered++;
        c->h_iov[2 * (size_t)i] = a; c->h_iov[2 * (size_t)i + 1] = b;
    }
    out->iov = c->h_iov; out->refs = nullptr;
}

static int download_normal(b2_ctx* c, b2_batch_result* out) {
    CU(cudaMemcpyAsync(c->h_totals, c->d_totals, 48, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (c->n_runs && c->fused_last) {
        // the fused kernel keeps slow replies in an overflow area behind the batch-shaped part of resp: traffic that is mostly
        // CRC'd / compressed / errors is better served (and may only fit) through the slot-scan pipeline
        const bool heavy = (uint64_t)c->h_totals[3] * 8 > c->h_totals[0];
        if ((c->h_totals[2] & 2u) && !(c->h_totals[2] & 1u)) {
            c->slow_heavy = true;
            int rc = launch_pipeline(c); if (rc != B2_OK) return rc;
            CU(cudaMemcpyAsync(c->h_totals, c->d_totals, 48, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
        }
        c->slow_heavy = heavy || c->slow_heavy;
    } else if (c->n_runs && c->slow_heavy && !c->small) {
        c->slow_heavy = ((uint64_t)c->h_totals[3] + c->h_totals[7]) * 8 > c->h_totals[0];   // ([7]: CRC-carrying echoes the classic pipeline verifies)
    }
    if (c->n_runs && (c->h_totals[2] & 3u)) {
        set_err(c->h_totals[2] & 1u ? "more messages than max_msgs" : "responses exceed max_resp_bytes"); return B2_E_CAPACITY;
    }
    // (k_fused / k_pack_slow: replies of parked messages are placed after the kernel's own end-of-area note, so the span is taken from the allocator)
    if (c->n_runs && c->fused_last) c->h_totals[1] = ((c->nbytes + 255u) & ~255u) + c->h_totals[9];
    const uint32_t n_msgs = c->n_runs ? c->h_totals[0] : 0, resp_bytes = c->n_runs ? c->h_totals[1] : 0;
    if (c->n_runs) CU(cudaMemcpyAsync(c->h_run_status, c->d_run_status, sizeof(b2_run_status) * c->n_runs, cudaMemcpyDeviceToHost, c->stream));
    if (n_msgs) CU(cudaMemcpyAsync(c->h_msgs, c->d_msgs, sizeof(b2_msg_desc) * (size_t)n_msgs, cudaMemcpyDeviceToHost, c->stream));
    if (resp_bytes) CU(cudaMemcpyAsync(c->h_resp, c->d_resp, resp_bytes, cudaMemcpyDeviceToHost, c->stream));
    const bool iovec = c->resp_mode == B2_RESP_IOVEC;
    if (n_msgs && c->cfg.by_ref && !iovec) CU(cudaMemcpyAsync(c->h_refs, c->d_refs, sizeof(b2_resp_ref) * (size_t)n_msgs, cudaMemcpyDeviceToHost, c->stream));
    if (n_msgs && iovec) CU(cudaMemcpyAsync(c->h_iov, c->d_iov, 32 * (size_t)n_msgs, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    out->refs = c->cfg.by_ref && !iovec ? c->h_refs : nullptr;
    out->iov = iovec ? c->h_iov : nullptr;
    out->runs = c->h_run_status; out->n_runs = c->n_runs;
    out->msgs = c->h_msgs; out->n_msgs = n_msgs;
    out->resp = c->h_resp; out->resp_bytes = resp_bytes;
    return B2_OK;
}

extern "C" int b2_batch_download(b2_ctx* c, b2_batch_result* out) {
    if (!c || !out || !c->executed) { set_err("no executed batch"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    memset(out, 0, sizeof *out);
    if (c->small) {
        if (!c->small_copy_queued) CU(cudaMemcpyAsync(c->h_small, c->d_small, c->small_total, cudaMemcpyDeviceToHost, c->stream));
        c->small_copy_queued = false;
        CU(cudaStreamSynchronize(c->stream));
        const uint32_t* tot = reinterpret_cast<const uint32_t*>(c->h_small);
        if (tot[2] & 3u) {
            // more messages / response bytes than the compact block holds: redo on the normal path
            c->small = false;
            int rc = launch_pipeline(c);
            if (rc != B2_OK) return rc;
            rc = download_normal(c, out);
            if (rc != B2_OK) return rc;
        } else {
            out->runs = reinterpret_cast<const b2_run_status*>(c->h_small + c->small_off_rs); out->n_runs = c->n_runs;
            out->msgs = reinterpret_cast<const b2_msg_desc*>(c->h_small + c->small_off_msgs); out->n_msgs = tot[0];
            out->resp = c->h_small + c->small_off_resp; out->resp_bytes = tot[1];
            out->refs = c->cfg.by_ref ? reinterpret_cast<const b2_resp_ref*>(c->h_small + c->small_off_refs) : nullptr;
            if (c->resp_mode == B2_RESP_IOVEC) refs_to_iov(c, out, c->host_bytes);
        }
    } else {
        int rc = download_normal(c, out);
        if (rc != B2_OK) return rc;
    }
    if (out->n_msgs) { const uint32_t now = (uint32_t)(c->covered / out->n_msgs); c->avg_frame = c->avg_frame ? (uint32_t)(((uint64_t)c->avg_frame * 3 + now) / 4) : now; }
    out->kernel_ms = c->last_kernel_ms; out->n_launches = c->last_launches;
    return B2_OK;
}

extern "C" int b2_batch_submit(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs) {
    int rc = b2_batch_upload(c, bytes, nbytes, runs, n_runs);
    if (rc != B2_OK) return rc;
    rc = launch_pipeline(c);
    if (rc != B2_OK) return rc;
    c->executed = true;
    if (c->small) { CU(cudaMemcpyAsync(c->h_small, c->d_small, c->small_total, cudaMemcpyDeviceToHost, c->stream)); c->small_copy_queued = true; }
    return B2_OK;
}

extern "C" int b2_batch_collect(b2_ctx* c, b2_batch_result* out) {
    int rc = b2_batch_download(c, out);
    if (rc != B2_OK) return rc;
    float ms = 0.f;
    if (c->n_stages) CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[c->n_stages]));
    c->last_kernel_ms = ms; out->kernel_ms = ms;
    return B2_OK;
}

extern "C" int b2_process_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs,
                                b2_batch_result* out) {
    int rc = b2_batch_submit(c, bytes, nbytes, runs, n_runs);
    if (rc != B2_OK) return rc;
    return b2_batch_collect(c, out);
}


// ---- the persistent latency path: submit ring + resident kernel (k_ring) ---------------------------------------------------------
static void ring_halt(b2_ctx* c) {
    if (!c->ring_ctl) return;
    c->ring_ctl[0] = 1; __sync_synchronize();
    cudaStreamSynchronize(c->ring_stream);
    c->ring_ctl[0] = 0; c->ring_ctl[1] = 0; __sync_synchronize();
}
static int ring_launch(b2_ctx* c) {
    RingDev R;
    R.slots = c->ring_slots; R.slot_stride = c->ring_stride; R.off_runs = c->ring_off_runs; R.off_in = c->ring_off_in; R.off_out = c->ring_off_out;
    R.ctl = c->ring_ctl; R.next_ticket = c->d_ring_ticket;
    unsigned long long idle_ms = 20; if (const char* e = getenv("B2_RING_IDLE_MS")) idle_ms = (unsigned long long)atoi(e);
    R.idle_ns = idle_ms * 1000000ull;
    R.d_bytes = c->d_bytes; R.d_meta = c->d_meta; R.d_small = c->d_small;
    const bool was_small = c->small; c->small = false;
    BatchPtrs B = make_ptrs(c);
    c->small = was_small;
    B.bytes = c->d_bytes;
    c->ring_ctl[1] = 1; __sync_synchronize();
    k_ring<<<1, kSmallThreads, sizeof(SmallSmem), c->ring_stream>>>(R, B, c->cfg);
    c->ring_launches++;
    CU(cudaGetLastError());
    return B2_OK;
}
extern "C" int b2_ring_start(b2_ctx* c) {
    if (!c) return B2_E_INVAL;
    CU(cudaSetDevice(c->opt.device));
    if (!c->ring_slots) {
        c->ring_off_runs = sizeof(RingSlotHdr);
        c->ring_off_in = (c->ring_off_runs + kSmallRuns * (uint32_t)sizeof(b2_run) + 255u) & ~255u;
        c->ring_off_out = (c->ring_off_in + kSmallBytes + 1024u + 255u) & ~255u;
        c->ring_stride = (uint32_t)((c->ring_off_out + kSmallBlock + 4095u) & ~4095u);
        CU(cudaHostAlloc((void**)&c->ring_slots, (size_t)c->ring_stride * kRingSlots, cudaHostAllocMapped | cudaHostAllocPortable));
        memset(c->ring_slots, 0, (size_t)c->ring_stride * kRingSlots);
        CU(cudaHostAlloc((void**)&c->ring_ctl, 64, cudaHostAllocMapped | cudaHostAllocPortable));
        memset((void*)c->ring_ctl, 0, 64);
        CU(cudaMalloc((void**)&c->d_ring_ticket, 4));
        const uint32_t one = 1; CU(cudaMemcpy(c->d_ring_ticket, &one, 4, cudaMemcpyHostToDevice));
        CU(cudaStreamCreateWithFlags(&c->ring_stream, cudaStreamNonBlocking));
        CU(cudaFuncSetAttribute(k_ring, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmallSmem)));
    }
    if (!c->ring_ctl[1]) return ring_launch(c);
    return B2_OK;
}
extern "C" int b2_ring_stop(b2_ctx* c) { if (!c) return B2_E_INVAL; cudaSetDevice(c->opt.device); ring_halt(c); return B2_OK; }

extern "C" int b2_ring_submit(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs, uint32_t* ticket) {
    if (!c || !bytes || !runs || !ticket || n_runs == 0) { set_err("null argument"); return B2_E_INVAL; }
    if (nbytes > kSmallBytes || n_runs > kSmallRuns) { set_err("b2_ring_submit serves batches up to 128 KiB / 512 runs: use b2_batch_submit"); return B2_E_CAPACITY; }
    if (!c->ring_slots) { int rc = b2_ring_start(c); if (rc != B2_OK) return rc; }
    const uint32_t t = c->ring_next, si = t % kRingSlots;
    if (!c->ring_collected[si]) { set_err("submit ring full: b2_ring_wait the oldest ticket first"); return B2_E_CAPACITY; }
    for (uint32_t r = 0; r < n_runs; r++)
        if ((runs[r].offset & 15u) || (uint64_t)runs[r].offset + runs[r].length > nbytes) { set_err("run offset must be 16-aligned and inside the batch"); return B2_E_INVAL; }
    uint8_t* slot = c->ring_slots + (size_t)si * c->ring_stride;
    RingSlotHdr* h = reinterpret_cast<RingSlotHdr*>(slot);
    // the batch bytes: in place when they already live in pinned + mapped memory (b2_block_alloc), else staged into the slot
    unsigned long long dev = 0;
    if (bytes == c->ring_pin_base) dev = c->ring_pin_dev;
    else {
        cudaPointerAttributes at; memset(&at, 0, sizeof at);
        if (cudaPointerGetAttributes(&at, bytes) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
            dev = (unsigned long long)(uintptr_t)at.devicePointer; c->ring_pin_base = bytes; c->ring_pin_dev = dev;
        } else cudaGetLastError();
    }
    if (!dev) { memcpy(slot + c->ring_off_in, bytes, nbytes); dev = (unsigned long long)(uintptr_t)(slot + c->ring_off_in); }
    memcpy(slot + c->ring_off_runs, runs, sizeof(b2_run) * (size_t)n_runs);
    uint32_t mb = nbytes / 12 + 1; if (mb > kSmallMsgs) mb = kSmallMsgs; if (mb > c->opt.max_msgs) mb = c->opt.max_msgs;
    h->n_runs = n_runs; h->nbytes = nbytes; h->small_msgs = mb; h->small_resp = nbytes + mb * 80 + 2048;
    h->off_rs = 64; h->off_msgs = 64 + n_runs * 32; h->off_refs = h->off_msgs + mb * 64; h->off_resp = (h->off_refs + mb * 16 + 255u) & ~255u;
    h->total = h->off_resp + h->small_resp; h->by_ref = c->cfg.by_ref; h->bytes_dev = dev;
    c->ring_bytes[si] = bytes; c->ring_collected[si] = false;
    __sync_synchronize();
    h->submit = t;
    __sync_synchronize();
    c->ring_next = t + 1;
    *ticket = t;
    if (!c->ring_ctl[1]) { CU(cudaSetDevice(c->opt.device)); return ring_launch(c); }   // the kernel idled out (or was never started)
    return B2_OK;
}

extern "C" int b2_ring_wait(b2_ctx* c, uint32_t ticket, b2_batch_result* out) {
    if (!c || !out || !c->ring_slots || ticket == 0 || ticket >= c->ring_next || ticket + kRingSlots < c->ring_next) { set_err("bad ring ticket"); return B2_E_INVAL; }
    const uint32_t si = ticket % kRingSlots;
    uint8_t* slot = c->ring_slots + (size_t)si * c->ring_stride;
    RingSlotHdr* h = reinterpret_cast<RingSlotHdr*>(slot);
    if (c->ring_collected[si]) { set_err("ticket already collected"); return B2_E_INVAL; }
    uint64_t spins = 0;
    while (h->done != ticket) {
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((++spins & 0xfffff) == 0) {
            if (!c->ring_ctl[1]) { CU(cudaSetDevice(c->opt.device)); int rc = ring_launch(c); if (rc != B2_OK) return rc; }   // lost the exit race: start it again
            if (cudaStreamQuery(c->ring_stream) != cudaErrorNotReady && h->done != ticket && !c->ring_ctl[1]) continue;
            if (spins > (1ull << 34)) { set_err("ring kernel did not answer"); return B2_E_CUDA; }
        }
    }
    __sync_synchronize();
    c->ring_collected[si] = true;
    memset(out, 0, sizeof *out);
    const uint8_t* ob = slot + c->ring_off_out;
    const uint32_t* tot = reinterpret_cast<const uint32_t*>(ob);
    if (tot[2] & 3u) {
        // more messages / reply bytes than the compact block holds: the big pipeline serves this batch (after the ring is quiet)
        for (uint32_t k = 0; k < kRingSlots; k++) if (!c->ring_collected[k]) { set_err("ring overflow fallback needs the other tickets collected first"); return B2_E_CAPACITY; }
        ring_halt(c);
        const bool allow = c->allow_small; c->allow_small = false;
        const int rc = b2_process_batch(c, c->ring_bytes[si], h->nbytes, reinterpret_cast<const b2_run*>(slot + c->ring_off_runs), h->n_runs, out);
        c->allow_small = allow;
        return rc;
    }
    out->runs = reinterpret_cast<const b2_run_status*>(ob + h->off_rs); out->n_runs = h->n_runs;
    out->msgs = reinterpret_cast<const b2_msg_desc*>(ob + h->off_msgs); out->n_msgs = tot[0];
    out->resp = ob + h->off_resp; out->resp_bytes = tot[1];
    out->refs = h->by_ref ? reinterpret_cast<const b2_resp_ref*>(ob + h->off_refs) : nullptr;
    if (c->resp_mode == B2_RESP_IOVEC) refs_to_iov(c, out, c->ring_bytes[si]);
    out->n_launches = 0; out->kernel_ms = 0.f;
    if (out->n_msgs) { const uint32_t now = h->nbytes / out->n_msgs; c->avg_frame = c->avg_frame ? (uint32_t)(((uint64_t)c->avg_frame * 3 + now) / 4) : now; }
    return B2_OK;
}
extern "C" uint64_t b2_ring_launches(b2_ctx* c) { return c ? c->ring_launches : 0; }
// device-side phase times of a collected ticket, ns since the kernel saw the doorbell: [0] header read [1] runs + bytes pulled [2] cut / decode / pack done [3] results pushed
extern "C" int b2_ring_phase_ns(b2_ctx* c, uint32_t ticket, uint64_t out[4]) {
    if (!c || !c->ring_slots || !out) return B2_E_INVAL;
    const RingSlotHdr* h = reinterpret_cast<const RingSlotHdr*>(c->ring_slots + (size_t)(ticket % kRingSlots) * c->ring_stride);
    for (int k = 0; k < 4; k++) out[k] = h->stamps[k + 1] - h->stamps[0];
    return B2_OK;
}

// measurement helper: wall-clock microseconds of `iters` back-to-back calls, one batch each, timed inside the library so that
// the caller's language runtime is not part of the number (bench.py's latency line)
extern "C" int b2_latency_probe(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs, uint32_t iters, int use_ring, float* us_out) {
    if (!c || !us_out) return B2_E_INVAL;
    b2_batch_result res;
    for (uint32_t i = 0; i < iters; i++) {
        timespec t0, t1; clock_gettime(CLOCK_MONOTONIC, &t0);
        int rc;
        if (use_ring) { uint32_t t = 0; rc = b2_ring_submit(c, bytes, nbytes, runs, n_runs, &t); if (rc == B2_OK) rc = b2_ring_wait(c, t, &res); }
        else rc = b2_process_batch(c, bytes, nbytes, runs, n_runs, &res);
        clock_gettime(CLOCK_MONOTONIC, &t1);
        if (rc != B2_OK) return rc;
        if (res.n_msgs == 0) { set_err("latency probe batch produced no messages"); return B2_E_INVAL; }
        us_out[i] = (float)((t1.tv_sec - t0.tv_sec) * 1e6 + (t1.tv_nsec - t0.tv_nsec) * 1e-3);
    }
    return B2_OK;
}

extern "C" int b2_stage_times(b2_ctx* c, const char** names, float* ms, int cap) {
    if (!c) return B2_E_INVAL;
    int n = c->n_stages < cap ? c->n_stages : cap;
    for (int i = 0; i < n; i++) {
        names[i] = c->stage_names[i];
        float t = 0.f;
        cudaEventElapsedTime(&t, c->ev[i], c->ev[i + 1]);
        ms[i] = t;
    }
    return c->n_stages;
}

// what the last upload / launch decided: [0] tile bytes [1] tiles [2] frame offsets kept per tile [3] 1 = the fused kernel served it
extern "C" int b2_batch_info(b2_ctx* c, uint32_t out[4]) {
    if (!c || !out) return B2_E_INVAL;
    out[0] = c->cfg.tile_bytes; out[1] = c->n_tiles; out[2] = c->cfg.spec_k; out[3] = c->fused_last ? 1u : 0u;
    return B2_OK;
}

extern "C" int b2_device_pci_bus_id(int device, char* out, int cap) {
    if (!out || cap < 13) return B2_E_INVAL;
    if (cudaDeviceGetPCIBusId(out, cap, device) != cudaSuccess) { cudaGetLastError(); return B2_E_CUDA; }
    return B2_OK;
}

extern "C" int b2_counters_read(b2_ctx* c, int64_t out[B2_N_COUNTERS]) {
    if (!c || !out) return B2_E_INVAL;
    CU(cudaSetDevice(c->opt.device));
    CU(cudaMemcpy(out, c->d_counters, 8 * B2_N_COUNTERS, cudaMemcpyDeviceToHost));
    return B2_OK;
}
extern "C" void* b2_counters_device_ptr(b2_ctx* c) { return c ? (void*)c->d_counters : nullptr; }
// ncclAllReduce(sendbuff, recvbuff, count, ncclInt64 = 4, ncclSum = 0, comm, stream) — nccl.h; looked up in the process, not linked
extern "C" int b2_counters_allreduce(b2_ctx* c, void* nccl_comm) {
    if (!c || !nccl_comm) { set_err("null argument"); return B2_E_INVAL; }
    typedef int (*allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
    static allreduce_fn fn = reinterpret_cast<allreduce_fn>(dlsym(RTLD_DEFAULT, "ncclAllReduce"));
    if (!fn) { set_err("ncclAllReduce is not loaded in this process"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    const int rc = fn(c->d_counters, c->d_counters, B2_N_COUNTERS, 4 /*ncclInt64*/, 0 /*ncclSum*/, nccl_comm, c->stream);
    if (rc != 0) { char code[16]; snprintf(code, sizeof code, "%d", rc); set_err("ncclAllReduce failed: ncclResult_t %s", code); return B2_E_CUDA; }
    CU(cudaStreamSynchronize(c->stream));
    return B2_OK;
}

// device pointers of the resident batch, for harnesses that time or inspect kernels directly
extern "C" void* b2_debug_resp_device_ptr(b2_ctx* c) { return c ? (void*)c->d_resp : nullptr; }

__global__ void k_crc32c_batch(const uint8_t* bytes, const uint32_t* offs, const uint32_t* lens, uint32_t n, uint32_t* out,
                               const uint32_t* adv, uint32_t init_crc = 0) {
    __shared__ uint32_t s_hot[kCrcHotWords];
    crc_tabs_to_smem(s_hot, adv);
    CrcTabs ct; ct.hot = s_hot; ct.tree = adv + kCrcHotWords;
    const uint32_t lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += n_warps) {
        const uint32_t c = warp_crc32c_update(init_crc ^ 0xffffffffu, bytes + offs[i], lens[i], lane, ct) ^ 0xffffffffu;   // Extend(init_crc, ...)
        if (lane == 0) out[i] = c;
    }
}

extern "C" int b2_crc32c_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const uint32_t* offs, const uint32_t* lens,
                               uint32_t n, uint32_t* out) {
    if (!c || !bytes || !offs || !lens || !out) { set_err("null argument"); return B2_E_INVAL; }
    if (nbytes > c->opt.max_batch_bytes || n > c->opt.max_msgs) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    for (uint32_t i = 0; i < n; i++) if ((uint64_t)offs[i] + lens[i] > nbytes) { set_err("slice outside buffer"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_frame_off, offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_slot, lens, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    if (n) k_crc32c_batch<<<c->n_sms * 8, 256, 0, c->stream>>>(c->d_bytes, c->d_frame_off, c->d_slot, n, (uint32_t*)c->d_aux, c->d_crc_adv);
    CU(cudaMemcpyAsync(out, c->d_aux, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

__global__ void k_snappy_batch(const uint8_t* bytes, const uint32_t* offs, const uint32_t* lens, uint32_t n, uint8_t* out,
                               const uint32_t* out_offs, const uint32_t* out_caps, int32_t* out_lens) {
    const uint32_t lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5;
    __shared__ __align__(16) uint8_t s_rings[8 * kSnapRing];
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += n_warps) {
        uint32_t produced = 0;
        const bool ok = out_caps[i] != 0xffffffffu &&
                        warp_snappy_decode(bytes + offs[i], lens[i], out + out_offs[i], out_caps[i], lane, produced, s_rings + (threadIdx.x >> 5) * kSnapRing);
        if (lane == 0) out_lens[i] = ok ? (int32_t)produced : -1;
    }
}

extern "C" int b2_snappy_uncompress_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const uint32_t* offs, const uint32_t* lens,
                                          uint32_t n, void* out, uint32_t out_cap, uint32_t* out_offs, int32_t* out_lens) {
    if (!c || !bytes || !offs || !lens || !out || !out_offs || !out_lens) { set_err("null argument"); return B2_E_INVAL; }
    if (nbytes > c->opt.max_batch_bytes || n > c->opt.max_msgs || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    // output layout from the announced lengths (the preamble varint), nothing else is read on the host
    std::vector<uint32_t> caps(n);
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        if ((uint64_t)offs[i] + lens[i] > nbytes) { set_err("slice outside buffer"); return B2_E_INVAL; }
        const uint8_t* p = (const uint8_t*)bytes + offs[i];
        uint32_t v = 0, shift = 0, k = 0; bool ok = false;
        while (k < lens[i] && shift < 32) { const uint32_t b = p[k++]; v |= (b & 0x7f) << shift; if (b < 128) { ok = true; break; } shift += 7; }
        out_offs[i] = (uint32_t)total;
        if (!ok || (uint64_t)v > 32ull * lens[i] + 64ull) { caps[i] = 0xffffffffu; continue; }   // cannot be a valid stream
        caps[i] = v;
        total += ((uint64_t)v + 15) & ~15ull;
        if (total > out_cap) { set_err("output exceeds out_cap"); return B2_E_CAPACITY; }
    }
    CU(cudaSetDevice(c->opt.device));
    uint32_t* d_offs = c->d_frame_off; uint32_t* d_lens = c->d_slot; uint32_t* d_ooffs = c->d_frame_run;
    uint32_t* d_caps = (uint32_t*)c->d_jobs; int32_t* d_olens = (int32_t*)c->d_aux;
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_offs, offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_lens, lens, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_ooffs, out_offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_caps, caps.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    if (n) k_snappy_batch<<<c->n_sms * 4, 256, 0, c->stream>>>(c->d_bytes, d_offs, d_lens, n, c->d_unz, d_ooffs, d_caps, d_olens);
    CU(cudaMemcpyAsync(out_lens, d_olens, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    if (total) CU(cudaMemcpyAsync(out, c->d_unz, total, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

__global__ void __launch_bounds__(256) k_snappy_compress_batch(const uint8_t* bytes, const uint32_t* offs, const uint32_t* lens, uint32_t n,
                                                               uint8_t* out, const uint32_t* out_offs, uint32_t* out_lens, uint16_t* tabs) {
    const uint32_t lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5, warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint16_t* table = tabs + (size_t)(warp % kSnappyWarps) * kSnappyMaxTable;
    for (uint32_t i = warp; i < n; i += n_warps) {
        const uint32_t c = warp_snappy_compress(bytes + offs[i], lens[i], out + out_offs[i], table, lane);
        if (lane == 0) out_lens[i] = c;
    }
}

extern "C" int b2_snappy_compress_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const uint32_t* offs, const uint32_t* lens,
                                        uint32_t n, void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens) {
    if (!c || !bytes || !offs || !lens || !out || !out_offs || !out_lens) { set_err("null argument"); return B2_E_INVAL; }
    if (nbytes > c->opt.max_batch_bytes || n > c->opt.max_msgs || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        if ((uint64_t)offs[i] + lens[i] > nbytes) { set_err("slice outside buffer"); return B2_E_INVAL; }
        out_offs[i] = (uint32_t)total;
        total += ((uint64_t)snappy_max_compressed_length(lens[i]) + 15) & ~15ull;
        if (total > out_cap) { set_err("output exceeds out_cap"); return B2_E_CAPACITY; }
    }
    CU(cudaSetDevice(c->opt.device));
    uint32_t* d_offs = c->d_frame_off; uint32_t* d_lens = c->d_slot; uint32_t* d_ooffs = c->d_frame_run; uint32_t* d_olens = (uint32_t*)c->d_aux;
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_offs, offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_lens, lens, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_ooffs, out_offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    if (n) k_snappy_compress_batch<<<c->n_sms * 4, 256, 0, c->stream>>>(c->d_bytes, d_offs, d_lens, n, c->d_unz, d_ooffs, d_olens, c->d_snappy_tab);
    CU(cudaMemcpyAsync(out_lens, d_olens, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    if (total) CU(cudaMemcpyAsync(out, c->d_unz, total, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}


// ---- leaf codecs with the REFERENCE's own signatures (seam 4: what a CompressHandler / ChecksumHandler body or any direct caller of
// butil::crc32c / butil::snappy would be re-pointed at).  They run on a process-wide default context (device $B2_DEVICE or 0, created on
// first use); one buffer per call is the latency-bound way to use a GPU — the batch forms above are the throughput path.
static std::mutex g_leaf_mu;
static b2_ctx* g_leaf_ctx = nullptr;
static b2_ctx* leaf_ctx(size_t need_bytes) {
    if (g_leaf_ctx && need_bytes + 4096 <= g_leaf_ctx->opt.max_batch_bytes) return g_leaf_ctx;
    if (g_leaf_ctx) { b2_ctx_destroy(g_leaf_ctx); g_leaf_ctx = nullptr; }
    b2_options o; memset(&o, 0, sizeof o);
    o.device = getenv("B2_DEVICE") ? atoi(getenv("B2_DEVICE")) : 0;
    size_t cap = 8u << 20; while (cap < need_bytes + 4096 && cap < (1ull << 30)) cap <<= 1;
    o.max_batch_bytes = (uint32_t)cap; o.max_msgs = 4096; o.max_runs = 16; o.max_resp_bytes = (uint32_t)(cap + cap / 4 + (1u << 20));
    if (b2_ctx_create(&o, &g_leaf_ctx) != B2_OK) g_leaf_ctx = nullptr;
    return g_leaf_ctx;
}
// butil::crc32c::Extend (src/butil/crc32c.h:24, crc32c.cc:379-454)
extern "C" uint32_t b2_crc32c_extend(uint32_t init_crc, const char* data, size_t n) {
    if (n == 0) return init_crc;
    std::lock_guard<std::mutex> g(g_leaf_mu);
    b2_ctx* c = leaf_ctx(n);
    if (!c || n > c->opt.max_batch_bytes) return 0;
    cudaSetDevice(c->opt.device);
    const uint32_t off = 0, len = (uint32_t)n; uint32_t out = 0;
    if (cudaMemcpyAsync(c->d_bytes, data, n, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) return 0;
    cudaMemcpyAsync(c->d_frame_off, &off, 4, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(c->d_slot, &len, 4, cudaMemcpyHostToDevice, c->stream);
    k_crc32c_batch<<<1, 32, 0, c->stream>>>(c->d_bytes, c->d_frame_off, c->d_slot, 1, (uint32_t*)c->d_aux, c->d_crc_adv, init_crc);
    cudaMemcpyAsync(&out, c->d_aux, 4, cudaMemcpyDeviceToHost, c->stream);
    cudaStreamSynchronize(c->stream);
    c->uploaded = false; c->executed = false;
    return out;
}
// butil::snappy::MaxCompressedLength / RawCompress / GetUncompressedLength / RawUncompress (third_party/snappy/snappy.h:112-141)
extern "C" size_t b2_snappy_max_compressed_length(size_t n) { return 32 + n + n / 6; }
extern "C" void b2_snappy_raw_compress(const char* input, size_t input_length, char* compressed, size_t* compressed_length) {
    *compressed_length = 0;
    std::lock_guard<std::mutex> g(g_leaf_mu);
    b2_ctx* c = leaf_ctx(input_length + input_length / 4);
    if (!c) return;
    const uint32_t off = 0, len = (uint32_t)input_length; uint32_t ooff = 0, olen = 0;
    const uint8_t dummy = 0;
    if (b2_snappy_compress_batch(c, input_length ? (const void*)input : (const void*)&dummy, len, &off, &len, 1, compressed,
                                 (uint32_t)(((b2_snappy_max_compressed_length(input_length) + 15) & ~(size_t)15)), &ooff, &olen) == B2_OK) *compressed_length = olen;
}
extern "C" int b2_snappy_get_uncompressed_length(const char* compressed, size_t n, size_t* result) {   // varint32 preamble (snappy.cc:690-711)
    uint32_t v = 0, shift = 0; size_t k = 0;
    for (;;) {
        if (shift >= 32 || k >= n) return 0;
        const uint32_t b = (uint8_t)compressed[k++]; v |= (b & 0x7f) << shift;
        if (b < 128) break;
        shift += 7;
    }
    *result = v; return 1;
}
extern "C" int b2_snappy_raw_uncompress(const char* compressed, size_t compressed_length, char* uncompressed) {
    size_t ulen = 0;
    if (!b2_snappy_get_uncompressed_length(compressed, compressed_length, &ulen)) return 0;
    std::lock_guard<std::mutex> g(g_leaf_mu);
    b2_ctx* c = leaf_ctx(compressed_length > ulen ? compressed_length : ulen);
    if (!c) return 0;
    const uint32_t off = 0, len = (uint32_t)compressed_length; uint32_t ooff = 0; int32_t olen = -1;
    std::vector<char> tmp(((ulen + 15) & ~(size_t)15) + 16);
    if (b2_snappy_uncompress_batch(c, compressed, len, &off, &len, 1, tmp.data(), (uint32_t)tmp.size(), &ooff, &olen) != B2_OK || olen < 0 || (size_t)olen != ulen) return 0;
    memcpy(uncompressed, tmp.data() + ooff, ulen);
    return 1;
}

extern "C" int b2_hpack_reset(b2_ctx* c, uint32_t conn, uint32_t max_table_size) {
    if (!c || conn >= B2_HPACK_MAX_CONNS || max_table_size > 4096) { set_err("bad connection / table size"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    k_hpack_reset<<<1, 1, 0, c->stream>>>(c->d_hpack, conn, max_table_size);
    CU(cudaStreamSynchronize(c->stream));
    return B2_OK;
}

extern "C" int b2_hpack_decode_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_hpack_block* blocks, uint32_t n,
                                     void* out, uint32_t per_block_cap, uint32_t* out_lens, int32_t* status, uint32_t* n_headers) {
    if (!c || !bytes || !blocks || !out || !out_lens || !status || !n_headers) { set_err("null argument"); return B2_E_INVAL; }
    if (nbytes > c->opt.max_batch_bytes || n > c->opt.max_msgs / 4 || (uint64_t)n * per_block_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    std::vector<uint32_t> conn(n), off(n), len(n), first;
    for (uint32_t i = 0; i < n; i++) {
        if (blocks[i].conn >= B2_HPACK_MAX_CONNS || (uint64_t)blocks[i].offset + blocks[i].length > nbytes) { set_err("bad block"); return B2_E_INVAL; }
        conn[i] = blocks[i].conn; off[i] = blocks[i].offset; len[i] = blocks[i].length;
        if (i == 0 || conn[i] != conn[i - 1]) first.push_back(i);
    }
    const uint32_t n_groups = (uint32_t)first.size();
    first.push_back(n);
    for (uint32_t g = 0; g < n_groups; g++)                       // a connection may appear in one group only
        for (uint32_t g2 = g + 1; g2 < n_groups; g2++) if (conn[first[g]] == conn[first[g2]]) { set_err("blocks of one connection must be adjacent"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    uint32_t* d_conn = c->d_frame_off; uint32_t* d_off = c->d_frame_run; uint32_t* d_len = c->d_slot;
    uint32_t* d_first = (uint32_t*)c->d_jobs; uint32_t* d_olens = (uint32_t*)c->d_aux; int32_t* d_st = (int32_t*)c->d_aux + n; uint32_t* d_nh = (uint32_t*)c->d_aux + 2 * (size_t)n;
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_conn, conn.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_off, off.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_len, len.data(), 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_first, first.data(), 4 * first.size(), cudaMemcpyHostToDevice, c->stream));
    if (n_groups) k_hpack_decode<<<(n_groups + 63) / 64, 64, 0, c->stream>>>(c->d_bytes, d_conn, d_off, d_len, d_first, n_groups, c->d_hpack, c->d_unz, per_block_cap, d_olens, d_st, d_nh);
    CU(cudaMemcpyAsync(out_lens, d_olens, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(status, d_st, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(n_headers, d_nh, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    if (n) CU(cudaMemcpyAsync(out, c->d_unz, (size_t)n * per_block_cap, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

extern "C" int b2_h2_scan_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs, uint32_t max_frame_size,
                                b2_h2_frame* frames, uint32_t cap_per_run, uint32_t* n_frames, uint32_t* consumed, uint32_t* err) {
    if (!c || !bytes || !runs || !frames || !n_frames || !consumed || !err) { set_err("null argument"); return B2_E_INVAL; }
    if (nbytes > c->opt.max_batch_bytes || n_runs > c->opt.max_runs || (uint64_t)n_runs * cap_per_run * sizeof(b2_h2_frame) > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    for (uint32_t r = 0; r < n_runs; r++) if ((uint64_t)runs[r].offset + runs[r].length > nbytes) { set_err("run outside buffer"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    static_assert(sizeof(b2_h2_frame) == sizeof(H2Frame), "frame layout");
    uint32_t* d_n = c->d_frame_off; uint32_t* d_cons = c->d_frame_run; uint32_t* d_err = c->d_slot;
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_meta, runs, sizeof(b2_run) * (size_t)n_runs, cudaMemcpyHostToDevice, c->stream));
    if (n_runs) k_h2_scan<<<(n_runs + 63) / 64, 64, 0, c->stream>>>(c->d_bytes, (const b2_run*)c->d_meta, n_runs, max_frame_size, (H2Frame*)c->d_unz, cap_per_run, d_n, d_cons, d_err);
    CU(cudaMemcpyAsync(n_frames, d_n, 4 * (size_t)n_runs, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(consumed, d_cons, 4 * (size_t)n_runs, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(err, d_err, 4 * (size_t)n_runs, cudaMemcpyDeviceToHost, c->stream));
    if (n_runs) CU(cudaMemcpyAsync(frames, c->d_unz, (size_t)n_runs * cap_per_run * sizeof(b2_h2_frame), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

// ---- h2 connections: the state is allocated on first use (B2_H2_MAX_CONNS x ~128 KiB) ------------------------
static int h2_ensure(b2_ctx* c) {
    if (c->d_h2) return B2_OK;
    CU(cudaSetDevice(c->opt.device));
    const size_t n_streams = (size_t)c->h2_max_conns * c->h2_pending;
    CU(cudaMalloc(&c->d_h2, sizeof(H2Conn) * (size_t)c->h2_max_conns));
    if (cudaMalloc(&c->d_h2_streams, sizeof(H2Stream) * n_streams) != cudaSuccess || cudaMalloc(&c->d_h2_slots, n_streams * c->h2_stream_bytes) != cudaSuccess) {
        cudaFree(c->d_h2); cudaFree(c->d_h2_streams); c->d_h2 = nullptr; c->d_h2_streams = nullptr;
        set_err("h2 stream pool does not fit: lower b2_h2_configure's capacities"); return B2_E_NOMEM;
    }
    CU(cudaMemset(c->d_h2, 0, sizeof(H2Conn) * (size_t)c->h2_max_conns));
    CU(cudaMemset(c->d_h2_streams, 0xff, sizeof(H2Stream) * n_streams));           // id = -1: free
    return B2_OK;
}
static H2Pool h2_pool(const b2_ctx* c) { H2Pool p; p.streams = c->d_h2_streams; p.slots = c->d_h2_slots; p.pending = c->h2_pending; p.stream_bytes = c->h2_stream_bytes; return p; }
extern "C" int b2_h2_configure(b2_ctx* c, uint32_t max_conns, uint32_t max_pending, uint32_t stream_bytes) {
    if (!c || c->d_h2) { set_err("b2_h2_configure must precede the first h2 call on the context"); return B2_E_INVAL; }
    if (max_conns == 0 || max_conns > B2_HPACK_MAX_CONNS || max_pending == 0 || max_pending > 65536 || stream_bytes < B2_H2_HEADER_BYTES + 16 || (stream_bytes & 15u)) {
        set_err("bad h2 capacities"); return B2_E_INVAL;
    }
    c->h2_max_conns = max_conns; c->h2_pending = max_pending; c->h2_stream_bytes = stream_bytes;
    return B2_OK;
}
extern "C" int b2_h2_conn_reset(b2_ctx* c, uint32_t conn) {
    if (!c || conn >= c->h2_max_conns) { set_err("bad connection index"); return B2_E_INVAL; }
    int rc = h2_ensure(c); if (rc != B2_OK) return rc;
    k_h2_conn_reset<<<1, 1, 0, c->stream>>>(c->d_h2, c->d_hpack, conn, h2_pool(c));
    CU(cudaStreamSynchronize(c->stream));
    return B2_OK;
}
extern "C" int b2_h2_process_batch(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_run* runs, uint32_t n_runs,
                                   b2_h2_run_status* rs, b2_h2_msg* msgs, uint32_t msg_cap, uint32_t* n_msgs,
                                   void* out, uint32_t out_cap) {
    if (!c || !bytes || !runs || !rs || !msgs || !n_msgs || !out) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_h2_msg) == 64 && sizeof(b2_h2_run_status) == 32, "h2 ABI layout");
    if (nbytes > c->opt.max_batch_bytes || n_runs > c->opt.max_runs || out_cap > 2ull * c->opt.max_resp_bytes || msg_cap > c->opt.max_msgs) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    *n_msgs = 0;
    if (n_runs == 0) return B2_OK;
    for (uint32_t r = 0; r < n_runs; r++) {
        if ((uint64_t)runs[r].offset + runs[r].length > nbytes) { set_err("run outside buffer"); return B2_E_INVAL; }
        if (runs[r].socket_id >= c->h2_max_conns) { set_err("connection index out of range"); return B2_E_INVAL; }
        for (uint32_t q = 0; q < r; q++) if (runs[q].socket_id == runs[r].socket_id) { set_err("one run per connection and batch"); return B2_E_INVAL; }
    }
    const uint32_t region = (out_cap / n_runs) & ~63u, per_run_msgs = msg_cap / n_runs;
    if (region < 256 || per_run_msgs == 0) { set_err("out_cap / msg_cap too small for the number of runs"); return B2_E_CAPACITY; }
    int rc = h2_ensure(c); if (rc != B2_OK) return rc;
    CU(cudaSetDevice(c->opt.device));
    b2_h2_run_status* d_rs = reinterpret_cast<b2_h2_run_status*>(c->d_run_status);      // 32 B each, like b2_run_status
    b2_h2_msg* d_msgs = reinterpret_cast<b2_h2_msg*>(c->d_msgs);                         // 64 B each, like b2_msg_desc
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_meta, runs, sizeof(b2_run) * (size_t)n_runs, cudaMemcpyHostToDevice, c->stream));
    k_h2_consume<<<(n_runs + 31) / 32, 32, 0, c->stream>>>(c->d_bytes, (const b2_run*)c->d_meta, n_runs, c->d_h2, c->d_hpack, c->d_methods, c->cfg.n_methods,
                                                            d_rs, d_msgs, per_run_msgs, c->d_unz, region, h2_pool(c));
    CU(cudaMemcpyAsync(rs, d_rs, sizeof(b2_h2_run_status) * (size_t)n_runs, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    // fetch only what was produced: every run owns `region` bytes (acks from its start, records/bodies from region/4) and
    // per_run_msgs descriptors — three strided copies, then the descriptors are compacted into one list (run order)
    uint32_t total = 0, max_msgs = 0, max_ctrl = 0, max_blob = 0;
    for (uint32_t r = 0; r < n_runs; r++) {
        total += rs[r].n_msgs; if (rs[r].n_msgs > max_msgs) max_msgs = rs[r].n_msgs;
        if (rs[r].ctrl_len > max_ctrl) max_ctrl = rs[r].ctrl_len;
        if (rs[r].first_msg > max_blob) max_blob = rs[r].first_msg;             // (the kernel reports the blob bytes it used here)
    }
    if (total > msg_cap) { set_err("msg_cap too small"); return B2_E_CAPACITY; }
    std::vector<b2_h2_msg> tmp((size_t)n_runs * (max_msgs ? max_msgs : 1));
    if (max_msgs) CU(cudaMemcpy2DAsync(tmp.data(), sizeof(b2_h2_msg) * (size_t)max_msgs, d_msgs, sizeof(b2_h2_msg) * (size_t)per_run_msgs,
                                       sizeof(b2_h2_msg) * (size_t)max_msgs, n_runs, cudaMemcpyDeviceToHost, c->stream));
    if (max_ctrl) CU(cudaMemcpy2DAsync(out, region, c->d_unz, region, max_ctrl, n_runs, cudaMemcpyDeviceToHost, c->stream));
    if (max_blob) CU(cudaMemcpy2DAsync((uint8_t*)out + region / 4, region, c->d_unz + region / 4, region, max_blob, n_runs, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    total = 0;
    for (uint32_t r = 0; r < n_runs; r++) {
        if (rs[r].n_msgs) memcpy(msgs + total, tmp.data() + (size_t)r * max_msgs, sizeof(b2_h2_msg) * (size_t)rs[r].n_msgs);
        rs[r].first_msg = total; total += rs[r].n_msgs;
    }
    c->h2_last_in = nbytes; c->h2_last_out = (uint64_t)region * n_runs;
    *n_msgs = total;
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

extern "C" int b2_h2_pack_responses(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_h2_response* resps, uint32_t n,
                                    void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens) {
    if (!c || (!bytes && nbytes) || !resps || !out || !out_offs || !out_lens) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_h2_response) == 48, "h2 response ABI layout");
    if (nbytes > c->opt.max_resp_bytes || n > c->opt.max_msgs || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    if (n == 0) return B2_OK;
    std::vector<uint32_t> first;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        const b2_h2_response& r = resps[i];
        const uint64_t body_lim = (r.flags & B2_H2_RESP_BODY_IN_INPUT) ? c->h2_last_in : (r.flags & B2_H2_RESP_BODY_IN_OUT) ? c->h2_last_out :
                                  (r.flags & B2_H2_RESP_BODY_IN_UNZ) ? c->h2_last_unz : nbytes;
        const uint64_t ct_lim = (r.flags & B2_H2_RESP_CT_IN_OUT) ? c->h2_last_out : nbytes;
        if (r.conn >= c->h2_max_conns || (uint64_t)r.body_off + r.body_len > body_lim || (uint64_t)r.content_type_off + r.content_type_len > ct_lim ||
            (uint64_t)r.grpc_message_off + r.grpc_message_len > nbytes || r.content_type_len > 256 || r.grpc_message_len > 512) { set_err("bad response descriptor"); return B2_E_INVAL; }
        if ((r.flags & (B2_H2_RESP_BODY_IN_OUT | B2_H2_RESP_CT_IN_OUT)) && c->h2_last_out > c->opt.max_resp_bytes) { set_err("last h2 out buffer too large to stay resident"); return B2_E_CAPACITY; }
        if (i == 0 || r.conn != resps[i - 1].conn) first.push_back(i);
        const uint64_t data = (uint64_t)r.body_len + 5;
        const uint64_t need = data + 9 * (data / 16384 + 4) + 2ull * (r.content_type_len + r.grpc_message_len + 64) + 13 + 16;
        out_offs[i] = (uint32_t)total;
        total = (total + need + 15) & ~15ull;
        if (total > out_cap) { set_err("out_cap too small"); return B2_E_CAPACITY; }
    }
    const uint32_t n_groups = (uint32_t)first.size();
    first.push_back(n);
    for (uint32_t g = 0; g < n_groups; g++)
        for (uint32_t g2 = g + 1; g2 < n_groups; g2++) if (resps[first[g]].conn == resps[first[g2]].conn) { set_err("responses of one connection must be adjacent"); return B2_E_INVAL; }
    int rc = h2_ensure(c); if (rc != B2_OK) return rc;
    CU(cudaSetDevice(c->opt.device));
    b2_h2_response* d_resps = reinterpret_cast<b2_h2_response*>(c->d_msgs);       // 48 B <= 64 B per entry
    uint32_t* d_first = c->d_frame_off; uint32_t* d_offs = c->d_frame_run; uint32_t* d_lens = c->d_slot;
    uint8_t* d_aux = c->d_unz + c->opt.max_resp_bytes;            // second half of the scratch: the first half may hold the last h2 out buffer
    if (nbytes) CU(cudaMemcpyAsync(d_aux, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_resps, resps, sizeof(b2_h2_response) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_first, first.data(), 4 * first.size(), cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_offs, out_offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    k_h2_pack<<<(n_groups + kH2PackWarps - 1) / kH2PackWarps, kH2PackWarps * 32, 0, c->stream>>>(d_aux, c->d_bytes, c->d_unz, c->d_h2_unz, d_resps, d_first, n_groups, c->d_h2, c->d_resp, d_offs, d_lens);
    CU(cudaMemcpyAsync(out_lens, d_lens, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(out, c->d_resp, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

// GzipDecompress of ProcessHttpRequest over messages of the last h2 batch: see include/b2rpc.h
extern "C" int b2_h2_decompress_requests(b2_ctx* c, const b2_h2_msg* msgs, uint32_t n, void* out, uint32_t out_cap, b2_h2_unz_result* res) {
    if (!c || (n && (!msgs || !res)) || (!out && out_cap)) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_h2_unz_result) == 16, "h2 unz ABI layout");
    if (c->h2_last_out == 0) { set_err("no h2 batch is live on this context"); return B2_E_INVAL; }
    if (n > c->opt.max_msgs || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    for (uint32_t i = 0; i < n; i++) {         // descriptors come from the caller: every range inside the buffers of the live batch
        const b2_h2_msg& m = msgs[i];
        const uint64_t lim = (m.flags & B2_H2_FLAG_BODY_IN_INPUT) ? c->h2_last_in : c->h2_last_out;
        const uint64_t out_end = std::max<uint64_t>((uint64_t)m.headers_off + m.headers_len, (m.flags & B2_H2_FLAG_BODY_IN_INPUT) ? 0 :
                                                    std::max<uint64_t>((uint64_t)m.body_off + m.body_len, (uint64_t)m.msg_off + m.msg_len));
        if ((uint64_t)m.headers_off + m.headers_len > c->h2_last_out || (uint64_t)m.body_off + m.body_len > lim || (uint64_t)m.msg_off + m.msg_len > lim) {
            set_err("a message lies outside the last h2 batch"); return B2_E_INVAL;
        }
        // b2_h2_pack_responses stages its bytes in the second half of the scratch: only the first max_resp_bytes of the out buffer stay
        if (out_end > c->opt.max_resp_bytes) { set_err("last h2 out buffer too large to stay resident"); return B2_E_CAPACITY; }
    }
    c->h2_last_unz = 0;
    if (n == 0) return B2_OK;
    CU(cudaSetDevice(c->opt.device));
    if (!c->d_h2_unz) CU(cudaMalloc(&c->d_h2_unz, (size_t)c->opt.max_resp_bytes + 16));
    b2_h2_msg* d_msgs = reinterpret_cast<b2_h2_msg*>(c->d_msgs);                 // the batch's own descriptors were fetched by b2_h2_process_batch
    b2_h2_unz_result* d_res = reinterpret_cast<b2_h2_unz_result*>(c->d_aux);      // 16 B <= sizeof(MsgAux) per message
    static_assert(sizeof(MsgAux) >= sizeof(b2_h2_unz_result), "unz results live in the aux array");
    CU(cudaMemcpyAsync(d_msgs, msgs, sizeof(b2_h2_msg) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    const uint32_t grid = (n + kH2UnzWarps - 1) / kH2UnzWarps;
    c->stage_names[0] = "h2_inflate_size"; c->stage_names[1] = "h2_unz_offsets"; c->stage_names[2] = "h2_inflate_write";
    CU(cudaEventRecord(c->ev[0], c->stream));
    k_h2_inflate<false><<<grid, kH2UnzWarps * 32, 0, c->stream>>>(c->d_bytes, c->d_unz, d_msgs, n, d_res, c->d_h2_unz);
    CU(cudaEventRecord(c->ev[1], c->stream));
    k_h2_unz_offsets<<<1, kUnzScanBlock, 0, c->stream>>>(d_res, n, out_cap);
    CU(cudaEventRecord(c->ev[2], c->stream));
    k_h2_inflate<true><<<grid, kH2UnzWarps * 32, 0, c->stream>>>(c->d_bytes, c->d_unz, d_msgs, n, d_res, c->d_h2_unz);
    CU(cudaEventRecord(c->ev[3], c->stream));
    c->n_stages = 3;
    CU(cudaMemcpyAsync(res, d_res, sizeof(b2_h2_unz_result) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    uint64_t end = 0;                                                             // only the bytes produced go back
    for (uint32_t i = 0; i < n; i++) if (res[i].status == B2_H2_UNZ_OK) end = std::max<uint64_t>(end, (uint64_t)res[i].out_off + res[i].out_len);
    if (end) {
        CU(cudaMemcpyAsync(out, c->d_h2_unz, (size_t)end, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    c->h2_last_unz = end;
    return B2_OK;
}

// client side of h2: see include/b2rpc.h
extern "C" int b2_h2_pack_requests(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_h2_request* reqs, uint32_t n,
                                   void* out, uint32_t out_cap, b2_h2_request_result* results) {
    if (!c || !bytes || !reqs || !out || !results) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_h2_request) == 48 && sizeof(b2_h2_request_result) == 16, "h2 request ABI layout");
    if (nbytes > c->opt.max_resp_bytes || n > c->opt.max_msgs || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    if (n == 0) return B2_OK;
    std::vector<uint32_t> first;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        const b2_h2_request& r = reqs[i];
        if (r.conn >= c->h2_max_conns || (uint64_t)r.path_off + r.path_len > nbytes || (uint64_t)r.authority_off + r.authority_len > nbytes ||
            (uint64_t)r.content_type_off + r.content_type_len > nbytes || (uint64_t)r.body_off + r.body_len > nbytes ||
            (uint64_t)r.extra_off + r.extra_len > nbytes) { set_err("bad request descriptor"); return B2_E_INVAL; }
        // the encoded header block must fit the kernel's shared-memory fragment: every header costs at most its bytes + 2 x 3 length bytes + 1
        uint64_t hdr = 4 * 16 + 64 + (uint64_t)r.path_len + r.authority_len + r.content_type_len + 16 + 32, n_extra = 0;
        for (uint32_t at = 0; at + 4 <= r.extra_len;) {
            const uint8_t* e = static_cast<const uint8_t*>(bytes) + r.extra_off + at;
            const uint32_t nl = e[0] | ((uint32_t)e[1] << 8), vl = e[2] | ((uint32_t)e[3] << 8);
            if (at + 4 + nl + vl > r.extra_len) { set_err("truncated extra header record"); return B2_E_INVAL; }
            if (nl + vl > kH2ReqFragCap / 2) { set_err("header too long"); return B2_E_INVAL; }
            hdr += nl + vl + 8; n_extra++; at += 4 + nl + vl;
        }
        if (hdr > kH2ReqFragCap || r.path_len + 16 > kH2ReqFragCap / 2 || r.authority_len + 16 > kH2ReqFragCap / 2 || r.content_type_len + 16 > kH2ReqFragCap / 2) { set_err("header block too long"); return B2_E_INVAL; }
        if (i == 0 || r.conn != reqs[i - 1].conn) first.push_back(i);
        const uint64_t data = (uint64_t)r.body_len + 5;
        const uint64_t need = 58 + hdr + 9 + data + 9 * (data / 16384 + 4) + 13 + 16;
        results[i].status = 0; results[i].stream_id = 0; results[i].out_off = (uint32_t)total; results[i].out_len = 0;
        total = (total + need + 15) & ~15ull;
        if (total > out_cap) { set_err("out_cap too small"); return B2_E_CAPACITY; }
    }
    const uint32_t n_groups = (uint32_t)first.size();
    first.push_back(n);
    for (uint32_t g = 0; g < n_groups; g++)
        for (uint32_t g2 = g + 1; g2 < n_groups; g2++) if (reqs[first[g]].conn == reqs[first[g2]].conn) { set_err("requests of one connection must be adjacent"); return B2_E_INVAL; }
    int rc = h2_ensure(c); if (rc != B2_OK) return rc;
    CU(cudaSetDevice(c->opt.device));
    b2_h2_request* d_reqs = reinterpret_cast<b2_h2_request*>(c->d_msgs);          // 48 B <= 64 B per entry
    b2_h2_request_result* d_res = reinterpret_cast<b2_h2_request_result*>(c->d_aux);
    static_assert(sizeof(MsgAux) >= sizeof(b2_h2_request_result), "results live in the aux array");
    uint32_t* d_first = c->d_frame_off;
    uint8_t* d_in = c->d_unz + c->opt.max_resp_bytes;             // second half of the scratch (as b2_h2_pack_responses)
    CU(cudaMemcpyAsync(d_in, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_reqs, reqs, sizeof(b2_h2_request) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_res, results, sizeof(b2_h2_request_result) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_first, first.data(), 4 * first.size(), cudaMemcpyHostToDevice, c->stream));
    k_h2_pack_req<<<(n_groups + kH2PackWarps - 1) / kH2PackWarps, kH2PackWarps * 32, 0, c->stream>>>(d_in, d_reqs, d_first, n_groups, c->d_h2, c->d_resp, d_res);
    CU(cudaMemcpyAsync(results, d_res, sizeof(b2_h2_request_result) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(out, c->d_resp, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}
extern "C" int b2_h2_conn_peer_update(b2_ctx* c, uint32_t conn, const b2_h2_peer_update* u) {
    if (!c || !u) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_h2_peer_update) == 24, "peer update ABI layout");
    if ((u->set & B2_H2_PEER_MAX_FRAME_SIZE) && (u->max_frame_size < 16384u || u->max_frame_size > 16777215u)) { set_err("max_frame_size out of range"); return B2_E_INVAL; }   // ParseH2Settings :166-211
    if ((u->set & B2_H2_PEER_STREAM_WINDOW) && u->stream_window_size > 0x7fffffffu) { set_err("stream_window_size out of range"); return B2_E_INVAL; }
    int rc = h2_ensure(c); if (rc != B2_OK) return rc;
    if (conn >= c->h2_max_conns) { set_err("conn out of range"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    int* d_rc = reinterpret_cast<int*>(c->d_slot); int h_rc = 0;
    k_h2_peer_update<<<1, 1, 0, c->stream>>>(c->d_h2, conn, *u, d_rc);
    CU(cudaMemcpyAsync(&h_rc, d_rc, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (h_rc != 0) { set_err("connection window would pass 2^31 - 1 (FLOW_CONTROL_ERROR)"); return B2_E_INVAL; }
    return B2_OK;
}
extern "C" int b2_h2_conn_set_next_stream_id(b2_ctx* c, uint32_t conn, uint32_t next_id) {
    if (!c) { set_err("null argument"); return B2_E_INVAL; }
    int rc = h2_ensure(c); if (rc != B2_OK) return rc;
    if (conn >= c->h2_max_conns) { set_err("conn out of range"); return B2_E_INVAL; }
    CU(cudaSetDevice(c->opt.device));
    k_h2_set_next_stream_id<<<1, 1, 0, c->stream>>>(c->d_h2, conn, next_id);
    CU(cudaStreamSynchronize(c->stream));
    return B2_OK;
}

extern "C" int b2_pack_requests(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_request* reqs, uint32_t n,
                                void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens) {
    if (!c || (!bytes && nbytes) || !reqs || !out || !out_offs || !out_lens) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_request) == 64 && sizeof(ReqDesc) == 64, "request ABI layout");
    if (nbytes > c->opt.max_batch_bytes || n > c->opt.max_msgs || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    if (n == 0) return B2_OK;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        const b2_request& r = reqs[i];
        if ((uint64_t)r.payload_off + r.payload_len > nbytes || (uint64_t)r.attachment_off + r.attachment_len > nbytes) { set_err("payload outside buffer"); return B2_E_INVAL; }
        const uint64_t pb = 6ull + r.payload_len;
        const uint64_t need = 12 + 512 + (r.compress_type == B2_COMPRESS_TYPE_SNAPPY ? snappy_max_compressed_length((uint32_t)pb) : pb) + r.attachment_len;
        out_offs[i] = (uint32_t)total;
        total = (total + need + 15) & ~15ull;
        if (total > out_cap) { set_err("out_cap too small"); return B2_E_CAPACITY; }
    }
    CU(cudaSetDevice(c->opt.device));
    ReqDesc* d_reqs = reinterpret_cast<ReqDesc*>(c->d_msgs);
    uint32_t* d_offs = c->d_frame_off; uint32_t* d_lens = c->d_slot;
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;       // the device copies of the last h2 batch are about to be overwritten
    if (nbytes) CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_reqs, reqs, sizeof(b2_request) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_offs, out_offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    k_pack_requests<<<c->n_sms * 4, 256, 0, c->stream>>>(c->d_bytes, d_reqs, n, c->d_methods, c->cfg.n_methods, c->d_resp, d_offs, d_lens, c->d_unz, c->d_snappy_tab, c->d_crc_adv);
    CU(cudaMemcpyAsync(out_lens, d_lens, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(out, c->d_resp, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}

// SendRpcResponse for replies the host produced: see include/b2rpc.h
extern "C" int b2_pack_responses(b2_ctx* c, const void* bytes, uint32_t nbytes, const b2_reply* reps, uint32_t n,
                                 void* out, uint32_t out_cap, uint32_t* out_offs, uint32_t* out_lens) {
    if (!c || (!bytes && nbytes) || !reps || !out || !out_offs || !out_lens) { set_err("null argument"); return B2_E_INVAL; }
    static_assert(sizeof(b2_reply) == 88 && sizeof(ReplyDesc) == 88, "reply ABI layout");
    if (nbytes > c->opt.max_batch_bytes || (uint64_t)n * sizeof(b2_reply) > (uint64_t)c->opt.max_msgs * 64 || out_cap > c->opt.max_resp_bytes) { set_err("exceeds ctx capacity"); return B2_E_CAPACITY; }
    if (n == 0) return B2_OK;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        const b2_reply& r = reps[i];
        if ((uint64_t)r.body_off + r.body_len > nbytes || (uint64_t)r.attachment_off + r.attachment_len > nbytes || (uint64_t)r.error_text_off + r.error_text_len > nbytes ||
            (uint64_t)r.checksum_value_off + r.checksum_value_len > nbytes || (r.extra_streams_off & 7u) || (uint64_t)r.extra_streams_off + 8ull * r.n_extra_streams > nbytes ||
            r.user_fields_off > nbytes) { set_err("reply field outside buffer"); return B2_E_INVAL; }
        uint64_t uf = 0, at = r.user_fields_off;                       // every record must lie inside the buffer: the kernel walks them
        for (uint32_t k = 0; k < r.n_user_fields; k++) {
            if (at + 8 > nbytes) { set_err("user field outside buffer"); return B2_E_INVAL; }
            uint32_t kl, vl; memcpy(&kl, static_cast<const uint8_t*>(bytes) + at, 4); memcpy(&vl, static_cast<const uint8_t*>(bytes) + at + 4, 4);
            if (at + 8 + (uint64_t)kl + vl > nbytes) { set_err("user field outside buffer"); return B2_E_INVAL; }
            uf += 24ull + kl + vl; at += 8ull + kl + vl;
        }
        const uint64_t body = r.compress_type == B2_COMPRESS_TYPE_SNAPPY ? snappy_max_compressed_length(r.body_len) : r.body_len;
        const uint64_t need = 12 + 128 + r.error_text_len + r.checksum_value_len + 11ull * r.n_extra_streams + uf + body + r.attachment_len;
        out_offs[i] = (uint32_t)total;
        total = (total + need + 15) & ~15ull;
        if (total > out_cap) { set_err("out_cap too small"); return B2_E_CAPACITY; }
    }
    CU(cudaSetDevice(c->opt.device));
    ReplyDesc* d_reps = reinterpret_cast<ReplyDesc*>(c->d_msgs);
    uint32_t* d_offs = c->d_frame_off; uint32_t* d_lens = c->d_slot;
    c->h2_last_in = 0; c->h2_last_out = 0; c->h2_last_unz = 0;
    if (nbytes) CU(cudaMemcpyAsync(c->d_bytes, bytes, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_reps, reps, sizeof(b2_reply) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(d_offs, out_offs, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    k_pack_responses<<<c->n_sms * 4, 256, 0, c->stream>>>(c->d_bytes, d_reps, n, c->d_resp, d_offs, d_lens, c->d_unz, c->d_snappy_tab, c->d_crc_adv);
    CU(cudaMemcpyAsync(out_lens, d_lens, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(out, c->d_resp, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->uploaded = false; c->executed = false;
    return B2_OK;
}
