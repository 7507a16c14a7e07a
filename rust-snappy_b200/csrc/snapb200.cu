// snapb200.cu -- libsnapb200.so: sm_100a kernels + the C ABI of include/snapb200.h.
// Built by __graft_entry__.build() with
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
// There is no CPU execution path in this library: every compute entry point
// launches the kernels below and fails with SB_E_NO_DEVICE when it cannot.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>
#include <sched.h>
#include <time.h>

#include "k1_compress.cuh"
#include "k2_decompress.cuh"
#include "k3_crc32c.cuh"
#include "k4_frame.cuh"
#include "k5_frame_decode.cuh"
#include "k7_streams.cuh"

namespace {

// ------------------------------------------------------------------ kernels
// K1: one CTA per SM: 7 parser/emitter pairs with their tables in shared memory + NG pairs with
// their tables in an L2-resident scratch; rings in global scratch; units taken from `work`
template <int NG>
__global__ void __launch_bounds__((7 + NG) * 64, 1)
k1_m7_kernel(sb_batch b, uint32_t flags, uint64_t* rings, uint16_t* gtables, uint32_t* work, uint32_t* crcs) {
    sbk::k1_compress_body_multi<7, NG>(b, flags, rings, gtables, work, crcs);
}
const int K1_MAX_NG = 7;
const size_t K1_M7_SMEM = sbk::k1_multi_smem(7, K1_MAX_NG);
// 48 registers -> 10 CTAs (40 warps) per SM; forcing 12/14 CTAs through launch bounds spills and measured 5% slower
__global__ void __launch_bounds__(128) k2_decompress_kernel(sb_batch b) { sbk::k2_decompress_body(b); }
__global__ void __launch_bounds__(256) k3_crc_kernel(sb_batch b) { sbk::k3_crc_body(b); }
__global__ void __launch_bounds__(256) k4_fill_lens_kernel(uint32_t* lens, uint64_t n, uint32_t nchunks) { sbk::k4_fill_lens_body(lens, n, nchunks); }
__global__ void __launch_bounds__(1024) k4_scan_local_kernel(sbk::FramePlan p) { sbk::k4_scan_local_body(p); }
__global__ void __launch_bounds__(1024) k4_scan_tiles_kernel(sbk::FramePlan p) { sbk::k4_scan_tiles_body(p); }
__global__ void __launch_bounds__(256) k4_gather_kernel(sbk::FramePlan p) { sbk::k4_gather_body(p); }
__global__ void __launch_bounds__(256) k5_parse_kernel(sbk::DecodePlan p) { sbk::k5_parse_body(p); }
__global__ void __launch_bounds__(32) k5_walk_kernel(sbk::DecodePlan p) { sbk::k5_walk_body(p); }
__global__ void __launch_bounds__(1024) k5_scan_local_kernel(sbk::DecodePlan p) { sbk::k5_scan_local_body(p); }
__global__ void __launch_bounds__(1024) k5_scan_tiles_kernel(sbk::DecodePlan p) { sbk::k5_scan_tiles_body(p); }
__global__ void __launch_bounds__(128) k5_decode_kernel(sbk::DecodePlan p) { sbk::k5_decode_body(p); }
__global__ void __launch_bounds__(32) k5_finish_kernel(sbk::DecodePlan p) { sbk::k5_finish_body(p); }
__global__ void __launch_bounds__(256) k6_generate_kernel(sbk::GenPlan g) { sbk::k6_generate_body(g); }
__global__ void __launch_bounds__(1024) k7_plan_kernel(sbk::StreamsPlan p) { sbk::k7_plan_body(p); }
__global__ void __launch_bounds__(1024) k7_unit_tiles_kernel(sbk::StreamsPlan p) { sbk::k7_unit_tiles_body(p); }
__global__ void __launch_bounds__(256) k7_expand_kernel(sbk::StreamsPlan p) { sbk::k7_expand_body(p); }
__global__ void __launch_bounds__(1024) k7_item_scan_kernel(sbk::StreamsPlan p) { sbk::k7_item_scan_body(p); }
__global__ void __launch_bounds__(1024) k7_item_tiles_kernel(sbk::StreamsPlan p) { sbk::k7_item_tiles_body(p); }
__global__ void __launch_bounds__(256) k7_gather_kernel(sbk::StreamsPlan p) { sbk::k7_gather_body(p); }
__global__ void __launch_bounds__(1024) k7_dplan_kernel(sbk::StreamsDecPlan p) { sbk::k7_dplan_body(p); }
__global__ void __launch_bounds__(1024) k7_dtiles_kernel(sbk::StreamsDecPlan p) { sbk::k7_dtiles_body(p); }
__global__ void __launch_bounds__(256) k7_dfill_kernel(sbk::StreamsDecPlan p) { sbk::k7_dfill_body(p); }
__global__ void __launch_bounds__(256) k7_dfinish_kernel(sbk::StreamsDecPlan p) { sbk::k7_dfinish_body(p); }
__global__ void __launch_bounds__(32) k7_dresult_kernel(sbk::StreamsDecPlan p) { sbk::k7_dresult_body(p); }

std::atomic<uint64_t> g_launches{0};
std::atomic<uint64_t> g_allocs{0};     // cudaMalloc / cudaHostAlloc / event + stream creations since load
const int K2_DEFAULT_CTAS_PER_SM = 16;
const int K1_DEFAULT_NG = 5;

int fail(sb_error* e, uint32_t code, uint64_t a = 0, uint64_t b = 0, uint64_t c = 0) {
    if (e) { e->code = code; e->_pad = 0; e->a = a; e->b = b; e->c = c; }
    return (int)code;
}
void ok(sb_error* e) { if (e) { e->code = 0; e->_pad = 0; e->a = e->b = e->c = 0; } }

#define CK(call)                                                                   \
    do {                                                                           \
        cudaError_t _e = (call);                                                   \
        if (_e != cudaSuccess) {                                                   \
            if (getenv("SNAPB200_DEBUG"))                                          \
                fprintf(stderr, "snapb200: %s -> %s (%s:%d)\n", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return fail(err, (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver || \
                              _e == cudaErrorNoKernelImageForDevice) ? SB_E_NO_DEVICE : SB_E_CUDA, (uint64_t)_e); \
        }                                                                          \
    } while (0)

// ------------------------------------------------------------- device state
// Grow-only pools: the first calls size them (or sb_reserve does), the steady state allocates nothing.
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t need(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        size_t want = n + n / 8 + 4096;
        g_allocs++;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, n); want = n; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T> T* as() { return (T*)p; }
};

// A lane = everything one host call needs besides the K1 scratch: three streams, the events of the wave pipeline,
// grow-only device staging and pinned descriptors, and a mutex. Two lanes per device: lane 0 serves the compress-side
// entry points, lane 1 the decompress-side ones, so that a caller running both directions from two threads gets
// H2D, kernels and D2H of both in flight at once (PCIe is full duplex; K2 fits beside K1's waves).
struct Lane {
    cudaStream_t s_compute = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_k[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};   // host-batch pipeline
    DevBuf in[2], slots[2], compact[2], lens[2], status[2], ptrs_in[2], ptrs_out[2], caps[2], ws[2];
    DevBuf sws[2];   // compress lane: everything of a raw-streams wave besides the K1 slots
    void* pinned[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // pinned staging: [0,1] descriptors in, [2,3] results out, [4] scalar results
    size_t pinned_cap[5] = {0, 0, 0, 0, 0};
    std::mutex mu;
};
struct Ctx {
    int dev = -1, sms = 0;
    std::atomic<bool> ready{false};
    DevBuf rings, gtables, work;   // K1 scratch: event rings, L2-resident tables, unit counter
    cudaEvent_t k1_done = nullptr; // K1 launches share that scratch: each waits for the previous one, whatever its stream
    std::mutex k1_mu;
    Lane lane[2];
};
const int LANE_ENC = 0, LANE_DEC = 1;
Ctx g_ctx[16];
std::mutex g_init_mu;

int init_ctx(Ctx& c, int dev, sb_error* err) {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    c.dev = dev; c.sms = prop.multiProcessorCount;
    CK(cudaFuncSetAttribute(k1_m7_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_M7_SMEM));
    CK(cudaFuncSetAttribute(k1_m7_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_M7_SMEM));
    CK(cudaFuncSetAttribute(k1_m7_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1_M7_SMEM));
    CK(c.rings.need((size_t)c.sms * (7 + K1_MAX_NG) * sbk::K1_RING_GW * 8));
    CK(c.gtables.need((size_t)c.sms * K1_MAX_NG * sbk::K1_TABLE_BYTES));
    CK(c.work.need(256));
    g_allocs += 19;
    CK(cudaEventCreateWithFlags(&c.k1_done, cudaEventDisableTiming));
    for (Lane& l : c.lane) {
        for (int k = 0; k < 2; k++) {
            CK(cudaEventCreateWithFlags(&l.ev_in[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&l.ev_k[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&l.ev_out[k], cudaEventDisableTiming));
        }
        CK(cudaStreamCreateWithFlags(&l.s_compute, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&l.s_h2d, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&l.s_d2h, cudaStreamNonBlocking));
    }
    return 0;
}
void destroy_partial(Ctx& c) {
    if (c.k1_done) { cudaEventDestroy(c.k1_done); c.k1_done = nullptr; }
    for (Lane& l : c.lane) {
        for (int k = 0; k < 2; k++) {
            if (l.ev_in[k]) { cudaEventDestroy(l.ev_in[k]); l.ev_in[k] = nullptr; }
            if (l.ev_k[k]) { cudaEventDestroy(l.ev_k[k]); l.ev_k[k] = nullptr; }
            if (l.ev_out[k]) { cudaEventDestroy(l.ev_out[k]); l.ev_out[k] = nullptr; }
        }
        if (l.s_compute) { cudaStreamDestroy(l.s_compute); l.s_compute = nullptr; }
        if (l.s_h2d) { cudaStreamDestroy(l.s_h2d); l.s_h2d = nullptr; }
        if (l.s_d2h) { cudaStreamDestroy(l.s_d2h); l.s_d2h = nullptr; }
    }
}

// First use per device is serialised (two threads making their first call together run one initialisation);
// a failed initialisation is undone and retried by the next call.
int get_ctx(Ctx** out, sb_error* err) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) return fail(err, SB_E_NO_DEVICE);
    Ctx& c = g_ctx[dev];
    if (!c.ready.load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lk(g_init_mu);
        if (!c.ready.load(std::memory_order_relaxed)) {
            const int rc = init_ctx(c, dev, err);
            if (rc) { destroy_partial(c); return rc; }
            c.ready.store(true, std::memory_order_release);
        }
    }
    *out = &c;
    return 0;
}

// Descriptor arrays (pointers, lengths) are staged through pinned memory: an async copy from
// pageable memory would not overlap with the running kernel.
int need_pinned(Lane& c, int slot, size_t n, sb_error* err) {
    if (n <= c.pinned_cap[slot]) return 0;
    if (c.pinned[slot]) { CK(cudaFreeHost(c.pinned[slot])); c.pinned[slot] = nullptr; c.pinned_cap[slot] = 0; }
    n += n / 4 + 4096;
    g_allocs++;
    CK(cudaHostAlloc(&c.pinned[slot], n, cudaHostAllocDefault));
    c.pinned_cap[slot] = n;
    return 0;
}

// ------------------------------------------------------------ launch helpers
int launch_k1(Ctx& c, const sb_batch& b, uint32_t flags, uint32_t* crcs, cudaStream_t st, sb_error* err) {
    if (b.count == 0) return 0;
    // SNAPB200_K1_NG = chains per SM with L2-resident tables next to the 7 shared-memory ones (0..7)
    static const int ng_env = getenv("SNAPB200_K1_NG") ? atoi(getenv("SNAPB200_K1_NG")) : K1_DEFAULT_NG;
    const unsigned ng = ng_env < 0 ? 0 : ng_env > K1_MAX_NG ? K1_MAX_NG : (unsigned)ng_env;
    // small batches spread over the SMs first (one shared-memory-table chain per SM is the fastest a block can
    // run); only batches with more units than that stack chains on an SM, L2-table chains last
    unsigned chains = (unsigned)(((uint64_t)b.count + c.sms - 1) / c.sms);
    if (chains > 7 + ng) chains = 7 + ng;
    unsigned mg = (unsigned)c.sms;
    if (mg > b.count) mg = b.count;
    std::lock_guard<std::mutex> k1lk(c.k1_mu);
    CK(cudaStreamWaitEvent(st, c.k1_done, 0));
    CK(cudaMemsetAsync(c.work.p, 0, 4, st));
    uint64_t* rg = c.rings.as<uint64_t>(); uint16_t* gt = c.gtables.as<uint16_t>(); uint32_t* wk = c.work.as<uint32_t>();
    // the template argument only bounds the chain count (launch bounds / register cap, scratch strides)
    if (ng > 5) k1_m7_kernel<7><<<mg, chains * 64, K1_M7_SMEM, st>>>(b, flags, rg, gt, wk, crcs);
    else if (ng > 0) k1_m7_kernel<5><<<mg, chains * 64, K1_M7_SMEM, st>>>(b, flags, rg, gt, wk, crcs);
    else k1_m7_kernel<0><<<mg, chains * 64, K1_M7_SMEM, st>>>(b, flags, rg, gt, wk, crcs);
    CK(cudaGetLastError());
    CK(cudaEventRecord(c.k1_done, st));
    g_launches++;
    return 0;
}
int launch_k2(Ctx& c, const sb_batch& b, cudaStream_t st, sb_error* err) {
    if (b.count == 0) return 0;
    const unsigned wpb = 4;
    uint64_t blocks = ((uint64_t)b.count + wpb - 1) / wpb;
    // resident CTAs per SM: each warp keeps a 64KB output history alive, and copy sources are
    // re-read from it -- too many streams in flight and the history falls out of the 126MB L2
    static const int per_sm = getenv("SNAPB200_K2_CTAS") ? atoi(getenv("SNAPB200_K2_CTAS")) : K2_DEFAULT_CTAS_PER_SM;
    unsigned grid = (unsigned)(per_sm * c.sms);
    if (grid > blocks) grid = (unsigned)blocks;
    k2_decompress_kernel<<<grid, 32 * wpb, wpb * sbk::K2_SMEM_PER_WARP, st>>>(b);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
int launch_k3(Ctx& c, const sb_batch& b, cudaStream_t st, sb_error* err) {
    if (b.count == 0) return 0;
    const unsigned wpb = 8;
    uint64_t blocks = ((uint64_t)b.count + wpb - 1) / wpb;
    unsigned grid = (unsigned)(8 * c.sms);
    if (grid > blocks) grid = (unsigned)blocks;
    k3_crc_kernel<<<grid, 32 * wpb, sbk::K3_TABLE_BYTES, st>>>(b);
    g_launches++;
    CK(cudaGetLastError());
    return 0;
}
// scan (tile-local, tiles) -> gather over a FramePlan whose slots/clens(/crcs) are filled
int launch_assemble(Ctx& c, const sbk::FramePlan& p, cudaStream_t st, sb_error* err) {
    if (p.nchunks == 0) return 0;
    const unsigned ntiles = (p.nchunks + sbk::K4_TILE - 1) / sbk::K4_TILE;
    k4_scan_local_kernel<<<ntiles, sbk::K4_TILE, 32 * sizeof(uint32_t), st>>>(p);
    k4_scan_tiles_kernel<<<1, 1024, 1024 * sizeof(uint64_t), st>>>(p);
    uint64_t blocks = ((uint64_t)p.nchunks + 7) / 8;
    unsigned grid = (unsigned)(8 * c.sms);
    if (grid > blocks) grid = (unsigned)blocks;
    k4_gather_kernel<<<grid, 256, 0, st>>>(p);
    g_launches += 3;
    CK(cudaGetLastError());
    return 0;
}

size_t put_varint(uint8_t* dst, uint64_t v) {   // reference src/bytes.rs:61-70
    size_t i = 0;
    while (v >= 0x80) { dst[i++] = (uint8_t)v | 0x80; v >>= 7; }
    dst[i++] = (uint8_t)v;
    return i;
}
// reference src/bytes.rs:73-90 (checked_shl fails only when shift >= 64)
size_t get_varint(const uint8_t* p, size_t n, uint64_t* out) {
    uint64_t v = 0;
    unsigned shift = 0;
    for (size_t i = 0; i < n; i++) {
        if (shift >= 64) return 0;
        uint8_t b = p[i];
        if (b < 0x80) { *out = v | ((uint64_t)b << shift); return i + 1; }
        v |= (uint64_t)(b & 0x7F) << shift;
        shift += 7;
    }
    return 0;
}

const uint64_t SB_MAX_INPUT = 0xFFFFFFFFull;
const uint32_t SB_MAX_BLOCK = 65536;
const uint32_t SB_MAX_CBLOCK = 76490;   // reference src/frame.rs:12

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- workspace layouts (caller-provided or pooled scratch; every sub-array 256-byte aligned)
struct EncodeWs { uint8_t* slots; uint32_t *lens_in, *clens, *crcs; uint64_t *offs, *tiles; };
uint64_t encode_ws_bytes(uint64_t n) {
    const uint64_t nchunks = (n + SB_MAX_BLOCK - 1) / SB_MAX_BLOCK;
    return align_up(nchunks * (uint64_t)sbk::kSlotStride, 256) + 3 * align_up(nchunks * 4 + 4, 256) +
           align_up((nchunks + 1) * 8, 256) + align_up((nchunks / sbk::K4_TILE + 3) * 8, 256) + 256;
}
EncodeWs carve_encode_ws(void* scratch, uint64_t nchunks) {
    uint8_t* p = (uint8_t*)align_up((size_t)scratch, 256);
    EncodeWs w;
    w.slots = p; p += align_up(nchunks * (uint64_t)sbk::kSlotStride, 256);
    w.lens_in = (uint32_t*)p; p += align_up(nchunks * 4 + 4, 256);
    w.clens = (uint32_t*)p; p += align_up(nchunks * 4 + 4, 256);
    w.crcs = (uint32_t*)p; p += align_up(nchunks * 4 + 4, 256);
    w.offs = (uint64_t*)p; p += align_up((nchunks + 1) * 8, 256);
    w.tiles = (uint64_t*)p;
    return w;
}

// Stream-ordered compress of one logical stream of n bytes at d_in into the final layout at d_out:
// frame=0 -> raw stream (varint + blocks), frame=1 -> frame chunks (optionally preceded by the stream
// identifier). No host synchronisation for n > 0; the outcome lands in *d_result (device).
int compress_stream_ws(Ctx& c, const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap, int frame, int ident,
                       uint64_t* d_chunk_offs, sb_frame_result* d_result, void* scratch, cudaStream_t st, sb_error* err) {
    const uint64_t nchunks64 = (n + SB_MAX_BLOCK - 1) / SB_MAX_BLOCK;
    if (nchunks64 > 0xFFFFFFFFull) return fail(err, SB_TOO_BIG, n, SB_MAX_INPUT);
    const uint32_t nchunks = (uint32_t)nchunks64;
    sbk::FramePlan p;
    memset(&p, 0, sizeof p);
    if (frame) { if (ident && n) { memcpy(p.head, "\xff\x06\x00\x00sNaPpY", 10); p.head_len = 10; } }
    else p.head_len = (uint32_t)put_varint(p.head, n);
    if (n == 0) {
        // nothing to compress: the prefix (raw: the one-byte varint; frame: nothing, src/write.rs:155-157) and the result
        sb_frame_result r;
        memset(&r, 0, sizeof r);
        r.bytes = p.head_len;
        if (p.head_len > cap) { r.status.code = SB_BUFFER_TOO_SMALL; r.status.a = cap; r.status.b = p.head_len; r.bytes = 0; }
        else if (p.head_len) CK(cudaMemcpyAsync(d_out, p.head, p.head_len, cudaMemcpyHostToDevice, st));
        if (d_result) CK(cudaMemcpyAsync(d_result, &r, sizeof r, cudaMemcpyHostToDevice, st));
        if (d_chunk_offs) { const uint64_t z = p.head_len; CK(cudaMemcpyAsync(d_chunk_offs, &z, 8, cudaMemcpyHostToDevice, st)); }
        CK(cudaStreamSynchronize(st));   // the sources above are on this stack frame
        return 0;
    }
    const EncodeWs w = carve_encode_ws(scratch, nchunks);
    k4_fill_lens_kernel<<<(nchunks + 255) / 256, 256, 0, st>>>(w.lens_in, n, nchunks);
    g_launches++;
    sb_batch b;
    memset(&b, 0, sizeof b);
    b.in_base = d_in; b.in_stride = SB_MAX_BLOCK; b.in_lens = w.lens_in;
    b.out_base = w.slots; b.out_stride = sbk::kSlotStride; b.out_cap_uniform = sbk::kSlotStride;
    b.out_lens = w.clens; b.count = nchunks;
    int rc = launch_k1(c, b, frame ? 1u : 0u, frame ? w.crcs : nullptr, st, err);   // frame chunks carry their own varint
    if (rc) return rc;
    p.in = d_in; p.n = n; p.slots = w.slots; p.clens = w.clens; p.crcs = w.crcs; p.nchunks = nchunks;
    p.frame = frame ? 1u : 0u; p.offs = d_chunk_offs ? d_chunk_offs : w.offs; p.tiles = w.tiles;
    p.out = d_out; p.cap = cap; p.result = d_result;
    return launch_assemble(c, p, st, err);
}

// ---- frame decode
struct DecodeWs { sbk::FChunk* chunks; uint64_t *ooff, *tiles; sb_error* statuses; sbk::DecodeCtl* ctl; };
uint64_t decode_ws_bytes(uint64_t max_chunks) {
    return align_up(max_chunks * sizeof(sbk::FChunk) + 64, 256) + align_up((max_chunks + 1) * 8, 256) +
           align_up((max_chunks / sbk::K4_TILE + 3) * 8, 256) + align_up(max_chunks * sizeof(sb_error) + 64, 256) + 512;
}
DecodeWs carve_decode_ws(void* scratch, uint64_t max_chunks) {
    uint8_t* p = (uint8_t*)align_up((size_t)scratch, 256);
    DecodeWs w;
    w.chunks = (sbk::FChunk*)p; p += align_up(max_chunks * sizeof(sbk::FChunk) + 64, 256);
    w.ooff = (uint64_t*)p; p += align_up((max_chunks + 1) * 8, 256);
    w.tiles = (uint64_t*)p; p += align_up((max_chunks / sbk::K4_TILE + 3) * 8, 256);
    w.statuses = (sb_error*)p; p += align_up(max_chunks * sizeof(sb_error) + 64, 256);
    w.ctl = (sbk::DecodeCtl*)p;
    return w;
}
sbk::DecodePlan make_decode_plan(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap, const uint64_t* d_index,
                                 uint32_t index_n, int fragment, sb_frame_result* d_result, void* scratch, uint32_t max_chunks) {
    const DecodeWs w = carve_decode_ws(scratch, max_chunks);
    sbk::DecodePlan p;
    memset(&p, 0, sizeof p);
    p.in = d_in; p.n = n; p.index = d_index; p.index_n = d_index ? index_n : 0; p.fragment = fragment ? 1u : 0u;
    p.chunks = w.chunks; p.cap_chunks = max_chunks; p.ooff = w.ooff; p.tiles = w.tiles; p.statuses = w.statuses; p.ctl = w.ctl;
    p.out = d_out; p.cap = cap; p.result = d_result;
    return p;
}
// phase 1: chunk table + output offsets (ctl->produced, ctl->go valid afterwards)
int decode_index_phase(Ctx& c, const sbk::DecodePlan& p, cudaStream_t st, sb_error* err) {
    CK(cudaMemsetAsync(p.ctl, 0, sizeof(sbk::DecodeCtl), st));
    if (p.index) { k5_parse_kernel<<<p.index_n ? (p.index_n + 255) / 256 : 1, 256, 0, st>>>(p); g_launches++; }
    k5_walk_kernel<<<1, 32, 0, st>>>(p);
    const unsigned ntiles = (p.cap_chunks + sbk::K4_TILE - 1) / sbk::K4_TILE;
    k5_scan_local_kernel<<<ntiles ? ntiles : 1, sbk::K4_TILE, 32 * sizeof(uint32_t), st>>>(p);
    k5_scan_tiles_kernel<<<1, 1024, 1024 * sizeof(uint64_t), st>>>(p);
    g_launches += 3;
    CK(cudaGetLastError());
    return 0;
}
// phase 2: payload decode + checksum + result
int decode_payload_phase(Ctx& c, const sbk::DecodePlan& p, cudaStream_t st, sb_error* err) {
    k5_decode_kernel<<<16 * c.sms, 128, sbk::K3_TABLE_BYTES + 4 * sbk::K2_SMEM_PER_WARP, st>>>(p);
    k5_finish_kernel<<<1, 32, 0, st>>>(p);
    g_launches += 2;
    CK(cudaGetLastError());
    return 0;
}

// ---- batches of raw streams of any size (K7 around K1 / K2)
// grid of a grid-stride kernel over `work` items, `per` items per CTA, at most `most` CTAs
unsigned grid_for(uint64_t work, unsigned per, unsigned most) {
    const uint64_t g = (work + per - 1) / per;
    return g == 0 ? 1u : g > most ? most : (unsigned)g;
}
// p: caller arrays, slots and meta carved; no host synchronisation
int compress_streams_run(Ctx& c, const sbk::StreamsPlan& p, cudaStream_t st, sb_error* err) {
    CK(cudaMemsetAsync(p.ctl, 0, sizeof(sbk::StreamsCtl), st));
    CK(cudaMemsetAsync(&p.ctl->first_bad, 0xFF, 4, st));
    const unsigned utiles = (p.count + sbk::K4_TILE - 1) / sbk::K4_TILE, itiles = (p.max_items + sbk::K4_TILE - 1) / sbk::K4_TILE;
    k7_plan_kernel<<<utiles ? utiles : 1, sbk::K4_TILE, 32 * sizeof(uint32_t), st>>>(p);
    k7_unit_tiles_kernel<<<1, 1024, 1024 * sizeof(uint64_t), st>>>(p);
    k7_expand_kernel<<<grid_for(p.max_items, 256, 16 * c.sms), 256, 0, st>>>(p);
    g_launches += 3;
    CK(cudaGetLastError());
    sb_batch b;
    memset(&b, 0, sizeof b);
    b.in_ptrs = p.item_ptr; b.in_lens = p.item_len;
    b.out_base = p.slots; b.out_stride = sbk::kSlotStride; b.out_cap_uniform = sbk::kSlotStride;
    b.out_lens = p.clens; b.count = p.max_items;
    int rc = launch_k1(c, b, 0u, nullptr, st, err);   // block bodies only: the unit's varint is written by the gather
    if (rc) return rc;
    k7_item_scan_kernel<<<itiles ? itiles : 1, sbk::K4_TILE, 32 * sizeof(uint32_t), st>>>(p);
    k7_item_tiles_kernel<<<1, 1024, 1024 * sizeof(uint64_t), st>>>(p);
    const uint64_t most = p.max_items > p.count ? p.max_items : p.count;
    k7_gather_kernel<<<grid_for(most, 8, 8 * c.sms), 256, 0, st>>>(p);
    g_launches += 3;
    CK(cudaGetLastError());
    return 0;
}
int decompress_streams_run(Ctx& c, const sbk::StreamsDecPlan& p, cudaStream_t st, sb_error* err) {
    CK(cudaMemsetAsync(&p.ctl->first_bad, 0xFF, 4, st));
    const unsigned tiles = (p.count + sbk::K4_TILE - 1) / sbk::K4_TILE;
    k7_dplan_kernel<<<tiles ? tiles : 1, sbk::K4_TILE, 32 * sizeof(uint64_t), st>>>(p);
    k7_dtiles_kernel<<<1, 1024, 1024 * sizeof(uint64_t), st>>>(p);
    k7_dfill_kernel<<<grid_for(p.count, 256, 16 * c.sms), 256, 0, st>>>(p);
    g_launches += 3;
    CK(cudaGetLastError());
    sb_batch b;
    memset(&b, 0, sizeof b);
    b.in_ptrs = p.in_ptrs; b.in_lens = p.k2_in_lens;
    b.out_ptrs = p.k2_out_ptrs; b.out_caps = p.k2_out_caps;
    b.out_lens = p.k2_out_lens; b.statuses = p.statuses; b.count = p.count;
    int rc = launch_k2(c, b, st, err);
    if (rc) return rc;
    k7_dfinish_kernel<<<grid_for(p.count, 256, 16 * c.sms), 256, 0, st>>>(p);
    k7_dresult_kernel<<<1, 32, 0, st>>>(p);
    g_launches += 2;
    CK(cudaGetLastError());
    return 0;
}
uint64_t streams_max_items(uint32_t count, uint64_t total_in) { return (uint64_t)count + total_in / SB_MAX_BLOCK; }
uint64_t streams_slots_bytes(uint64_t max_items) { return align_up(max_items * (uint64_t)sbk::kSlotStride, 256); }

}  // namespace

// =========================================================================
extern "C" {

const char* sb_version(void) { return "snapb200 0.2 (sm_100a)"; }
uint64_t sb_launch_count(void) { return g_launches.load(); }
uint64_t sb_alloc_count(void) { return g_allocs.load(); }

size_t sb_max_compress_len(size_t input_len) {
    uint64_t n = (uint64_t)input_len;
    if (n > SB_MAX_INPUT) return 0;
    uint64_t m = 32 + n + n / 6;
    return m > SB_MAX_INPUT ? 0 : (size_t)m;
}

size_t sb_frame_max_len(size_t n) {
    size_t chunks = (n + SB_MAX_BLOCK - 1) / SB_MAX_BLOCK;
    return 10 + chunks * (8 + (size_t)SB_MAX_CBLOCK);
}

// Pin the calling thread to the CPUs of the NUMA node the device hangs off, so that its pinned allocations and
// staging copies stay local (a rank per GPU on a two-socket box otherwise streams through the far socket).
int sb_bind_host_thread_to_device_numa(int device) {
    char bus[32];
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return -1;
    for (char* q = bus; *q; q++) if (*q >= 'A' && *q <= 'Z') *q = (char)(*q - 'A' + 'a');
    char path[160];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return -1;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return -1;
    cpu_set_t allowed, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) { fclose(f); return -1; }
    int lo, hi, any = 0;
    while (fscanf(f, "%d", &lo) == 1) {
        hi = lo;
        int ch = fgetc(f);
        if (ch == '-') { if (fscanf(f, "%d", &hi) != 1) break; ch = fgetc(f); }
        for (int k = lo; k <= hi && k < CPU_SETSIZE; k++) if (CPU_ISSET(k, &allowed)) { CPU_SET(k, &want); any = 1; }
        if (ch != ',') break;
    }
    fclose(f);
    if (!any) return -1;
    if (sched_setaffinity(0, sizeof want, &want) != 0) return -1;
    return node;
}

// Size the per-device pools of the host entry points ahead of time: waves of up to `wave_units` units with
// `wave_in_bytes` uncompressed and `wave_out_bytes` compressed bytes (both lanes) then run without any allocation.
int sb_reserve(size_t wave_units, size_t wave_in_bytes, size_t wave_out_bytes, sb_error* err) {
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    for (int ln = 0; ln < 2; ln++) {
        Lane& l = c->lane[ln];
        std::lock_guard<std::mutex> lk(l.mu);
        for (int b = 0; b < 2; b++) {
            CK(l.in[b].need((ln == LANE_ENC ? wave_in_bytes : wave_out_bytes) + wave_units * 16 + 64));
            if (ln == LANE_ENC) CK(l.slots[b].need(wave_units * (size_t)sbk::kSlotStride));
            CK(l.compact[b].need((ln == LANE_ENC ? wave_out_bytes : wave_in_bytes) + wave_units * 16 + 64));
            CK(l.lens[b].need(wave_units * 4 + 4));
            CK(l.caps[b].need(wave_units * 8 + 8));
            CK(l.status[b].need(wave_units * sizeof(sb_error) + 64));
            CK(l.ptrs_in[b].need(wave_units * 8 + 8));
            CK(l.ptrs_out[b].need(wave_units * 8 + 8));
            CK(l.ws[b].need(align_up((wave_units / sbk::K4_TILE + 3) * 8, 256) + align_up((wave_units + 1) * 8, 256) + 1024));
            if (ln == LANE_ENC) CK(l.sws[b].need(sbk::k7_meta_bytes(wave_units, wave_units)));
            rc = need_pinned(l, b, wave_units * 24 + 64, err); if (rc) return rc;
            rc = need_pinned(l, 2 + b, wave_units * (4 + sizeof(sb_error)) + 64, err); if (rc) return rc;
        }
        rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    }
    ok(err);
    return 0;
}

uint64_t sb_frame_encode_scratch_bytes(uint64_t n) { return encode_ws_bytes(n); }
uint64_t sb_frame_decode_scratch_bytes(uint32_t max_chunks) { return decode_ws_bytes(max_chunks); }

int sb_compress(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err) {
    if ((!in && n) || !out || !out_n) return fail(err, SB_E_INVALID);
    const size_t need = sb_max_compress_len(n);
    if (need == 0) return fail(err, SB_TOO_BIG, (uint64_t)n, SB_MAX_INPUT);
    if (cap < need) return fail(err, SB_BUFFER_TOO_SMALL, (uint64_t)cap, (uint64_t)need);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_ENC];
    std::lock_guard<std::mutex> lk(l.mu);
    CK(l.in[0].need(n + 64));
    CK(l.compact[0].need(need + 64));
    CK(l.ws[0].need(encode_ws_bytes(n) + sizeof(sb_frame_result) + 256));
    rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    if (n) CK(cudaMemcpyAsync(l.in[0].p, in, n, cudaMemcpyHostToDevice, l.s_compute));
    sb_frame_result* d_res = (sb_frame_result*)((uint8_t*)l.ws[0].p + align_up(encode_ws_bytes(n), 256));
    rc = compress_stream_ws(*c, l.in[0].as<uint8_t>(), n, l.compact[0].as<uint8_t>(), need, 0, 0, nullptr, d_res, l.ws[0].p, l.s_compute, err);
    if (rc) return rc;
    sb_frame_result* res = (sb_frame_result*)l.pinned[4];
    CK(cudaMemcpyAsync(res, d_res, sizeof *res, cudaMemcpyDeviceToHost, l.s_compute));
    CK(cudaStreamSynchronize(l.s_compute));
    if (res->status.code) { if (err) *err = res->status; return (int)res->status.code; }
    CK(cudaMemcpyAsync(out, l.compact[0].p, res->bytes, cudaMemcpyDeviceToHost, l.s_compute));
    CK(cudaStreamSynchronize(l.s_compute));
    *out_n = (size_t)res->bytes;
    ok(err);
    return 0;
}

int sb_decompress_len(const uint8_t* in, size_t n, size_t* out_len, sb_error* err) {
    // reference src/decompress.rs:30-35, 362-374 -- header arithmetic only
    if (!out_len || (!in && n)) return fail(err, SB_E_INVALID);
    if (n == 0) { *out_len = 0; ok(err); return 0; }
    uint64_t v;
    size_t h = get_varint(in, n, &v);
    if (h == 0) return fail(err, SB_HEADER);
    if (v > SB_MAX_INPUT) return fail(err, SB_TOO_BIG, v, SB_MAX_INPUT);
    *out_len = (size_t)v;
    ok(err);
    return 0;
}

int sb_decompress(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err) {
    if ((!in && n) || (!out && cap) || !out_n) return fail(err, SB_E_INVALID);
    if (n == 0) return fail(err, SB_EMPTY);
    if (n > SB_MAX_INPUT) return fail(err, SB_E_INVALID);
    // the header decides how much device output we need; the kernel re-validates everything
    uint64_t v = 0;
    size_t h = get_varint(in, n, &v);
    uint64_t dcap = (h && v <= SB_MAX_INPUT && v <= cap) ? v : 0;
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_DEC];
    std::lock_guard<std::mutex> lk(l.mu);
    CK(l.in[0].need(n + 64));
    CK(l.compact[0].need(dcap + 64));
    CK(l.status[0].need(sizeof(sb_error) + 16));
    rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    CK(cudaMemcpyAsync(l.in[0].p, in, n, cudaMemcpyHostToDevice, l.s_compute));
    sb_batch b;
    memset(&b, 0, sizeof b);
    b.in_base = l.in[0].as<uint8_t>(); b.in_len_uniform = (uint32_t)n;
    b.out_base = l.compact[0].as<uint8_t>();
    b.out_cap_uniform = cap > SB_MAX_INPUT ? (uint32_t)SB_MAX_INPUT : (uint32_t)cap;
    b.statuses = l.status[0].as<sb_error>();
    b.out_lens = (uint32_t*)((uint8_t*)l.status[0].p + sizeof(sb_error));
    b.count = 1;
    rc = launch_k2(*c, b, l.s_compute, err);
    if (rc) return rc;
    struct Res { sb_error e; uint32_t len; uint32_t pad; };
    Res* res = (Res*)l.pinned[4];
    CK(cudaMemcpyAsync(res, l.status[0].p, sizeof(sb_error) + 8, cudaMemcpyDeviceToHost, l.s_compute));
    CK(cudaStreamSynchronize(l.s_compute));
    if (res->e.code) { if (err) *err = res->e; return (int)res->e.code; }
    if (res->len) CK(cudaMemcpy(out, l.compact[0].p, res->len, cudaMemcpyDeviceToHost));
    *out_n = res->len;
    ok(err);
    return 0;
}

int sb_crc32c_masked(const uint8_t* in, size_t n, uint32_t* out, sb_error* err) {
    if ((!in && n) || !out || n > SB_MAX_INPUT) return fail(err, SB_E_INVALID);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_ENC];
    std::lock_guard<std::mutex> lk(l.mu);
    CK(l.in[0].need(n + 64));
    CK(l.lens[0].need(16));
    if (n) CK(cudaMemcpyAsync(l.in[0].p, in, n, cudaMemcpyHostToDevice, l.s_compute));
    sb_batch b;
    memset(&b, 0, sizeof b);
    b.in_base = l.in[0].as<uint8_t>(); b.in_len_uniform = (uint32_t)n;
    b.out_lens = l.lens[0].as<uint32_t>(); b.count = 1;
    rc = launch_k3(*c, b, l.s_compute, err);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, l.lens[0].p, 4, cudaMemcpyDeviceToHost, l.s_compute));
    CK(cudaStreamSynchronize(l.s_compute));
    ok(err);
    return 0;
}

// ---------------------------------------------------------- device batches
int sb_compress_batch_device(const sb_batch* batch, void* stream, sb_error* err) {
    if (!batch || !batch->out_lens) return fail(err, SB_E_INVALID);
    if (!batch->in_lens && batch->in_len_uniform > SB_MAX_BLOCK) return fail(err, SB_TOO_BIG, batch->in_len_uniform, SB_MAX_BLOCK);
    if (!batch->out_caps && !batch->in_lens && batch->out_cap_uniform < sb_max_compress_len(batch->in_len_uniform))
        return fail(err, SB_BUFFER_TOO_SMALL, batch->out_cap_uniform, sb_max_compress_len(batch->in_len_uniform));
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    rc = launch_k1(*c, *batch, 1u, nullptr, (cudaStream_t)stream, err);
    if (rc) return rc;
    ok(err);
    return 0;
}

int sb_decompress_batch_device(const sb_batch* batch, void* stream, sb_error* err) {
    if (!batch) return fail(err, SB_E_INVALID);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    rc = launch_k2(*c, *batch, (cudaStream_t)stream, err);
    if (rc) return rc;
    ok(err);
    return 0;
}

int sb_crc32c_masked_batch_device(const sb_batch* batch, void* stream, sb_error* err) {
    if (!batch || !batch->out_lens) return fail(err, SB_E_INVALID);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    rc = launch_k3(*c, *batch, (cudaStream_t)stream, err);
    if (rc) return rc;
    ok(err);
    return 0;
}

int sb_generate_blocks_device(const uint8_t* d_text, uint64_t text_len, uint8_t* d_out, uint64_t stride,
                              uint32_t len, uint64_t first, uint64_t count, uint64_t mul, void* stream, sb_error* err) {
    if (!d_text || !d_out || text_len < len) return fail(err, SB_E_INVALID);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    if (count == 0) return 0;
    sbk::GenPlan g{d_text, text_len, d_out, stride, len, first, count, mul};
    uint64_t blocks = (count + 7) / 8;
    unsigned grid = (unsigned)(16 * c->sms);
    if (grid > blocks) grid = (unsigned)blocks;
    k6_generate_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g);
    g_launches++;
    CK(cudaGetLastError());
    ok(err);
    return 0;
}

// ------------------------------------------------------------ host batches
// Waves of units are staged H2D on one stream, run on a second, and drained D2H
// on a third, double buffered, so PCIe traffic overlaps the kernels. The host thread
// never waits for a copy: ordering between the streams is all events.
namespace {
const size_t WAVE_BYTES = (size_t)1 << 30;

struct Wave { size_t first, count; uint64_t in_bytes; };

extern "C++" {
template <class Len>   // uint32_t: 64KB units; uint64_t: raw streams of any size
std::vector<Wave> plan_waves(const Len* in_lens, size_t count, const uint32_t* out_caps) {
    std::vector<Wave> w;
    size_t i = 0;
    while (i < count) {
        Wave cur{i, 0, 0};
        uint64_t outb = 0;
        // ramp-up: the first waves are small so the first kernel starts after ~1 ms of H2D, not ~10
        const size_t limit = w.size() == 0 ? WAVE_BYTES / 16 : w.size() == 1 ? WAVE_BYTES / 4 : WAVE_BYTES;
        while (i < count && cur.count < (1u << 20)) {
            uint64_t add = in_lens[i], oadd = out_caps ? out_caps[i] : 0;
            if (cur.count && (cur.in_bytes + add > limit || outb + oadd > 2 * limit)) break;
            cur.in_bytes += add + 16; outb += oadd; cur.count++; i++;
        }
        w.push_back(cur);
    }
    return w;
}
}  // extern "C++"

// Shared body of sb_compress_batch_host (caller's offsets) and sb_compress_batch_host_packed (the library packs the
// streams back to back and REPORTS the offsets: a caller cannot know compressed sizes in advance).
int compress_batch_host_impl(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                             uint8_t* out_base, const uint64_t* out_offs_in, uint64_t out_cap_total, uint64_t* out_offs_ret,
                             uint32_t* out_lens, size_t count, sb_error* err) {
    const bool packed = out_offs_in == nullptr;
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_ENC];
    std::lock_guard<std::mutex> lk(l.mu);
    std::vector<Wave> waves = plan_waves(in_lens, count, nullptr);
    std::vector<uint64_t> doff;
    auto stage_in = [&](size_t wi) -> int {
        const Wave& w = waves[wi];
        const int b = (int)(wi & 1);
        CK(l.in[b].need(w.in_bytes + 64));
        CK(l.slots[b].need(w.count * (size_t)sbk::kSlotStride));
        CK(l.lens[b].need(w.count * 4 + 4));
        CK(l.caps[b].need(w.count * 4 + 4));
        CK(l.ptrs_in[b].need(w.count * 8 + 8));
        // coalesce units that are contiguous on the host into single copies
        doff.resize(w.count);
        uint64_t at = 0;
        size_t i = 0;
        while (i < w.count) {
            size_t j = i;
            uint64_t run = 0;
            const uint64_t h0 = in_offs[w.first + i];
            while (j < w.count && in_offs[w.first + j] == h0 + run) { doff[j] = at + run; run += in_lens[w.first + j]; j++; }
            if (run) CK(cudaMemcpyAsync(l.in[b].as<uint8_t>() + at, in_base + h0, run, cudaMemcpyHostToDevice, l.s_h2d));
            at += (run + 15) & ~(uint64_t)15;
            i = j;
        }
        // pinned[b] was last read by the H2D of wave wi-2, whose kernel has completed (the loop below waited for it)
        { int prc = need_pinned(l, b, w.count * 12 + 64, err); if (prc) return prc; }
        uint64_t* ptrs = (uint64_t*)l.pinned[b];
        uint32_t* plen = (uint32_t*)(ptrs + w.count);
        for (size_t k = 0; k < w.count; k++) ptrs[k] = (uint64_t)(uintptr_t)(l.in[b].as<uint8_t>() + doff[k]);
        memcpy(plen, in_lens + w.first, w.count * 4);
        CK(cudaMemcpyAsync(l.ptrs_in[b].p, ptrs, w.count * 8, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaMemcpyAsync(l.caps[b].p, plen, w.count * 4, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaEventRecord(l.ev_in[b], l.s_h2d));
        return 0;
    };
    const bool timing = getenv("SNAPB200_TIMING") != nullptr;
    auto now_ms = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    const double t_begin = now_ms();
    uint64_t packed_at = 0;
    if (!waves.empty()) { rc = stage_in(0); if (rc) return rc; }
    for (size_t wi = 0; wi < waves.size(); wi++) {
        const Wave& w = waves[wi];
        const int b = (int)(wi & 1);
        if (timing) fprintf(stderr, "[compress wave %zu] t=%.2f launch (count %zu)\n", wi, now_ms() - t_begin, w.count);
        CK(cudaStreamWaitEvent(l.s_compute, l.ev_in[b], 0));
        if (wi >= 2) CK(cudaStreamWaitEvent(l.s_compute, l.ev_out[b], 0));   // wave wi-2 (same buffers) fully drained
        sb_batch bt;
        memset(&bt, 0, sizeof bt);
        bt.in_ptrs = (const uint8_t* const*)l.ptrs_in[b].p; bt.in_lens = l.caps[b].as<uint32_t>();
        bt.out_base = l.slots[b].as<uint8_t>(); bt.out_stride = sbk::kSlotStride; bt.out_cap_uniform = sbk::kSlotStride;
        bt.out_lens = l.lens[b].as<uint32_t>(); bt.count = (uint32_t)w.count;
        rc = launch_k1(*c, bt, 1u, nullptr, l.s_compute, err);
        if (rc) return rc;
        // pack the wave's streams back to back on the device (offsets by scan), so the drain is one D2H
        uint64_t worst = 0;
        for (size_t k = 0; k < w.count; k++) worst += sb_max_compress_len(in_lens[w.first + k]);
        CK(l.compact[b].need(worst + 64));
        const size_t tiles_bytes = align_up((w.count / sbk::K4_TILE + 3) * 8, 256);
        CK(l.ws[b].need(tiles_bytes + align_up((w.count + 1) * 8, 256) + 1024));
        sbk::FramePlan p;
        memset(&p, 0, sizeof p);
        p.slots = l.slots[b].as<uint8_t>(); p.clens = l.lens[b].as<uint32_t>(); p.nchunks = (uint32_t)w.count;
        p.frame = 0; p.head_len = 0; p.tiles = (uint64_t*)l.ws[b].p; p.offs = (uint64_t*)((uint8_t*)l.ws[b].p + tiles_bytes);
        p.out = l.compact[b].as<uint8_t>(); p.cap = l.compact[b].cap; p.result = nullptr;
        rc = launch_assemble(*c, p, l.s_compute, err);
        if (rc) return rc;
        // results come back through pinned staging: a D2H copy into the caller's (pageable) array
        // would block this thread until the kernel is done and serialise the next wave's H2D behind it
        { int prc = need_pinned(l, 2 + b, w.count * 12 + 64, err); if (prc) return prc; }
        uint32_t* plens = (uint32_t*)l.pinned[2 + b];
        uint64_t* poffs = (uint64_t*)(plens + ((w.count + 2) & ~(size_t)1));
        CK(cudaMemcpyAsync(plens, l.lens[b].p, w.count * 4, cudaMemcpyDeviceToHost, l.s_compute));
        CK(cudaMemcpyAsync(poffs, p.offs, (w.count + 1) * 8, cudaMemcpyDeviceToHost, l.s_compute));
        CK(cudaEventRecord(l.ev_k[b], l.s_compute));
        if (wi + 1 < waves.size()) { rc = stage_in(wi + 1); if (rc) return rc; }   // overlaps the kernel above
        if (timing) fprintf(stderr, "[compress wave %zu] t=%.2f staged next\n", wi, now_ms() - t_begin);
        CK(cudaEventSynchronize(l.ev_k[b]));
        memcpy(out_lens + w.first, plens, w.count * 4);
        const uint64_t run = poffs[w.count];
        if (timing) fprintf(stderr, "[compress wave %zu] t=%.2f kernel done (%llu bytes)\n", wi, now_ms() - t_begin, (unsigned long long)run);
        CK(cudaStreamWaitEvent(l.s_d2h, l.ev_k[b], 0));
        if (packed) {
            if (packed_at + run > out_cap_total) return fail(err, SB_BUFFER_TOO_SMALL, out_cap_total, packed_at + run);
            for (size_t k = 0; k < w.count; k++) out_offs_ret[w.first + k] = packed_at + poffs[k];
            if (run) CK(cudaMemcpyAsync(out_base + packed_at, l.compact[b].p, run, cudaMemcpyDeviceToHost, l.s_d2h));
            packed_at += run;
        } else {
            // caller's offsets: host-contiguous destinations travel as one copy per run
            size_t k = 0;
            while (k < w.count) {
                size_t j = k;
                uint64_t len = 0;
                const uint64_t h0 = out_offs_in[w.first + k];
                while (j < w.count && out_offs_in[w.first + j] == h0 + len) { len += plens[j]; j++; }
                if (len) CK(cudaMemcpyAsync(out_base + h0, l.compact[b].as<uint8_t>() + poffs[k], len, cudaMemcpyDeviceToHost, l.s_d2h));
                k = j;
            }
        }
        CK(cudaEventRecord(l.ev_out[b], l.s_d2h));
    }
    if (packed) out_offs_ret[count] = packed_at;
    CK(cudaStreamSynchronize(l.s_d2h));
    CK(cudaStreamSynchronize(l.s_compute));
    ok(err);
    return 0;
}
}  // namespace

int sb_compress_batch_host(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                           uint8_t* out_base, const uint64_t* out_offs, const uint32_t* out_caps,
                           uint32_t* out_lens, size_t count, sb_error* err) {
    if (!in_base || !in_offs || !in_lens || !out_base || !out_offs || !out_lens) return fail(err, SB_E_INVALID);
    for (size_t i = 0; i < count; i++) {
        if (in_lens[i] > SB_MAX_BLOCK) return fail(err, SB_TOO_BIG, in_lens[i], SB_MAX_BLOCK);   // one block per unit in the batched form
        if (out_caps && out_caps[i] < sb_max_compress_len(in_lens[i]))
            return fail(err, SB_BUFFER_TOO_SMALL, out_caps[i], sb_max_compress_len(in_lens[i]));
    }
    return compress_batch_host_impl(in_base, in_offs, in_lens, out_base, out_offs, 0, nullptr, out_lens, count, err);
}

int sb_compress_batch_host_packed(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                                  uint8_t* out_base, uint64_t out_cap, uint64_t* out_offs, uint32_t* out_lens,
                                  size_t count, sb_error* err) {
    if (!in_base || !in_offs || !in_lens || !out_base || !out_offs || !out_lens) return fail(err, SB_E_INVALID);
    for (size_t i = 0; i < count; i++)
        if (in_lens[i] > SB_MAX_BLOCK) return fail(err, SB_TOO_BIG, in_lens[i], SB_MAX_BLOCK);
    return compress_batch_host_impl(in_base, in_offs, in_lens, out_base, nullptr, out_cap, out_offs, out_lens, count, err);
}

int sb_decompress_batch_host(const uint8_t* in_base, const uint64_t* in_offs, const uint32_t* in_lens,
                             uint8_t* out_base, const uint64_t* out_offs, const uint32_t* out_caps,
                             uint32_t* out_lens, sb_error* statuses, size_t count, sb_error* err) {
    if (!in_base || !in_offs || !in_lens || !out_base || !out_offs || !out_caps || !out_lens || !statuses)
        return fail(err, SB_E_INVALID);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_DEC];
    std::lock_guard<std::mutex> lk(l.mu);
    std::vector<Wave> waves = plan_waves(in_lens, count, out_caps);
    std::vector<uint64_t> pout[2];
    // H2D of wave wi into buffer set wi&1 (copy stream; overlaps the previous wave's kernel)
    auto stage_in = [&](size_t wi) -> int {
        const Wave& w = waves[wi];
        const int b = (int)(wi & 1);
        uint64_t out_total = 0;
        for (size_t k = 0; k < w.count; k++) out_total += ((uint64_t)out_caps[w.first + k] + 15) & ~(uint64_t)15;
        CK(l.in[b].need(w.in_bytes + 64));
        CK(l.compact[b].need(out_total + 64));
        CK(l.lens[b].need(w.count * 4 + 4));
        CK(l.caps[b].need(w.count * 8 + 8));
        CK(l.status[b].need(w.count * sizeof(sb_error)));
        CK(l.ptrs_in[b].need(w.count * 8 + 8));
        CK(l.ptrs_out[b].need(w.count * 8 + 8));
        { int prc = need_pinned(l, b, w.count * 24 + 64, err); if (prc) return prc; }
        uint64_t* sp = (uint64_t*)l.pinned[b];      // [count] in pointers, [count] out pointers, then lengths and caps
        pout[b].resize(w.count);
        uint64_t at = 0, oat = 0;
        size_t i = 0;
        while (i < w.count) {                                      // host-contiguous units travel as one copy
            size_t j = i;
            uint64_t run = 0;
            const uint64_t h0 = in_offs[w.first + i];
            while (j < w.count && in_offs[w.first + j] == h0 + run) {
                sp[j] = (uint64_t)(uintptr_t)(l.in[b].as<uint8_t>() + at + run); run += in_lens[w.first + j]; j++;
            }
            if (run) CK(cudaMemcpyAsync(l.in[b].as<uint8_t>() + at, in_base + h0, run, cudaMemcpyHostToDevice, l.s_h2d));
            at += (run + 15) & ~(uint64_t)15;
            i = j;
        }
        for (size_t k = 0; k < w.count; k++) {
            pout[b][k] = (uint64_t)(uintptr_t)(l.compact[b].as<uint8_t>() + oat);
            sp[w.count + k] = pout[b][k];
            oat += ((uint64_t)out_caps[w.first + k] + 15) & ~(uint64_t)15;
        }
        uint32_t* sl = (uint32_t*)(sp + 2 * w.count);
        memcpy(sl, in_lens + w.first, w.count * 4);
        memcpy(sl + w.count, out_caps + w.first, w.count * 4);
        CK(cudaMemcpyAsync(l.ptrs_in[b].p, sp, w.count * 8, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaMemcpyAsync(l.ptrs_out[b].p, sp + w.count, w.count * 8, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaMemcpyAsync(l.caps[b].p, sl, w.count * 8, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaEventRecord(l.ev_in[b], l.s_h2d));
        return 0;
    };
    if (!waves.empty()) { rc = stage_in(0); if (rc) return rc; }
    for (size_t wi = 0; wi < waves.size(); wi++) {
        const Wave& w = waves[wi];
        const int b = (int)(wi & 1);
        CK(cudaStreamWaitEvent(l.s_compute, l.ev_in[b], 0));
        if (wi >= 2) CK(cudaStreamWaitEvent(l.s_compute, l.ev_out[b], 0));   // wave wi-2 (same buffers) fully drained
        sb_batch bt;
        memset(&bt, 0, sizeof bt);
        bt.in_ptrs = (const uint8_t* const*)l.ptrs_in[b].p; bt.in_lens = l.caps[b].as<uint32_t>();
        bt.out_ptrs = (uint8_t* const*)l.ptrs_out[b].p; bt.out_caps = l.caps[b].as<uint32_t>() + w.count;
        bt.out_lens = l.lens[b].as<uint32_t>(); bt.statuses = l.status[b].as<sb_error>(); bt.count = (uint32_t)w.count;
        rc = launch_k2(*c, bt, l.s_compute, err);
        if (rc) return rc;
        { int prc = need_pinned(l, 2 + b, w.count * (4 + sizeof(sb_error)) + 64, err); if (prc) return prc; }
        sb_error* pst = (sb_error*)l.pinned[2 + b];
        uint32_t* pln = (uint32_t*)(pst + w.count);
        CK(cudaMemcpyAsync(pln, l.lens[b].p, w.count * 4, cudaMemcpyDeviceToHost, l.s_compute));
        CK(cudaMemcpyAsync(pst, l.status[b].p, w.count * sizeof(sb_error), cudaMemcpyDeviceToHost, l.s_compute));
        CK(cudaEventRecord(l.ev_k[b], l.s_compute));
        // the next wave's staging writes pout[b^1] only: this wave's pout[b] stays valid for the drain below
        if (wi + 1 < waves.size()) { rc = stage_in(wi + 1); if (rc) return rc; }   // overlaps the kernel above and the previous drain
        CK(cudaEventSynchronize(l.ev_k[b]));
        memcpy(out_lens + w.first, pln, w.count * 4);
        memcpy(statuses + w.first, pst, w.count * sizeof(sb_error));
        // drain on the third stream; contiguous destinations whose caps are exactly filled go out as one copy
        CK(cudaStreamWaitEvent(l.s_d2h, l.ev_k[b], 0));
        const uint64_t cbase = (uint64_t)(uintptr_t)l.compact[b].p;
        size_t k = 0;
        while (k < w.count) {
            size_t j = k;
            uint64_t run = 0;
            const uint64_t h0 = out_offs[w.first + k];
            const uint64_t d0 = pout[b][k] - cbase;
            while (j < w.count && out_offs[w.first + j] == h0 + run && pout[b][j] - cbase == d0 + run) {
                run += out_lens[w.first + j];
                const bool full = out_lens[w.first + j] == out_caps[w.first + j] && (out_caps[w.first + j] & 15u) == 0;
                j++;
                if (!full) break;
            }
            if (run) CK(cudaMemcpyAsync(out_base + h0, l.compact[b].as<uint8_t>() + d0, run, cudaMemcpyDeviceToHost, l.s_d2h));
            k = j;
        }
        CK(cudaEventRecord(l.ev_out[b], l.s_d2h));
    }
    CK(cudaStreamSynchronize(l.s_d2h));
    CK(cudaStreamSynchronize(l.s_compute));
    ok(err);
    return 0;
}

// ------------------------------------------------------- batches of raw streams
uint64_t sb_compress_streams_scratch_bytes(uint32_t count, uint64_t total_in) {
    const uint64_t m = streams_max_items(count, total_in);
    return streams_slots_bytes(m) + sbk::k7_meta_bytes(count, m);
}

int sb_compress_streams_device_ws(const uint8_t* const* d_in_ptrs, const uint64_t* d_in_lens, uint32_t count,
                                  uint64_t total_in, uint8_t* d_out, uint64_t cap, uint64_t* d_out_offs,
                                  sb_error* d_statuses, sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes,
                                  void* stream, sb_error* err) {
    if ((count && (!d_in_ptrs || !d_in_lens)) || (!d_out && cap) || !d_out_offs || !d_result || !scratch) return fail(err, SB_E_INVALID);
    const uint64_t m = streams_max_items(count, total_in);
    if (m > 0xFFFFFFFFull) return fail(err, SB_E_INVALID, m, 0xFFFFFFFFull);   // K1 counts units in 32 bits
    const uint64_t need = sb_compress_streams_scratch_bytes(count, total_in);
    if (scratch_bytes < need) return fail(err, SB_BUFFER_TOO_SMALL, scratch_bytes, need);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    sbk::StreamsPlan p;
    memset(&p, 0, sizeof p);
    p.in_ptrs = d_in_ptrs; p.in_lens = d_in_lens; p.count = count; p.max_items = (uint32_t)m; p.total_in = total_in;
    p.slots = (uint8_t*)align_up((size_t)scratch, 256);
    sbk::k7_carve_meta(p, p.slots + streams_slots_bytes(m));
    p.out = d_out; p.cap = cap; p.out_offs = d_out_offs; p.statuses = d_statuses; p.result = d_result;
    rc = compress_streams_run(*c, p, (cudaStream_t)stream, err);
    if (rc) return rc;
    ok(err);
    return 0;
}

uint64_t sb_decompress_streams_scratch_bytes(uint32_t count) { return sbk::k7_dec_bytes(count); }

int sb_decompress_streams_device_ws(const uint8_t* const* d_in_ptrs, const uint64_t* d_in_lens, uint32_t count,
                                    uint8_t* d_out, uint64_t cap, uint64_t* d_out_offs, sb_error* d_statuses,
                                    sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes,
                                    void* stream, sb_error* err) {
    if ((count && (!d_in_ptrs || !d_in_lens || !d_statuses)) || (!d_out && cap) || !d_out_offs || !d_result || !scratch)
        return fail(err, SB_E_INVALID);
    if (scratch_bytes < sbk::k7_dec_bytes(count)) return fail(err, SB_BUFFER_TOO_SMALL, scratch_bytes, sbk::k7_dec_bytes(count));
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    sbk::StreamsDecPlan p;
    memset(&p, 0, sizeof p);
    p.in_ptrs = d_in_ptrs; p.in_lens = d_in_lens; p.count = count;
    p.out = d_out; p.cap = cap; p.out_offs = d_out_offs; p.statuses = d_statuses; p.result = d_result;
    sbk::k7_carve_dec(p, scratch);
    rc = decompress_streams_run(*c, p, (cudaStream_t)stream, err);
    if (rc) return rc;
    ok(err);
    return 0;
}

// Host form: waves as in sb_compress_batch_host_packed (H2D, K7 + K1, D2H on three streams, double buffered); a unit
// larger than a wave gets a wave of its own. Every unit is checked up front, so a wave never fails on the device.
int sb_compress_streams_host_packed(const uint8_t* in_base, const uint64_t* in_offs, const uint64_t* in_lens, size_t count,
                                    uint8_t* out_base, uint64_t out_cap, uint64_t* out_offs, sb_error* err) {
    if ((count && (!in_base || !in_offs || !in_lens || !out_base)) || !out_offs) return fail(err, SB_E_INVALID);
    for (size_t i = 0; i < count; i++)
        if (sb_max_compress_len(in_lens[i]) == 0) return fail(err, SB_TOO_BIG, in_lens[i], SB_MAX_INPUT);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_ENC];
    std::lock_guard<std::mutex> lk(l.mu);
    const std::vector<Wave> waves = plan_waves(in_lens, count, (const uint32_t*)nullptr);
    auto stage_in = [&](size_t wi) -> int {
        const Wave& w = waves[wi];
        const int b = (int)(wi & 1);
        CK(l.in[b].need(w.in_bytes + 64));
        CK(l.ptrs_in[b].need(w.count * 8 + 8));
        CK(l.caps[b].need(w.count * 8 + 8));
        // pinned[b] was last read by the H2D of wave wi-2, whose kernels have completed (the loop below waited for them)
        { int prc = need_pinned(l, b, w.count * 16 + 64, err); if (prc) return prc; }
        uint64_t* ptrs = (uint64_t*)l.pinned[b];
        uint64_t* lens = ptrs + w.count;
        uint64_t at = 0;
        size_t i = 0;
        while (i < w.count) {                                      // host-contiguous units travel as one copy
            size_t j = i;
            uint64_t run = 0;
            const uint64_t h0 = in_offs[w.first + i];
            while (j < w.count && in_offs[w.first + j] == h0 + run) {
                ptrs[j] = (uint64_t)(uintptr_t)(l.in[b].as<uint8_t>() + at + run); run += in_lens[w.first + j]; j++;
            }
            if (run) CK(cudaMemcpyAsync(l.in[b].as<uint8_t>() + at, in_base + h0, run, cudaMemcpyHostToDevice, l.s_h2d));
            at += (run + 15) & ~(uint64_t)15;
            i = j;
        }
        memcpy(lens, in_lens + w.first, w.count * 8);
        CK(cudaMemcpyAsync(l.ptrs_in[b].p, ptrs, w.count * 8, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaMemcpyAsync(l.caps[b].p, lens, w.count * 8, cudaMemcpyHostToDevice, l.s_h2d));
        CK(cudaEventRecord(l.ev_in[b], l.s_h2d));
        return 0;
    };
    auto drain_all = [&]() { cudaStreamSynchronize(l.s_h2d); cudaStreamSynchronize(l.s_compute); cudaStreamSynchronize(l.s_d2h); };
    uint64_t packed_at = 0;
    if (!waves.empty()) { rc = stage_in(0); if (rc) return rc; }
    for (size_t wi = 0; wi < waves.size(); wi++) {
        const Wave& w = waves[wi];
        const int b = (int)(wi & 1);
        CK(cudaStreamWaitEvent(l.s_compute, l.ev_in[b], 0));
        if (wi >= 2) CK(cudaStreamWaitEvent(l.s_compute, l.ev_out[b], 0));   // wave wi-2 (same buffers) fully drained
        uint64_t worst = 0;
        for (size_t k = 0; k < w.count; k++) worst += sb_max_compress_len(in_lens[w.first + k]);
        const uint64_t m = streams_max_items((uint32_t)w.count, w.in_bytes);
        CK(l.compact[b].need(worst + 64));
        CK(l.slots[b].need(m * (size_t)sbk::kSlotStride));
        CK(l.sws[b].need(sbk::k7_meta_bytes(w.count, m)));
        CK(l.ptrs_out[b].need(w.count * 8 + 8));
        sbk::StreamsPlan p;
        memset(&p, 0, sizeof p);
        p.in_ptrs = (const uint8_t* const*)l.ptrs_in[b].p; p.in_lens = l.caps[b].as<uint64_t>();
        p.count = (uint32_t)w.count; p.max_items = (uint32_t)m; p.total_in = w.in_bytes;
        p.slots = l.slots[b].as<uint8_t>();
        p.result = sbk::k7_carve_meta(p, l.sws[b].p);
        p.out = l.compact[b].as<uint8_t>(); p.cap = l.compact[b].cap; p.out_offs = l.ptrs_out[b].as<uint64_t>();
        rc = compress_streams_run(*c, p, l.s_compute, err);
        if (rc) { drain_all(); return rc; }
        { int prc = need_pinned(l, 2 + b, w.count * 8 + 8 + sizeof(sb_frame_result) + 64, err); if (prc) { drain_all(); return prc; } }
        sb_frame_result* pres = (sb_frame_result*)l.pinned[2 + b];
        uint64_t* poffs = (uint64_t*)(pres + 1);
        CK(cudaMemcpyAsync(pres, p.result, sizeof *pres, cudaMemcpyDeviceToHost, l.s_compute));
        CK(cudaMemcpyAsync(poffs, p.out_offs, (w.count + 1) * 8, cudaMemcpyDeviceToHost, l.s_compute));
        CK(cudaEventRecord(l.ev_k[b], l.s_compute));
        if (wi + 1 < waves.size()) { rc = stage_in(wi + 1); if (rc) { drain_all(); return rc; } }   // overlaps the kernels above
        CK(cudaEventSynchronize(l.ev_k[b]));
        if (pres->status.code) { const sb_error e = pres->status; drain_all(); if (err) *err = e; return (int)e.code; }
        const uint64_t run = poffs[w.count];
        if (packed_at + run > out_cap) { drain_all(); return fail(err, SB_BUFFER_TOO_SMALL, out_cap, packed_at + run); }
        for (size_t k = 0; k < w.count; k++) out_offs[w.first + k] = packed_at + poffs[k];
        CK(cudaStreamWaitEvent(l.s_d2h, l.ev_k[b], 0));
        if (run) CK(cudaMemcpyAsync(out_base + packed_at, l.compact[b].p, run, cudaMemcpyDeviceToHost, l.s_d2h));
        CK(cudaEventRecord(l.ev_out[b], l.s_d2h));
        packed_at += run;
    }
    out_offs[count] = packed_at;
    CK(cudaStreamSynchronize(l.s_d2h));
    CK(cudaStreamSynchronize(l.s_compute));
    ok(err);
    return 0;
}

// -------------------------------------------------------------- frame format
// Stream-ordered, caller-provided scratch, no allocation, no host synchronisation (n > 0).
int sb_frame_encode_device_ws(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap, int include_ident,
                              uint64_t* d_chunk_offs, sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes,
                              void* stream, sb_error* err) {
    if ((!d_in && n) || (!d_out && n) || !d_result || (!scratch && n)) return fail(err, SB_E_INVALID);
    if (scratch_bytes < encode_ws_bytes(n)) return fail(err, SB_BUFFER_TOO_SMALL, scratch_bytes, encode_ws_bytes(n));
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    rc = compress_stream_ws(*c, d_in, n, d_out, cap, 1, include_ident, d_chunk_offs, d_result, scratch,
                            (cudaStream_t)stream, err);
    if (rc) return rc;
    ok(err);
    return 0;
}

int sb_frame_encode_device(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap,
                           int include_ident, uint64_t* out_n, void* stream, sb_error* err) {
    if ((!d_in && n) || !out_n || (!d_out && n)) return fail(err, SB_E_INVALID);
    if (cap < sb_frame_max_len(n) - (include_ident ? 0 : 10)) return fail(err, SB_BUFFER_TOO_SMALL, cap, sb_frame_max_len(n));
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_ENC];
    std::lock_guard<std::mutex> lk(l.mu);
    cudaStream_t st = (cudaStream_t)stream;
    CK(l.ws[0].need(encode_ws_bytes(n) + sizeof(sb_frame_result) + 256));
    rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    sb_frame_result* d_res = (sb_frame_result*)((uint8_t*)l.ws[0].p + align_up(encode_ws_bytes(n), 256));
    rc = compress_stream_ws(*c, d_in, n, d_out, cap, 1, include_ident, nullptr, d_res, l.ws[0].p, st, err);
    if (rc) return rc;
    sb_frame_result* res = (sb_frame_result*)l.pinned[4];
    CK(cudaMemcpyAsync(res, d_res, sizeof *res, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (res->status.code) { if (err) *err = res->status; return (int)res->status.code; }
    *out_n = res->bytes;
    ok(err);
    return 0;
}

int sb_frame_encode_ex(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, int include_ident, sb_error* err);
int sb_frame_encode(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err) {
    return sb_frame_encode_ex(in, n, out, cap, out_n, 1, err);
}
int sb_frame_encode_ex(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, int include_ident, sb_error* err) {
    if ((!in && n) || !out_n || (!out && n)) return fail(err, SB_E_INVALID);
    if (n == 0) { *out_n = 0; ok(err); return 0; }              // src/write.rs:155-157: nothing is written
    if (cap < sb_frame_max_len(n)) return fail(err, SB_BUFFER_TOO_SMALL, cap, sb_frame_max_len(n));
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_ENC];
    std::lock_guard<std::mutex> lk(l.mu);
    CK(l.in[1].need(n + 64));
    CK(l.compact[1].need(sb_frame_max_len(n) + 64));
    CK(l.ws[1].need(encode_ws_bytes(n) + sizeof(sb_frame_result) + 256));
    rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    CK(cudaMemcpyAsync(l.in[1].p, in, n, cudaMemcpyHostToDevice, l.s_compute));
    sb_frame_result* d_res = (sb_frame_result*)((uint8_t*)l.ws[1].p + align_up(encode_ws_bytes(n), 256));
    rc = compress_stream_ws(*c, l.in[1].as<uint8_t>(), n, l.compact[1].as<uint8_t>(), sb_frame_max_len(n), 1, include_ident,
                            nullptr, d_res, l.ws[1].p, l.s_compute, err);
    if (rc) return rc;
    sb_frame_result* res = (sb_frame_result*)l.pinned[4];
    CK(cudaMemcpyAsync(res, d_res, sizeof *res, cudaMemcpyDeviceToHost, l.s_compute));
    CK(cudaStreamSynchronize(l.s_compute));
    if (res->status.code) { if (err) *err = res->status; return (int)res->status.code; }
    CK(cudaMemcpyAsync(out, l.compact[1].p, res->bytes, cudaMemcpyDeviceToHost, l.s_compute));
    CK(cudaStreamSynchronize(l.s_compute));
    *out_n = (size_t)res->bytes;
    ok(err);
    return 0;
}

// Device-resident frame decode, stream ordered, caller-provided scratch (reference src/read.rs:104-239).
//   d_chunk_offs/nchunks: optional index (offset of every chunk header, d_chunk_offs[nchunks] = n) -- the array
//     sb_frame_encode_device_ws emits; without it one thread walks the headers (~1 us per chunk).
//   flags bit0: the stream has no identifier (a rank's fragment of a sharded stream).
int sb_frame_decode_device_ws(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap,
                              const uint64_t* d_chunk_offs, uint32_t nchunks, uint32_t flags,
                              sb_frame_result* d_result, void* scratch, uint64_t scratch_bytes, uint32_t max_chunks,
                              void* stream, sb_error* err) {
    if ((!d_in && n) || (!d_out && cap) || !d_result || !scratch || max_chunks == 0) return fail(err, SB_E_INVALID);
    if (d_chunk_offs && nchunks > max_chunks) return fail(err, SB_E_INVALID, nchunks, max_chunks);
    if (scratch_bytes < decode_ws_bytes(max_chunks)) return fail(err, SB_BUFFER_TOO_SMALL, scratch_bytes, decode_ws_bytes(max_chunks));
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const sbk::DecodePlan p = make_decode_plan(d_in, n, d_out, cap, d_chunk_offs, nchunks, (int)(flags & 1u), d_result, scratch, max_chunks);
    rc = decode_index_phase(*c, p, st, err);
    if (rc) return rc;
    rc = decode_payload_phase(*c, p, st, err);
    if (rc) return rc;
    if (getenv("SNAPB200_DEBUG_FRAME")) {
        sbk::DecodeCtl h;
        cudaStreamSynchronize(st);
        cudaMemcpy(&h, p.ctl, sizeof h, cudaMemcpyDeviceToHost);
        fprintf(stderr, "[frame decode] n=%llu index_n=%u fragment=%u cap_chunks=%u -> nchunks=%u need_serial=%u produced=%llu walk_err=%u(%llu,%llu) go=%u first_bad=%u\n",
                (unsigned long long)n, p.index_n, p.fragment, p.cap_chunks, h.nchunks, h.need_serial, (unsigned long long)h.produced,
                h.walk_err.code, (unsigned long long)h.walk_err.a, (unsigned long long)h.walk_err.b, h.go, h.first_bad);
    }
    ok(err);
    return 0;
}

// Convenience form: pooled scratch, waits for the result (host sb_frame_result).
int sb_frame_decode_device(const uint8_t* d_in, uint64_t n, uint8_t* d_out, uint64_t cap,
                           const uint64_t* d_chunk_offs, uint32_t nchunks, uint32_t flags,
                           sb_frame_result* result, void* stream, sb_error* err) {
    if (!result) return fail(err, SB_E_INVALID);
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_DEC];
    std::lock_guard<std::mutex> lk(l.mu);
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t maxc = d_chunk_offs ? (uint64_t)nchunks + 1 : n / 1024 + 4096;
    rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    for (;;) {
        if (maxc > 0xFFFFFFF0ull) return fail(err, SB_E_INVALID);
        CK(l.ws[1].need(decode_ws_bytes(maxc) + sizeof(sb_frame_result) + 256));
        sb_frame_result* d_res = (sb_frame_result*)((uint8_t*)l.ws[1].p + align_up(decode_ws_bytes(maxc), 256));
        sb_error e2;
        rc = sb_frame_decode_device_ws(d_in, n, d_out, cap, d_chunk_offs, nchunks, flags, d_res, l.ws[1].p, decode_ws_bytes(maxc),
                                       (uint32_t)maxc, st, &e2);
        if (rc) { if (err) *err = e2; return rc; }
        sb_frame_result* res = (sb_frame_result*)l.pinned[4];
        CK(cudaMemcpyAsync(res, d_res, sizeof *res, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (res->status.code == SB_E_INVALID && res->status.b == 1 && maxc < n / 8 + 16) { maxc = maxc * 8; continue; }   // chunk table too small
        *result = *res;
        break;
    }
    ok(err);
    return 0;
}

// read::FrameDecoder + read_to_end over host memory (reference src/read.rs:104-239): the stream is uploaded once
// and decoded by the device path above (header walk, K2, checksum); the first failure IN STREAM ORDER is reported
// and the bytes produced before it are returned, like a reader that fails on its n-th read.
int sb_frame_decode(const uint8_t* in, size_t n, uint8_t* out, size_t cap, size_t* out_n, sb_error* err) {
    if ((!in && n) || !out_n) return fail(err, SB_E_INVALID);
    if (n == 0) { *out_n = 0; ok(err); return 0; }
    Ctx* c;
    int rc = get_ctx(&c, err);
    if (rc) return rc;
    Lane& l = c->lane[LANE_DEC];
    std::lock_guard<std::mutex> lk(l.mu);
    cudaStream_t st = l.s_compute;
    CK(l.in[1].need(n + 64));
    rc = need_pinned(l, 4, 4096, err); if (rc) return rc;
    CK(cudaMemcpyAsync(l.in[1].p, in, n, cudaMemcpyHostToDevice, st));
    uint64_t maxc = n / 1024 + 4096;
    sbk::DecodeCtl* hc = (sbk::DecodeCtl*)l.pinned[4];
    sbk::DecodePlan p;
    for (;;) {
        CK(l.ws[1].need(decode_ws_bytes(maxc) + sizeof(sb_frame_result) + 256));
        sb_frame_result* d_res = (sb_frame_result*)((uint8_t*)l.ws[1].p + align_up(decode_ws_bytes(maxc), 256));
        p = make_decode_plan(l.in[1].as<uint8_t>(), n, nullptr, out ? cap : ~0ull, nullptr, 0, 0, d_res, l.ws[1].p, (uint32_t)maxc);
        rc = decode_index_phase(*c, p, st, err);
        if (rc) return rc;
        CK(cudaMemcpyAsync(hc, p.ctl, sizeof(sbk::DecodeCtl), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (hc->walk_err.code == SB_E_INVALID && hc->walk_err.b == 1 && maxc < n / 8 + 16) { maxc *= 8; continue; }
        break;
    }
    const uint64_t produced = hc->produced;
    // Sizing call: only possible failures that precede any data check are reported by the full call.
    if (!out) { *out_n = (size_t)produced; ok(err); return 0; }
    if (produced > cap) return fail(err, SB_BUFFER_TOO_SMALL, cap, produced);
    CK(l.compact[1].need(produced + 64));
    p.out = l.compact[1].as<uint8_t>();
    rc = decode_payload_phase(*c, p, st, err);
    if (rc) return rc;
    sb_frame_result* res = (sb_frame_result*)((uint8_t*)l.pinned[4] + 512);
    CK(cudaMemcpyAsync(res, p.result, sizeof *res, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (res->bytes) CK(cudaMemcpy(out, l.compact[1].p, res->bytes, cudaMemcpyDeviceToHost));
    *out_n = (size_t)res->bytes;
    if (res->status.code) { if (err) *err = res->status; return (int)res->status.code; }
    ok(err);
    return 0;
}

// ---------------------------------------------------------- libsnappy C API
int snappy_compress(const char* input, size_t input_length, char* compressed, size_t* compressed_length) {
    if (!compressed_length) return 1;
    sb_error e;
    size_t n = 0;
    int rc = sb_compress((const uint8_t*)input, input_length, (uint8_t*)compressed, *compressed_length, &n, &e);
    if (rc == SB_BUFFER_TOO_SMALL) return 2;
    if (rc) return 1;
    *compressed_length = n;
    return 0;
}
int snappy_uncompress(const char* compressed, size_t compressed_length, char* uncompressed, size_t* uncompressed_length) {
    if (!uncompressed_length) return 1;
    sb_error e;
    size_t n = 0;
    int rc = sb_decompress((const uint8_t*)compressed, compressed_length, (uint8_t*)uncompressed, *uncompressed_length, &n, &e);
    if (rc == SB_BUFFER_TOO_SMALL) return 2;
    if (rc) return 1;
    *uncompressed_length = n;
    return 0;
}
size_t snappy_max_compressed_length(size_t source_length) { return 32 + source_length + source_length / 6; }
int snappy_uncompressed_length(const char* compressed, size_t compressed_length, size_t* result) {
    sb_error e;
    if (!result || compressed_length == 0) return 1;
    return sb_decompress_len((const uint8_t*)compressed, compressed_length, result, &e) ? 1 : 0;
}

#ifdef K1_PROFILE
// profile build only (tools/k1_phase_profile.sh): read / reset the parser phase timers
int sb_debug_k1_profile(unsigned long long* out16, int reset) {
    cudaDeviceSynchronize();
    if (out16 && cudaMemcpyFromSymbol(out16, g_k1_prof, sizeof(unsigned long long) * 16) != cudaSuccess) return 1;
    if (reset) { unsigned long long z[16] = {0}; if (cudaMemcpyToSymbol(g_k1_prof, z, sizeof z) != cudaSuccess) return 1; }
    return 0;
}
#endif

}  // extern "C"
