// hoh_api.cu — C-ABI of libhohgpu.so (declared in include/hohgpu.h): context, scratch memory,
// kernel launches for the batched entry points and the compat shims with the reference's value
// semantics.  No CPU implementation of any stage lives here: every entry point launches kernels
// from hoh_kernels.cuh and fails with HOH_E_CUDA when there is no device.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "hoh_kernels.cuh"

using namespace hohk;

namespace {

enum Slot {
    S_FREQS = 0, S_CUM, S_HEADS, S_ENCMETA, S_DECMETA, S_RESID, S_STREAMS, S_DSTREAMS, S_DRESULTS,
    S_IO_A, S_IO_B, S_IO_C, S_IO_D, S_IO_E, S_RESULTS, S_TOP, S_BP, S_HIST, S_COST, S_SUMS, S_MASKS,
    S_WIDE_TOP, S_WIDE_BP, S_MISC, S_L_MAPS, S_L_IDX, S_L_HDR, S_L_U32, S_L_STATUS, S_L_RR, S_L_RES, S_LZ_PX, S_LZ_STATE, S_LZ_SIDE, S_LZ_COUNTS, S_LZ_SLABS, S_LZ_RES, S_LZ_BONUS, S_LZ_KEYS, S_LZ_VALS, S_LZ_FLAG, S_T_NUKE, S_T_LZ, S_T_U32, S_T_P8, S_T_P9, S_T_O8, S_T_O9, S_T_R8, S_T_R9, S_T_MORE_SHAPES, S_T_LAST = S_T_NUKE + 4 * 9 - 1, S_D_TILES, S_D_PLANES, S_D_LZSYM, S_D_IDXSYM, S_D_RESID, S_D_OUT, S_D_BACKREF, S_D_MAPS,
    S_D_STREAMS, S_D_RES_A, S_D_RES_B, S_D_TOP, S_D_BP, S_D_PSTATUS, S_L_NEED, S_L_ORDER, S_R_SLOTS, S_R_STATUS, S_COUNT
};

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
    uint64_t epoch = 0;  // the top-level call (root context's `epoch`) that last asked for this buffer
};

constexpr int kPipeDepth = 4;  // most chunks in flight in a host-buffer call (hoh_*_images*_host)

}  // namespace

struct hoh_ctx {
    int device = 0;
    int sm_count = 148;
    // hoh_layer_encode_batch since the last hoh_debug_layer_stats: {candidates coded, planes the size intervals did not
    // settle, planes} (device counters, summed over the child contexts when read)
    uint32_t* d_layer_stats = nullptr;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    uint64_t launches = 0;
    // image shape / mode (and crop size) the cached scratch of the chunked walks was sized for: hoh_encode_images,
    // hoh_decode_images, hoh_decode_regions
    uint64_t enc_key = 0, dec_key = 0, roi_key = 0;
    char err[512] = {0};
    Buf scratch[S_COUNT];
    cudaEvent_t ev[16][2] = {};
    void* flush = nullptr;
    size_t flush_bytes = 0;
    std::map<uint64_t, double*> e_tabs;  // plane size -> device table of -log2(f/size)
    bool smem_opt_in = false;
    // host-buffer pipeline of the four host calls (hoh_{en,de}code_images[_s0]_host): copy streams, per-slot events,
    // pinned offset staging
    bool pipe_ready = false;
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[kPipeDepth] = {}, ev_comp[kPipeDepth] = {}, ev_d2h[kPipeDepth] = {}, ev_off[kPipeDepth] = {};
    cudaEvent_t ev_start = nullptr;
    uint64_t* h_off[kPipeDepth] = {};
    size_t h_off_cap[kPipeDepth] = {};
    // Child contexts (own stream, own scratch), created on first use by child_of():
    //   child[b]            slot b of the s0 host calls: codes its chunks and holds their staging
    //   child[0], child[1]  the 8-bit / 9-bit layer_encode forks of hoh_encode_images
    //   child[2], child[3]  staging of slots 0 / 1 of the whole-tile host calls
    // new_shape() frees the scratch of ctx, child[0] and child[1], and the whole-tile host calls reach it from inside
    // their pipeline, so whole-tile staging must never sit in one of those three.
    hoh_ctx* child[4] = {};
    // Scratch of EARLIER top-level calls stays cached (the next call of the same kind reuses it) but is given back when an
    // allocation fails: the root context counts top-level calls (`epoch`, bumped by the outermost entry point: `depth`),
    // every buffer remembers the call that last asked for it, and scratch() frees the others before it gives up.
    hoh_ctx* parent = nullptr;
    uint64_t epoch = 1;
    int depth = 0;
    // side streams for launches that are independent of each other and each bound by the serial chain of a
    // stream (the table-size classes of one entropy batch): they overlap instead of queueing
    bool aux_ready = false;
    cudaStream_t aux[8] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[8] = {};
    // per-kernel profiling (hoh_profile_*)
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;       // event 0 = begin, event i = after launch i
    std::vector<const char*> prof_names;        // name of launch i (index i-1)
    std::vector<cudaEvent_t> prof_pool;
    std::vector<std::string> prof_keys;
    std::vector<double> prof_ms;
    std::vector<uint64_t> prof_launches;
};

namespace {

// Every entry point runs on the context's device whatever the caller's current device is, and puts the
// caller's device back on return (a process may hold contexts on several GPUs, or share the thread with torch).
inline hoh_ctx* root_of(hoh_ctx* c) {
    while (c->parent) c = c->parent;
    return c;
}
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    hoh_ctx* root = nullptr;
    explicit DeviceGuard(const hoh_ctx* ctx);
    ~DeviceGuard() {
        if (root) root->depth--;
        if (switched) cudaSetDevice(prev);
    }
};

const uint16_t kStockMasks[14] = {  // layer_encode.hpp:159-175
    0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd, 0xfffb, 0xfff7, 0xffef, 0xffdf, 0xff7f, 0xfdff, 0xffff};

DeviceGuard::DeviceGuard(const hoh_ctx* ctx) {
    if (!ctx) return;
    root = root_of(const_cast<hoh_ctx*>(ctx));
    if (root->depth++ == 0) root->epoch++;  // a new top-level call: what the previous ones left cached is now stale
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    if (prev != ctx->device && cudaSetDevice(ctx->device) == cudaSuccess) switched = true;
}

int fail_cuda(hoh_ctx* c, cudaError_t e, const char* what) {
    if (c) snprintf(c->err, sizeof c->err, "%s: %s", what, cudaGetErrorString(e));
    return HOH_E_CUDA;
}

#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return fail_cuda(ctx, e_, #call);   \
    } while (0)

int prof_mark(hoh_ctx* ctx, const char* name);

#define LAUNCHED(name)                                             \
    do {                                                           \
        ctx->launches++;                                           \
        cudaError_t e_ = cudaGetLastError();                       \
        if (e_ != cudaSuccess) return fail_cuda(ctx, e_, name);    \
        if (ctx->profiling) {                                      \
            int p_ = prof_mark(ctx, name);                         \
            if (p_ != HOH_OK) return p_;                           \
        }                                                          \
    } while (0)

#define TRY(expr)                   \
    do {                            \
        int s_ = (expr);            \
        if (s_ != HOH_OK) return s_; \
    } while (0)

int prof_mark(hoh_ctx* ctx, const char* name) {
    cudaEvent_t ev;
    if (!ctx->prof_pool.empty()) {
        ev = ctx->prof_pool.back();
        ctx->prof_pool.pop_back();
    } else {
        CK(cudaEventCreate(&ev));
    }
    CK(cudaEventRecord(ev, ctx->stream));
    ctx->prof_events.push_back(ev);
    if (name) ctx->prof_names.push_back(name);
    return HOH_OK;
}

// Frees every cached scratch buffer of the context tree that the CURRENT top-level call has not asked for.
void free_stale_scratch(hoh_ctx* c, uint64_t epoch) {
    for (auto& b : c->scratch)
        if (b.p && b.epoch != epoch) {
            cudaFree(b.p);
            b.p = nullptr;
            b.cap = 0;
        }
    for (hoh_ctx* ch : c->child)
        if (ch) free_stale_scratch(ch, epoch);
}

int scratch(hoh_ctx* ctx, Slot slot, size_t bytes, void** out) {
    Buf& b = ctx->scratch[slot];
    hoh_ctx* root = root_of(ctx);
    if (bytes == 0) bytes = 16;
    if (b.cap < bytes) {
        if (b.p) {
            CK(cudaStreamSynchronize(ctx->stream));
            CK(cudaFree(b.p));
            b.p = nullptr;
            b.cap = 0;
        }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&b.p, want);
        if (e == cudaErrorMemoryAllocation) {
            // e.g. a decode of a large batch right after its encode: the encoder's scratch is still cached and
            // scratch_budget() counted it as reusable.  Nothing of an earlier call is in use once the device is idle.
            cudaGetLastError();
            CK(cudaDeviceSynchronize());
            free_stale_scratch(root, root->epoch);
            b.p = nullptr;
            e = cudaMalloc(&b.p, want);
            if (e == cudaErrorMemoryAllocation) {  // without the 12 % of slack
                cudaGetLastError();
                want = bytes;
                e = cudaMalloc(&b.p, want);
            }
        }
        if (e != cudaSuccess) {
            b.p = nullptr;
            return fail_cuda(ctx, e, "cudaMalloc(scratch)");
        }
        b.cap = want;
    }
    b.epoch = root->epoch;
    *out = b.p;
    return HOH_OK;
}

template <typename T>
int scratch_t(hoh_ctx* ctx, Slot slot, size_t count, T** out) {
    void* p = nullptr;
    TRY(scratch(ctx, slot, count * sizeof(T), &p));
    *out = reinterpret_cast<T*>(p);
    return HOH_OK;
}

// Bytes of scratch one chunk of a chunked walk (hoh_encode_images / hoh_decode_images) may plan for.  The entropy
// kernels last as long as one stream's chain however few streams a launch has, so fewer, larger chunks are faster:
// half of the device's memory (90 GB on a B200), but no more than 55 % of what is free now plus what this context
// and its children already hold as scratch (that memory is reused by the walk).  HOH_SCRATCH_GB overrides.
size_t scratch_budget(hoh_ctx* ctx) {
    if (const char* e = getenv("HOH_SCRATCH_GB")) return (size_t)(atof(e) * (double)((size_t)1 << 30));
    size_t held = 0;
    for (int i = 0; i < S_COUNT; i++) held += ctx->scratch[i].cap;
    for (hoh_ctx* ch : ctx->child)
        if (ch)
            for (int i = 0; i < S_COUNT; i++) held += ch->scratch[i].cap;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return (size_t)8 << 30;
    size_t budget = (size_t)((double)(free_b + held) * 0.55);
    if (budget > total_b / 2) budget = total_b / 2;
    if (budget < ((size_t)1 << 30)) budget = (size_t)1 << 30;
    return budget;
}

int new_shape(hoh_ctx* ctx, uint64_t key, uint64_t& slot);

inline unsigned blocks_for(uint64_t items, unsigned per_block) { return (unsigned)((items + per_block - 1) / per_block); }
inline unsigned grid_cap(uint64_t items, unsigned per_block, unsigned cap = 148u * 32u) {
    uint64_t b = (items + per_block - 1) / per_block;
    if (b < 1) b = 1;
    return (unsigned)(b > cap ? cap : b);
}

int ensure_smem_opt_in(hoh_ctx* ctx) {
    if (ctx->smem_opt_in) return HOH_OK;
    const int big = 200 * 1024;
    CK(cudaFuncSetAttribute(k_rans_encode<uint16_t, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_encode<uint16_t, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_encode<uint32_t, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_encode_ws<uint16_t, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_encode_ws<uint16_t, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_encode_ws<uint32_t, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_encode_ws<uint16_t, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_decode<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_decode<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_decode_tiles_s0<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_decode_tiles_s0<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_tile_unpredict_s0<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_tile_unpredict_s0<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_unpredict_fastpath_wave, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_decode_static_direct<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(k_rans_decode_static_direct<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    ctx->smem_opt_in = true;
    return HOH_OK;
}

int aux_init(hoh_ctx* ctx) {
    if (ctx->aux_ready) return HOH_OK;
    for (int k = 0; k < 8; k++) {
        CK(cudaStreamCreateWithFlags(&ctx->aux[k], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->ev_join[k], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    ctx->aux_ready = true;
    return HOH_OK;
}
// everything queued on the context's stream so far happens before what is queued on aux[0..count) from now on
int aux_fork(hoh_ctx* ctx, int count) {
    TRY(aux_init(ctx));
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    for (int k = 0; k < count; k++) CK(cudaStreamWaitEvent(ctx->aux[k], ctx->ev_fork, 0));
    return HOH_OK;
}
int aux_join(hoh_ctx* ctx, int count) {
    for (int k = 0; k < count; k++) {
        CK(cudaEventRecord(ctx->ev_join[k], ctx->aux[k]));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[k], 0));
    }
    return HOH_OK;
}

// The dynamic shared memory to ask for so that an SM holds at most `per_sm` CTAs of a kernel that needs `smem` bytes
// (sm_100: 228 KB per SM, 1 KB of it reserved per resident CTA).  The entropy kernels are bound by instruction-pipe
// throughput, so an SM's time grows with the number of warps it holds, and the block scheduler does not balance CTAs
// across SMs when several launches run side by side: capping the count at the even share keeps the slowest SM short.
size_t smem_for_cap(size_t smem, unsigned per_sm) {
    const size_t sm_total = 228u * 1024u;
    size_t need = sm_total / (per_sm + 1u) - 1024u + 128u;
    need = (need + 127u) & ~(size_t)127u;
    return smem > need ? smem : need;
}

// ... for a launch of `grid` one-warp-chain CTAs on this device: the even share per SM when the launch is a large single
// wave (a small launch is left alone: it may be one of several pipeline chunks in flight that share the SMs).
size_t smem_even_share(const hoh_ctx* ctx, size_t smem, unsigned grid, unsigned min_share = 8u) {
    const unsigned share = (grid + (unsigned)ctx->sm_count - 1u) / (unsigned)ctx->sm_count;
    if (const char* e = getenv("HOH_ENC_CAP")) return atoi(e) > 0 ? smem_for_cap(smem, (unsigned)atoi(e)) : smem;
    return share >= min_share ? smem_for_cap(smem, share) : smem;
}

// First half: normalised tables, stream heads and the size estimates (EncMeta::est) of n streams.
int build_tables(hoh_ctx* ctx, const hoh_enc_stream* d_streams, size_t n, const uint32_t* freqs, uint32_t** cum_out,
                 uint8_t** heads_out, EncMeta** meta_out) {
    TRY(scratch_t(ctx, S_CUM, n * kCumRow, cum_out));
    TRY(scratch_t(ctx, S_HEADS, n * HOH_HEAD_CAP, heads_out));
    TRY(scratch_t(ctx, S_ENCMETA, n, meta_out));
    TRY(ensure_smem_opt_in(ctx));
    k_build_tables<<<blocks_for(n, kTableWarps), kTableWarps * 32, 0, ctx->stream>>>(d_streams, (uint32_t)n, freqs,
                                                                                    *cum_out, *heads_out, *meta_out);
    LAUNCHED("k_build_tables");
    return HOH_OK;
}
// Second half: the coder and the finish.  order / n_active (device, optional): code only the streams listed (padded8 only).
int encode_with_tables(hoh_ctx* ctx, const hoh_enc_stream* d_streams, size_t n, const uint16_t* d_symbols, uint8_t* d_out,
                       hoh_stream_result* d_results, uint32_t* cum, uint8_t* heads, EncMeta* meta, uint32_t max_range,
                       uint32_t max_prob_bits, uint32_t min_prob_bits, bool padded8, const uint32_t* order = nullptr,
                       const uint32_t* n_active = nullptr) {
    if (order && !padded8) return HOH_E_ARG;
    // one launch per (table width, window-size class); every warp takes part in exactly one of them.  The
    // launches are independent and each lasts as long as its longest stream, so they go to side streams and
    // overlap (not while profiling: the per-kernel event times would no longer add up).
    const uint32_t classes[5] = {0, 64, 128, 256, HOH_MAX_RANGE + 1};
    const bool overlap = !ctx->profiling;
    if (overlap) TRY(aux_fork(ctx, 8));
    for (int c = 0; c < 4; c++) {
        if (classes[c] >= max_range + 1) break;
        const uint32_t rows = classes[c + 1];
        const size_t stage = 2 * 32 * kBulkStride * sizeof(uint16_t);
        const size_t smem16 = (size_t)rows * 32 * sizeof(uint16_t) + stage, smem32 = (size_t)rows * 32 * sizeof(uint32_t) + stage;
        cudaStream_t s16 = overlap ? ctx->aux[2 * c] : ctx->stream, s32 = overlap ? ctx->aux[2 * c + 1] : ctx->stream;
        // warps whose streams all have prob_bits >= 14 take the short division chain; the others (only when the caller
        // cannot rule them out) the LOW_BITS instantiation: every warp runs in exactly one of the two
        static const char* const names16[4] = {"k_rans_encode<u16>[rows<=64]", "k_rans_encode<u16>[rows<=128]",
                                               "k_rans_encode<u16>[rows<=256]", "k_rans_encode<u16>[rows<=513]"};
        static const char* const names16l[4] = {"k_rans_encode<u16,low>[rows<=64]", "k_rans_encode<u16,low>[rows<=128]",
                                                "k_rans_encode<u16,low>[rows<=256]", "k_rans_encode<u16,low>[rows<=513]"};
        static const char* const names32[4] = {"k_rans_encode<u32>[rows<=64]", "k_rans_encode<u32>[rows<=128]",
                                               "k_rans_encode<u32>[rows<=256]", "k_rans_encode<u32>[rows<=513]"};
        const size_t hand = 2 * kWsGroup * 32 * sizeof(uint4);
        size_t ws16 = (size_t)rows * 32 * sizeof(uint16_t) + hand, ws32 = (size_t)rows * 32 * sizeof(uint32_t) + hand;
        // BASELINE config 2: 1 536 CTAs = 10.4 per SM; left to itself the block scheduler puts up to 14 on some SMs while
        // the other classes' launches come and go (encode 14.5 ms), capped at 11 everywhere 12.9 ms
        ws16 = smem_even_share(ctx, ws16, blocks_for(n, 32));
        ws32 = smem_even_share(ctx, ws32, blocks_for(n, 32));
        if (padded8) {
            k_rans_encode_ws<uint16_t, 0><<<blocks_for(n, 32), 64, ws16, s16>>>(
                d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 1u, order, n_active);
        } else {
            k_rans_encode<uint16_t, false><<<blocks_for(n, 32), 32, smem16, s16>>>(
                d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 1u);
        }
        LAUNCHED(names16[c]);
        if (min_prob_bits < 14) {
            if (padded8) {  // prob_bits 12-13, and below 12: two more instantiations
                k_rans_encode_ws<uint16_t, 2><<<blocks_for(n, 32), 64, ws16, s16>>>(
                    d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 1u, order, n_active);
                LAUNCHED(names16l[c]);
                k_rans_encode_ws<uint16_t, 1><<<blocks_for(n, 32), 64, ws16, s16>>>(
                    d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 1u, order, n_active);
            } else {
                k_rans_encode<uint16_t, true><<<blocks_for(n, 32), 32, smem16, s16>>>(
                    d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 1u);
            }
            LAUNCHED(names16l[c]);
        }
        if (max_prob_bits > 15) {  // 32-bit table lanes; prob_bits >= 16 there, so never LOW_BITS
            if (padded8) {
                k_rans_encode_ws<uint32_t, 0><<<blocks_for(n, 32), 64, ws32, s32>>>(
                    d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 0u, order, n_active);
            } else {
                k_rans_encode<uint32_t, false><<<blocks_for(n, 32), 32, smem32, s32>>>(
                    d_streams, (uint32_t)n, d_symbols, cum, d_out, meta, classes[c], rows, 0u);
            }
            LAUNCHED(names32[c]);
        }
    }
    if (overlap) TRY(aux_join(ctx, 8));
    k_finish_streams<<<blocks_for(n, 4), 128, 0, ctx->stream>>>(d_streams, (uint32_t)n, d_symbols, heads, meta, d_out,
                                                                d_results, order, n_active);
    LAUNCHED("k_finish_streams");
    return HOH_OK;
}

// Shared tail of the encode pipeline once the raw histograms are in `freqs`.
// min_prob_bits: a lower bound the CALLER guarantees for every stream's prob_bits (0 = unknown).
// padded8: the CALLER guarantees that every stream's symbols start 16-byte aligned and are readable up to the next
// multiple of 8 symbols (planes at a stride rounded up to 8): the warp-specialised encoder then reads them directly.
int encode_from_freqs(hoh_ctx* ctx, const hoh_enc_stream* d_streams, size_t n, const uint16_t* d_symbols,
                      uint8_t* d_out, hoh_stream_result* d_results, const uint32_t* freqs,
                      uint32_t max_range, uint32_t max_prob_bits, uint32_t min_prob_bits, bool padded8 = false) {
    uint32_t* cum;
    uint8_t* heads;
    EncMeta* meta;
    TRY(build_tables(ctx, d_streams, n, freqs, &cum, &heads, &meta));
    return encode_with_tables(ctx, d_streams, n, d_symbols, d_out, d_results, cum, heads, meta, max_range, max_prob_bits,
                              min_prob_bits, padded8);
}

int decode_common(hoh_ctx* ctx, const hoh_dec_stream* d_streams, size_t n, const uint8_t* d_in, size_t in_bytes,
                  uint16_t* d_symbols, hoh_dec_result* d_results) {
    uint32_t* cum;
    DecMeta* meta;
    TRY(scratch_t(ctx, S_CUM, n * kCumRow, &cum));
    TRY(scratch_t(ctx, S_DECMETA, n, &meta));
    TRY(ensure_smem_opt_in(ctx));
    k_parse_streams<<<blocks_for(n, kTableWarps), kTableWarps * 32, 0, ctx->stream>>>(d_streams, (uint32_t)n, d_in,
                                                                                     in_bytes, cum, meta, d_results);
    LAUNCHED("k_parse_streams");
    k_unpack_stored<<<(unsigned)n, 256, 0, ctx->stream>>>(d_streams, d_in, in_bytes, meta, d_symbols);
    LAUNCHED("k_unpack_stored");
    // one launch per table-size class; every warp takes part in exactly one of them
    const uint32_t classes[5] = {0, 64, 128, 256, HOH_MAX_RANGE + 3};
    const bool overlap = !ctx->profiling;  // as in encode_from_freqs
    if (overlap) TRY(aux_fork(ctx, 4));
    for (int c = 0; c < 4; c++) {
        const uint32_t rows = classes[c + 1];
        const size_t fixed = (size_t)rows * 32 * sizeof(uint32_t) + 32 * kRingWords * sizeof(uint32_t) +
                             32 * kDecStride * sizeof(uint16_t);
        cudaStream_t sc = overlap ? ctx->aux[c] : ctx->stream;
        // (the even share of CTAs per SM, as for the fused decoder and the encoder: an SM that the block scheduler
        // loads with twice its share makes the whole launch last twice as long)
        const unsigned dec_share = getenv("HOH_DEC_CAP") ? (unsigned)atoi(getenv("HOH_DEC_CAP")) : 4u;
        const size_t lut_bytes = (size_t)kLutSize * 32 * (rows <= 256 ? 1 : 2);
        const size_t smem = dec_share ? smem_even_share(ctx, fixed + lut_bytes, blocks_for(n, 32), dec_share) : fixed + lut_bytes;
        if (rows <= 256) {
            k_rans_decode<uint8_t><<<blocks_for(n, 32), 32, smem, sc>>>(
                d_streams, (uint32_t)n, d_in, in_bytes, cum, meta, d_symbols, d_results, classes[c], rows);
        } else {
            k_rans_decode<uint16_t><<<blocks_for(n, 32), 32, smem, sc>>>(
                d_streams, (uint32_t)n, d_in, in_bytes, cum, meta, d_symbols, d_results, classes[c], rows);
        }
        static const char* const names[4] = {"k_rans_decode[rows<=64]", "k_rans_decode[rows<=128]",
                                             "k_rans_decode[rows<=256]", "k_rans_decode[rows<=515]"};
        LAUNCHED(names[c]);
    }
    if (overlap) TRY(aux_join(ctx, 4));
    return HOH_OK;
}

TileGeom to_geom(const hoh_tile_geometry& g) {
    TileGeom t;
    t.width = g.width;
    t.height = g.height;
    t.x_tiles = g.x_tiles;
    t.y_tiles = g.y_tiles;
    t.tile_w = g.tile_w;
    t.tile_h = g.tile_h;
    t.tiles_per_image = g.tiles_per_image;
    t.plane_stride = (g.tile_w * g.tile_h + 7u) & ~7u;
    return t;
}

// -log2(f / size) for f = 0..size+1 computed with the host libm (the reference's std::log2,
// layer_encode.hpp:143) so that the doubles the search compares are the reference's doubles.  This is
// a constant table that depends only on the plane size, not on any image data.
int cost_table_for(hoh_ctx* ctx, uint64_t size, double** out, uint32_t* len) {
    *len = (uint32_t)(size + 2);
    auto it = ctx->e_tabs.find(size);
    if (it != ctx->e_tabs.end()) {
        *out = it->second;
        return HOH_OK;
    }
    std::vector<double> tab(size + 2);
    for (uint64_t f = 0; f < size + 2; f++) tab[f] = -std::log2((double)f / (double)size);
    double* d = nullptr;
    CK(cudaMalloc(&d, tab.size() * sizeof(double)));
    CK(cudaMemcpyAsync(d, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->e_tabs[size] = d;
    *out = d;
    return HOH_OK;
}

}  // namespace

namespace {
// full != 0: every stream must hold one symbol per pixel of its tile (no LZ map given): a dense stream coded with
// a NUKE map would otherwise decode into a tile of wrong pixels without anyone noticing
__global__ void k_merge_status(const hoh_dec_result* __restrict__ res, uint64_t n, TileGeom g, uint32_t full,
                               int32_t* __restrict__ status) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n || status[i] != HOH_S_OK) return;
    int32_t st = res[i].status;
    if (st == HOH_S_OK && full) {
        uint32_t x0, y0, tw, th;
        tile_rect(g, (uint32_t)((i / 3u) % g.tiles_per_image), x0, y0, tw, th);
        if (res[i].n != tw * th) st = HOH_S_BAD_LAYER;
    }
    status[i] = st;
}
__global__ void k_normalize_only(uint32_t* __restrict__ freqs, uint32_t* __restrict__ cum, uint32_t range,
                                 uint32_t target, int32_t* __restrict__ status) {
    __shared__ uint32_t s_f[kFreqRow], s_sc[kFreqRow], s_cum[kFreqRow + 8];
    const uint32_t lane = threadIdx.x;
    for (uint32_t i = lane; i < range; i += 32) s_f[i] = freqs[i];
    __syncwarp();
    int st = warp_normalize(s_f, s_sc, s_cum, range, target);
    if (st == HOH_S_OK) {
        for (uint32_t i = lane; i < range; i += 32) freqs[i] = s_f[i];
        for (uint32_t i = lane; i <= range; i += 32) cum[i] = s_cum[i];
    }
    if (lane == 0) *status = st;
}
}  // namespace

namespace {
// channelpredict_all (prediction.hpp:153) for many planes, every pixel in parallel (encode side)
int predict_all_parallel(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth, int x_tiles,
                         int y_tiles, const uint16_t* d_tile_maps, uint16_t* d_resid, uint64_t resid_stride) {
    // one kernel, 32 x 16 pixel tiles
    const uint64_t tpr = ((uint64_t)w + kPaTx - 1) / kPaTx, tpp = tpr * (((uint64_t)h + kPaTy - 1) / kPaTy);
    if (n_planes * tpp > 0x7fffffffull) return HOH_E_UNSUPPORTED;
    k_predict_all_fused<<<(unsigned)(n_planes * tpp), 256, 0, ctx->stream>>>(
        d_planes, n_planes, w, h, depth, x_tiles, y_tiles, d_tile_maps, d_resid, resid_stride, fastdiv_make((uint32_t)tpp),
        fastdiv_make((uint32_t)tpr), fastdiv_make((uint32_t)((w + x_tiles - 1) / x_tiles)),
        fastdiv_make((uint32_t)((h + y_tiles - 1) / y_tiles)));
    LAUNCHED("k_predict_all_fused");
    return HOH_OK;
}

template <typename T>
int stage_in(hoh_ctx* ctx, Slot slot, const T* host, size_t count, T** dev) {
    TRY(scratch_t(ctx, slot, count ? count : 1, dev));
    if (count) CK(cudaMemcpyAsync(*dev, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return HOH_OK;
}
template <typename T>
int stage_out(hoh_ctx* ctx, T* host, const T* dev, size_t count) {
    if (count) CK(cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return HOH_OK;
}
}  // namespace

namespace {
// The chunked walks size their scratch from what the device has free plus what the context already holds, which
// is only true while the held buffers have the proportions the walk wants: when the image shape or mode changes
// between calls, the cached scratch of the previous shape is released first.
int new_shape(hoh_ctx* ctx, uint64_t key, uint64_t& slot) {
    if (slot == key) return HOH_OK;
    if (slot != 0) {
        // this context's own codec scratch and the two children the encoder forks into; NOT children 2 and 3,
        // which hold the staging buffers of a host-buffer call that may be the caller of this very function
        CK(cudaStreamSynchronize(ctx->stream));
        hoh_ctx* who[3] = {ctx, ctx->child[0], ctx->child[1]};
        for (hoh_ctx* c : who) {
            if (!c) continue;
            CK(cudaStreamSynchronize(c->stream));
            for (auto& b : c->scratch) {
                if (b.p) CK(cudaFree(b.p));
                b.p = nullptr;
                b.cap = 0;
            }
        }
    }
    slot = key;
    return HOH_OK;
}

// Child context k of ctx (roles: hoh_ctx::child), created on first use.
int child_of(hoh_ctx* ctx, int k, hoh_ctx** out) {
    if (!ctx->child[k]) {
        if (hoh_ctx_create(ctx->device, nullptr, &ctx->child[k]) != HOH_OK) return HOH_E_CUDA;
        ctx->child[k]->parent = ctx;
    }
    *out = ctx->child[k];
    return HOH_OK;
}
}  // namespace

// =================================================================================================
// context
// =================================================================================================
extern "C" {

int hoh_ctx_create(int device, void* cuda_stream, hoh_ctx** out) {
    if (!out) return HOH_E_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) return HOH_E_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return HOH_E_CUDA;
    hoh_ctx* ctx = new hoh_ctx();
    ctx->device = device;
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->sm_count <= 0)
        ctx->sm_count = 148;
    if (cuda_stream) {
        ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return HOH_E_CUDA;
        }
        ctx->own_stream = true;
    }
    *out = ctx;
    return HOH_OK;
}

void hoh_ctx_destroy(hoh_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& b : ctx->scratch)
        if (b.p) cudaFree(b.p);
    for (auto& kv : ctx->e_tabs) cudaFree(kv.second);
    if (ctx->flush) cudaFree(ctx->flush);
    if (ctx->d_layer_stats) cudaFree(ctx->d_layer_stats);
    for (auto& pair : ctx->ev)
        for (auto& ev : pair)
            if (ev) cudaEventDestroy(ev);
    for (auto ev : ctx->prof_events) cudaEventDestroy(ev);
    for (auto ev : ctx->prof_pool) cudaEventDestroy(ev);
    for (hoh_ctx* ch : ctx->child)
        if (ch) hoh_ctx_destroy(ch);
    if (ctx->s_h2d) cudaStreamDestroy(ctx->s_h2d);
    if (ctx->s_d2h) cudaStreamDestroy(ctx->s_d2h);
    for (int k = 0; k < kPipeDepth; k++) {
        if (ctx->ev_h2d[k]) cudaEventDestroy(ctx->ev_h2d[k]);
        if (ctx->ev_comp[k]) cudaEventDestroy(ctx->ev_comp[k]);
        if (ctx->ev_d2h[k]) cudaEventDestroy(ctx->ev_d2h[k]);
        if (ctx->ev_off[k]) cudaEventDestroy(ctx->ev_off[k]);
        if (ctx->h_off[k]) cudaFreeHost(ctx->h_off[k]);
    }
    if (ctx->ev_start) cudaEventDestroy(ctx->ev_start);
    for (int k = 0; k < 8; k++) {
        if (ctx->aux[k]) cudaStreamDestroy(ctx->aux[k]);
        if (ctx->ev_join[k]) cudaEventDestroy(ctx->ev_join[k]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int hoh_release_scratch(hoh_ctx* ctx) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    for (auto& b : ctx->scratch) {
        if (b.p) CK(cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    for (hoh_ctx* ch : ctx->child)
        if (ch) TRY(hoh_release_scratch(ch));
    return HOH_OK;
}

int hoh_sync(hoh_ctx* ctx) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    return HOH_OK;
}

const char* hoh_strerror(int status) {
    switch (status) {
        case HOH_OK: return "ok";
        case HOH_E_CUDA: return "CUDA runtime error (no device, or a call failed)";
        case HOH_E_ARG: return "bad argument";
        case HOH_E_UNSUPPORTED: return "outside the supported domain of the hot path";
        case HOH_E_CAPACITY: return "output buffer too small";
        case HOH_E_STREAM: return "a stream failed (see per-stream status)";
        default: return "unknown status";
    }
}

const char* hoh_last_cuda_error(hoh_ctx* ctx) { return ctx ? ctx->err : "no context"; }
uint64_t hoh_launch_count(hoh_ctx* ctx) { return ctx ? ctx->launches : 0; }

int hoh_debug_layer_stats(hoh_ctx* ctx, uint64_t out[3]) {
    if (!ctx || !out) return HOH_E_ARG;
    DeviceGuard guard_(ctx);
    out[0] = out[1] = out[2] = 0;
    hoh_ctx* all[5] = {ctx, ctx->child[0], ctx->child[1], ctx->child[2], ctx->child[3]};
    for (hoh_ctx* c : all) {
        if (!c || !c->d_layer_stats) continue;
        uint32_t v[4];
        CK(cudaStreamSynchronize(c->stream));
        CK(cudaMemcpy(v, c->d_layer_stats, sizeof v, cudaMemcpyDeviceToHost));
        CK(cudaMemset(c->d_layer_stats, 0, sizeof v));
        for (int k = 0; k < 3; k++) out[k] += v[k];
    }
    return HOH_OK;
}

int hoh_dev_alloc(hoh_ctx* ctx, size_t bytes, void** dptr) {
    DeviceGuard guard_(ctx);
    if (!ctx || !dptr) return HOH_E_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMalloc(dptr, bytes ? bytes : 16));
    return HOH_OK;
}
int hoh_dev_free(hoh_ctx* ctx, void* dptr) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaFree(dptr));
    return HOH_OK;
}
int hoh_dev_memset(hoh_ctx* ctx, void* dptr, int value, size_t bytes) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaMemsetAsync(dptr, value, bytes, ctx->stream));
    return HOH_OK;
}
int hoh_host_alloc(hoh_ctx* ctx, size_t bytes, void** hptr) {
    DeviceGuard guard_(ctx);
    if (!ctx || !hptr) return HOH_E_ARG;
    CK(cudaHostAlloc(hptr, bytes ? bytes : 16, cudaHostAllocDefault));
    return HOH_OK;
}
int hoh_host_free(hoh_ctx* ctx, void* hptr) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaFreeHost(hptr));
    return HOH_OK;
}
int hoh_h2d(hoh_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return HOH_OK;
}
int hoh_d2h(hoh_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    CK(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return HOH_OK;
}
int hoh_timer_start(hoh_ctx* ctx, int slot) {
    DeviceGuard guard_(ctx);
    if (!ctx || slot < 0 || slot >= 16) return HOH_E_ARG;
    for (int k = 0; k < 2; k++)
        if (!ctx->ev[slot][k]) CK(cudaEventCreate(&ctx->ev[slot][k]));
    CK(cudaEventRecord(ctx->ev[slot][0], ctx->stream));
    return HOH_OK;
}
int hoh_timer_stop(hoh_ctx* ctx, int slot) {
    DeviceGuard guard_(ctx);
    if (!ctx || slot < 0 || slot >= 16 || !ctx->ev[slot][1]) return HOH_E_ARG;
    CK(cudaEventRecord(ctx->ev[slot][1], ctx->stream));
    return HOH_OK;
}
int hoh_timer_elapsed_ms(hoh_ctx* ctx, int slot, float* ms) {
    DeviceGuard guard_(ctx);
    if (!ctx || slot < 0 || slot >= 16 || !ms || !ctx->ev[slot][1]) return HOH_E_ARG;
    CK(cudaEventSynchronize(ctx->ev[slot][1]));
    CK(cudaEventElapsedTime(ms, ctx->ev[slot][0], ctx->ev[slot][1]));
    return HOH_OK;
}
int hoh_profile_begin(hoh_ctx* ctx) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    for (auto ev : ctx->prof_events) ctx->prof_pool.push_back(ev);
    ctx->prof_events.clear();
    ctx->prof_names.clear();
    ctx->prof_keys.clear();
    ctx->prof_ms.clear();
    ctx->prof_launches.clear();
    TRY(prof_mark(ctx, nullptr));
    ctx->profiling = true;
    return HOH_OK;
}
int hoh_profile_end(hoh_ctx* ctx) {
    DeviceGuard guard_(ctx);
    if (!ctx || !ctx->profiling) return HOH_E_ARG;
    ctx->profiling = false;
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i + 1 < ctx->prof_events.size(); i++) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->prof_events[i], ctx->prof_events[i + 1]));
        const std::string key = ctx->prof_names[i];
        size_t k = 0;
        while (k < ctx->prof_keys.size() && ctx->prof_keys[k] != key) k++;
        if (k == ctx->prof_keys.size()) {
            ctx->prof_keys.push_back(key);
            ctx->prof_ms.push_back(0.0);
            ctx->prof_launches.push_back(0);
        }
        ctx->prof_ms[k] += ms;
        ctx->prof_launches[k]++;
    }
    return HOH_OK;
}
int hoh_profile_count(hoh_ctx* ctx) { return ctx ? (int)ctx->prof_keys.size() : 0; }
int hoh_profile_entry(hoh_ctx* ctx, int index, const char** name, double* total_ms, uint64_t* launches) {
    DeviceGuard guard_(ctx);
    if (!ctx || index < 0 || index >= (int)ctx->prof_keys.size()) return HOH_E_ARG;
    if (name) *name = ctx->prof_keys[index].c_str();
    if (total_ms) *total_ms = ctx->prof_ms[index];
    if (launches) *launches = ctx->prof_launches[index];
    return HOH_OK;
}
int hoh_flush_l2(hoh_ctx* ctx) {
    DeviceGuard guard_(ctx);
    if (!ctx) return HOH_E_ARG;
    if (!ctx->flush) {
        ctx->flush_bytes = 256ull << 20;  // > 126 MB L2
        CK(cudaMalloc(&ctx->flush, ctx->flush_bytes));
    }
    CK(cudaMemsetAsync(ctx->flush, 0x5a, ctx->flush_bytes, ctx->stream));
    return HOH_OK;
}

// =================================================================================================
// batched entropy coding
// =================================================================================================
size_t hoh_enc_slab_bytes(size_t n, uint32_t prob_bits) {
    // every symbol emits at most one 32-bit word and at most prob_bits bits on average, plus the
    // two flush words, the header room in front and slack
    size_t payload = ((n * (size_t)prob_bits + 31) / 32) * 4 + 64;
    size_t total = payload + HOH_HEAD_CAP + 64;
    size_t stored = n * 2 + 64;  // stored-mode rewrite: at most 9 bits per symbol
    if (stored > total) total = stored;
    return (total + 15) & ~(size_t)15;
}

int hoh_encode_entropy_batch(hoh_ctx* ctx, const hoh_enc_stream* d_streams, size_t n_streams,
                             const uint16_t* d_symbols, uint8_t* d_out, hoh_stream_result* d_results,
                             uint32_t max_range, uint32_t max_prob_bits, uint32_t max_n) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_streams || !d_out || !d_results) return HOH_E_ARG;
    if (n_streams == 0) return HOH_OK;
    if (max_range == 0 || max_range > HOH_MAX_RANGE || max_prob_bits == 0 || max_prob_bits > HOH_MAX_PROB_BITS)
        return HOH_E_UNSUPPORTED;
    (void)max_n;
    uint32_t* freqs;
    TRY(scratch_t(ctx, S_FREQS, n_streams * kFreqRow, &freqs));
    k_histogram<<<(unsigned)n_streams, 256, 0, ctx->stream>>>(d_streams, d_symbols, freqs);
    LAUNCHED("k_histogram");
    return encode_from_freqs(ctx, d_streams, n_streams, d_symbols, d_out, d_results, freqs, max_range, max_prob_bits, 0);
}

int hoh_decode_entropy_batch(hoh_ctx* ctx, const hoh_dec_stream* d_streams, size_t n_streams,
                             const uint8_t* d_in, size_t in_bytes, uint16_t* d_symbols,
                             hoh_dec_result* d_results, uint32_t max_n) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_streams || !d_in || !d_symbols || !d_results) return HOH_E_ARG;
    if (n_streams == 0) return HOH_OK;
    if (in_bytes < 32) return HOH_E_ARG;  // hohgpu.h, input contract: 32 zero bytes of padding are part of in_bytes
    (void)max_n;
    return decode_common(ctx, d_streams, n_streams, d_in, in_bytes, d_symbols, d_results);
}

int hoh_rans_encode_static(hoh_ctx* ctx, const uint16_t* d_symbols, size_t n, uint32_t stream_len,
                           const uint32_t* d_cum, uint32_t range, uint32_t prob_bits, uint8_t* d_out,
                           uint32_t slab_bytes, uint32_t* d_payload_bytes) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_symbols || !d_cum || !d_out || !d_payload_bytes) return HOH_E_ARG;
    if (range == 0 || range > HOH_MAX_RANGE || prob_bits == 0 || prob_bits > HOH_MAX_PROB_BITS) return HOH_E_UNSUPPORTED;
    if (stream_len == 0 || stream_len % 8 || slab_bytes % 16) return HOH_E_ARG;
    if (n == 0) return HOH_OK;
    const uint64_t streams = (n + stream_len - 1) / stream_len;
    const unsigned sgrid = blocks_for(streams, kStaticWarps * 32);
    if (prob_bits >= 14) {
        k_rans_encode_static<0><<<sgrid, kStaticWarps * 32, 0, ctx->stream>>>(d_symbols, n, stream_len, d_cum, range, prob_bits, d_out,
                                                                          slab_bytes, d_payload_bytes);
    } else {
        k_rans_encode_static<1><<<sgrid, kStaticWarps * 32, 0, ctx->stream>>>(d_symbols, n, stream_len, d_cum, range, prob_bits, d_out,
                                                                          slab_bytes, d_payload_bytes);
    }
    LAUNCHED("k_rans_encode_static");
    return HOH_OK;
}

int hoh_rans_decode_static(hoh_ctx* ctx, const uint8_t* d_in, uint32_t slab_bytes,
                           const uint32_t* d_payload_bytes, size_t n, uint32_t stream_len,
                           const uint32_t* d_cum, uint32_t range, uint32_t prob_bits, uint16_t* d_symbols) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_symbols || !d_cum || !d_in || !d_payload_bytes) return HOH_E_ARG;
    if (range == 0 || range > HOH_MAX_RANGE || prob_bits == 0 || prob_bits > HOH_MAX_PROB_BITS) return HOH_E_UNSUPPORTED;
    if (stream_len == 0 || stream_len % 8 || slab_bytes % 16) return HOH_E_ARG;
    if (n == 0) return HOH_OK;
    const uint64_t streams = (n + stream_len - 1) / stream_len;
    if (prob_bits <= 15) {  // the slot -> symbol table fits shared memory: direct lookups
        const size_t sym_bytes = range <= 256 ? 1 : 2;
        const size_t smem = (size_t)kStaticDirectWarps * 32 * kRingWords * 4 + (size_t)kStaticDirectWarps * 32 * kDecStride * 2 +
                            (size_t)HOH_MAX_RANGE * 4 + ((size_t)sym_bytes << prob_bits);
        TRY(ensure_smem_opt_in(ctx));
        const unsigned blocks = blocks_for(streams, kStaticDirectWarps * 32);
        if (range <= 256)
            k_rans_decode_static_direct<uint8_t><<<blocks, kStaticDirectWarps * 32, smem, ctx->stream>>>(
                d_in, slab_bytes, d_payload_bytes, n, stream_len, d_cum, range, prob_bits, d_symbols);
        else
            k_rans_decode_static_direct<uint16_t><<<blocks, kStaticDirectWarps * 32, smem, ctx->stream>>>(
                d_in, slab_bytes, d_payload_bytes, n, stream_len, d_cum, range, prob_bits, d_symbols);
        LAUNCHED("k_rans_decode_static_direct");
        return HOH_OK;
    }
    k_rans_decode_static<<<blocks_for(streams, kStaticDecWarps * 32), kStaticDecWarps * 32, 0, ctx->stream>>>(
        d_in, slab_bytes, d_payload_bytes, n, stream_len, d_cum, range, prob_bits, d_symbols);
    LAUNCHED("k_rans_decode_static");
    return HOH_OK;
}

// =================================================================================================
// batched tile codec, mode 0
// =================================================================================================
int hoh_tile_geometry_for(uint32_t width, uint32_t height, hoh_tile_geometry* out) {
    if (!out || width == 0 || height == 0) return HOH_E_ARG;
    hoh_tile_geometry g;
    g.width = width;
    g.height = height;
    if ((width >= 512 || height >= 512) && width >= 256 && height >= 256) {  // choh.cpp:454
        g.x_tiles = width / 256;
        g.y_tiles = height / 256;
    } else {
        g.x_tiles = g.y_tiles = 1;
    }
    g.tile_w = (width + g.x_tiles - 1) / g.x_tiles;   // choh.cpp:459
    g.tile_h = (height + g.y_tiles - 1) / g.y_tiles;  // choh.cpp:460
    g.tiles_per_image = g.x_tiles * g.y_tiles;
    g.streams_per_image = 3 * g.tiles_per_image;
    *out = g;
    return HOH_OK;
}

size_t hoh_encode_images_out_bytes(const hoh_tile_geometry* g, size_t n_images) {
    if (!g) return 0;
    return hoh_enc_slab_bytes((size_t)g->tile_w * g->tile_h, 15) * g->streams_per_image * n_images;
}

int hoh_encode_images_s0(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_images, uint32_t width, uint32_t height,
                         const uint8_t* d_nuke, uint8_t* d_out, size_t out_bytes, hoh_stream_result* d_results,
                         uint8_t* d_packed, size_t packed_cap, uint64_t* d_packed_off) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_rgb || !d_out || !d_results) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    if ((uint64_t)hg.tile_w * hg.tile_h >= (1u << 21)) return HOH_E_UNSUPPORTED;  // varint.hpp:39-45
    const TileGeom g = to_geom(hg);
    const uint64_t n_tiles = (uint64_t)n_images * g.tiles_per_image, n_streams = n_tiles * 3;
    const uint32_t slab = (uint32_t)hoh_enc_slab_bytes((size_t)g.tile_w * g.tile_h, 15);
    if (out_bytes < n_streams * slab) return HOH_E_CAPACITY;
    uint16_t* resid;
    uint32_t* freqs;
    hoh_enc_stream* streams;
    TRY(scratch_t(ctx, S_RESID, n_streams * g.plane_stride, &resid));
    TRY(scratch_t(ctx, S_FREQS, n_streams * kFreqRow, &freqs));
    TRY(scratch_t(ctx, S_STREAMS, n_streams, &streams));
    if (g.width % 4 == 0 && g.tile_w % 4 == 0 && g.tile_w <= 1024) {
        k_tile_residuals_s0<<<(unsigned)n_tiles, 256, 0, ctx->stream>>>(d_rgb, g, resid, freqs);
    } else {
        k_tile_residuals_s0_generic<<<(unsigned)n_tiles, 256, 0, ctx->stream>>>(d_rgb, g, resid, freqs);
    }
    LAUNCHED("k_tile_residuals_s0");
    k_make_tile_streams<<<blocks_for(n_streams, 256), 256, 0, ctx->stream>>>(g, n_tiles, slab, streams);
    LAUNCHED("k_make_tile_streams");
    if (d_nuke) {  // layer_encode.hpp:93-99: only the residuals of pixels no LZ match covers are coded
        k_compact_nuke<<<blocks_for(n_streams * 32, 128), 128, 0, ctx->stream>>>(g, n_tiles, d_nuke, g.plane_stride, resid,
                                                                                streams);
        LAUNCHED("k_compact_nuke");
        k_histogram<<<(unsigned)n_streams, 256, 0, ctx->stream>>>(streams, resid, freqs);
        LAUNCHED("k_histogram");
    }
    TRY(encode_from_freqs(ctx, streams, n_streams, resid, d_out, d_results, freqs, 512, 15, 15, true));
    if (d_packed) {
        if (!d_packed_off) return HOH_E_ARG;
        k_scan_sizes<<<1, 1024, 0, ctx->stream>>>(d_results, (uint32_t)n_streams, d_packed_off);
        LAUNCHED("k_scan_sizes");
        k_gather_streams<<<(unsigned)n_streams, 256, 0, ctx->stream>>>(d_results, d_out, d_packed_off, d_packed,
                                                                       packed_cap);
        LAUNCHED("k_gather_streams");
    }
    return HOH_OK;
}


int hoh_decode_images_s0(hoh_ctx* ctx, const uint8_t* d_packed, size_t packed_bytes, const uint64_t* d_packed_off,
                         size_t n_images, uint32_t width, uint32_t height, const uint16_t* d_backref,
                         uint8_t* d_rgb, int32_t* d_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_packed || !d_packed_off || !d_rgb || !d_status) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    if (packed_bytes < 32) return HOH_E_ARG;  // input contract (hohgpu.h)
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const TileGeom g = to_geom(hg);
    const uint64_t n_tiles = (uint64_t)n_images * g.tiles_per_image, n_streams = n_tiles * 3;
    uint16_t* resid;
    hoh_dec_stream* streams;
    hoh_dec_result* results;
    TRY(scratch_t(ctx, S_DSTREAMS, n_streams, &streams));
    TRY(scratch_t(ctx, S_DRESULTS, n_streams, &results));
    // Fused path: entropy decode, un-prediction, colour inverse and scatter in one kernel (k_rans_decode_tiles_s0);
    // needs equal tiles whose rows are whole groups of 8 pixels and 8-byte aligned image rows.
    const bool fused = !d_backref && g.tile_w * g.x_tiles == g.width && g.tile_h * g.y_tiles == g.height && g.tile_w % 8 == 0 &&
                       g.tile_w >= 16 && g.width % 8 == 0 && (reinterpret_cast<uintptr_t>(d_rgb) & 7u) == 0 &&
                       !getenv("HOH_NO_FUSED_DECODE");
    if (fused) {
        uint32_t* cum;
        DecMeta* meta;
        TRY(scratch_t(ctx, S_CUM, n_streams * kCumRow, &cum));
        TRY(scratch_t(ctx, S_DECMETA, n_streams, &meta));
        TRY(ensure_smem_opt_in(ctx));
        k_make_tile_dec_streams<<<blocks_for(n_streams, 256), 256, 0, ctx->stream>>>(g, n_tiles, d_packed, packed_bytes,
                                                                                     d_packed_off, streams, d_status);
        LAUNCHED("k_make_tile_dec_streams");
        k_parse_streams<<<blocks_for(n_streams, kTableWarps), kTableWarps * 32, 0, ctx->stream>>>(
            streams, (uint32_t)n_streams, d_packed, packed_bytes, cum, meta, results);
        LAUNCHED("k_parse_streams");
        const uint32_t classes[5] = {0, 64, 128, 256, HOH_MAX_RANGE + 3};
        const bool overlap = !ctx->profiling;
        if (overlap) TRY(aux_fork(ctx, 4));
        const unsigned grid = blocks_for(n_tiles, kFusedTiles);
        for (int c = 0; c < 4; c++) {
            const uint32_t rows = classes[c + 1];
            const size_t fixed = (size_t)rows * 32 * sizeof(uint32_t) + 32 * kRingWords * sizeof(uint32_t) + kFusedStage;
            // The kernel is bound by instruction-pipe throughput, so an SM's time grows with the number of warps it
            // holds: 13 CTAs of the smallest class would fit one SM, and with the other classes' launches running
            // beside it the block scheduler does fill some SMs that far while others hold 10.  Asking for the even
            // share caps every SM at 12 (BASELINE config 2: 1 639 warps = 11.07 per SM).
            const size_t lut_bytes = (size_t)kLutSize * 32 * (rows <= 256 ? 1 : 2);
            const size_t smem = smem_even_share(ctx, fixed + lut_bytes, grid);
            cudaStream_t sc = overlap ? ctx->aux[c] : ctx->stream;
            if (rows <= 256) {
                k_rans_decode_tiles_s0<uint8_t><<<grid, 32, smem, sc>>>(
                    streams, (uint32_t)n_streams, d_packed, packed_bytes, cum, meta, results, g, d_rgb, d_status, classes[c], rows);
            } else {
                k_rans_decode_tiles_s0<uint16_t><<<grid, 32, smem, sc>>>(
                    streams, (uint32_t)n_streams, d_packed, packed_bytes, cum, meta, results, g, d_rgb, d_status, classes[c], rows);
            }
            static const char* const names[4] = {"k_rans_decode_tiles_s0[rows<=64]", "k_rans_decode_tiles_s0[rows<=128]",
                                                 "k_rans_decode_tiles_s0[rows<=256]", "k_rans_decode_tiles_s0[rows<=515]"};
            LAUNCHED(names[c]);
        }
        if (overlap) TRY(aux_join(ctx, 4));
        return HOH_OK;
    }
    TRY(scratch_t(ctx, S_RESID, n_streams * g.plane_stride, &resid));
    const size_t unp_smem = (size_t)kUnpWarps * ((32 * kRingStride + g.tile_w + (g.tile_w + 1) / 2 + 3) & ~(size_t)3) * sizeof(uint32_t);
    if (unp_smem > 200 * 1024) return HOH_E_UNSUPPORTED;
    k_make_tile_dec_streams<<<blocks_for(n_streams, 256), 256, 0, ctx->stream>>>(g, n_tiles, d_packed, packed_bytes,
                                                                                 d_packed_off, streams, d_status);
    LAUNCHED("k_make_tile_dec_streams");
    TRY(decode_common(ctx, streams, n_streams, d_packed, packed_bytes, resid, results));
    k_merge_status<<<blocks_for(n_streams, 256), 256, 0, ctx->stream>>>(results, n_streams, g, d_backref ? 0u : 1u, d_status);
    LAUNCHED("k_merge_status");
    if (d_backref) {  // unprediction.hpp:63-65: copies make a pixel depend on any earlier one -> raster walk per plane
        uint16_t* planes;
        TRY(scratch_t(ctx, S_D_OUT, n_streams * g.plane_stride, &planes));
        k_tile_unpredict_s0_backref<<<blocks_for(n_streams, 64), 64, 0, ctx->stream>>>(resid, g, n_tiles, results, d_backref,
                                                                                      planes, d_status);
        LAUNCHED("k_tile_unpredict_s0_backref");
        k_tile_store_s0<<<(unsigned)n_tiles, 256, 0, ctx->stream>>>(planes, g, d_rgb);
        LAUNCHED("k_tile_store_s0");
        return HOH_OK;
    }
    if (g.width % 4 == 0 && g.tile_w % 4 == 0) {
        k_tile_unpredict_s0<true><<<blocks_for(n_tiles, kUnpWarps), kUnpWarps * 32, unp_smem, ctx->stream>>>(resid, g, n_tiles, d_rgb);
    } else {
        k_tile_unpredict_s0<false><<<blocks_for(n_tiles, kUnpWarps), kUnpWarps * 32, unp_smem, ctx->stream>>>(resid, g, n_tiles, d_rgb);
    }
    LAUNCHED("k_tile_unpredict_s0");
    return HOH_OK;
}

} // extern "C" (reopened below)

// Host-buffer tile codec: the batch is cut into chunks of whole images that flow through a three-stage pipeline —
// H2D copy (own stream), kernels, D2H copy (own stream) — so PCIe traffic in both directions overlaps the kernels and
// each other.  Chunk c goes through slot c % depth; a slot owns device staging, a pinned offset table and four events
// that hand the staging from one stage to the next.  The host waits only on those small offset tables: an encoded
// chunk's total decides how many bytes to fetch and where they go, and a decode slot's table is refilled on the host.
// The s0 calls keep kPipeDepth chunks in flight.  Their entropy kernels are bound by the serial chain of a stream, not
// by how many streams run (one chunk alone takes almost as long as the whole batch), so the chunks' kernels must
// themselves run CONCURRENTLY: each slot codes on its own child context (own stream, own scratch memory) and the GPU
// co-schedules their kernels.  The whole-tile calls keep two chunks in flight, coded on the context itself
// (tile_chunk_plan gives the reason).
namespace {

// The context that codes a slot's chunks, the context whose scratch holds its device staging, that staging and the
// pinned copy of its offset table.
struct PipeSlot {
    hoh_ctx* run = nullptr;
    hoh_ctx* stage = nullptr;
    uint8_t *rgb = nullptr, *packed = nullptr;
    uint64_t *off = nullptr, *h_off = nullptr;
    void* rec = nullptr;  // per-unit records: hoh_stream_result / hoh_tile_result (encode), int32_t status (decode)
};

// One host-buffer call: chunk c holds images bounds[c] .. bounds[c+1] and goes through slot c % depth.  A unit is one
// entry of the offset table: a stream (s0 calls) or a tile (whole-tile calls).  Every unit has a record, except in
// hoh_decode_regions_host, which has one status per image (recs = 1).
struct Pipe {
    hoh_ctx* ctx;
    std::vector<size_t> bounds;
    size_t raw1, units, rec_bytes;  // per image: bytes of pixels and units; bytes of one record
    size_t recs;                    // records per image
    size_t max_chunk = 0;           // images in the largest chunk
    int depth;
    PipeSlot slot[kPipeDepth];
    Pipe(hoh_ctx* c, std::vector<size_t> b, int max_depth, size_t raw_per_image, size_t units_per_image, size_t rec)
        : ctx(c), bounds(std::move(b)), raw1(raw_per_image), units(units_per_image), rec_bytes(rec), recs(units_per_image) {
        for (size_t k = 0; k < chunks(); k++) max_chunk = std::max(max_chunk, bounds[k + 1] - bounds[k]);
        depth = (int)std::min(chunks(), (size_t)max_depth);
    }
    size_t chunks() const { return bounds.size() - 1; }
};

int pipe_init(hoh_ctx* ctx) {
    if (ctx->pipe_ready) return HOH_OK;
    CK(cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking));
    for (int k = 0; k < kPipeDepth; k++) {
        CK(cudaEventCreateWithFlags(&ctx->ev_h2d[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_comp[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_d2h[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_off[k], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&ctx->ev_start, cudaEventDisableTiming));
    ctx->pipe_ready = true;
    return HOH_OK;
}
int pinned_off(hoh_ctx* ctx, int k, size_t entries, uint64_t** out) {
    if (ctx->h_off_cap[k] < entries) {
        if (ctx->h_off[k]) CK(cudaFreeHost(ctx->h_off[k]));
        ctx->h_off[k] = nullptr;
        CK(cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_off[k]), entries * sizeof(uint64_t), cudaHostAllocDefault));
        ctx->h_off_cap[k] = entries;
    }
    *out = ctx->h_off[k];
    return HOH_OK;
}
// smallest steady chunk in bytes of pixels (HOH_PIPE_CHUNK_KB: for tests, so that small batches take the chunked path)
size_t pipe_chunk_floor() {
    if (const char* e = getenv("HOH_PIPE_CHUNK_KB")) return (size_t)atol(e) << 10;
    return (size_t)64 << 20;
}
size_t chunk_images_for(size_t n_images, size_t raw_per_image) {
    // about 8 chunks, but not below ~64 MB of pixels per chunk (small batches are not worth pipelining)
    size_t per = (n_images + 7) / 8;
    const size_t min_per = pipe_chunk_floor() / (raw_per_image ? raw_per_image : 1) + 1;
    if (per < min_per) per = min_per;
    if (per > n_images) per = n_images;
    return per;
}
// Chunk boundaries (image indices, n_chunks + 1 of them) of an s0 host call.  What the pipeline cannot hide is its
// head and its tail: before the first chunk's kernels have run nothing flows back, and the last chunk's kernels and
// fetch run after the last byte has gone in.  A chunk's kernels last about as long whatever its size (one stream's
// serial chain), so both ends are made of short chunks that double up to the steady size: per/8, per/4, per/2, per, ...,
// per, per/2, per/4, per/8 (never below ~32 MB of pixels).
std::vector<size_t> chunk_plan(size_t n_images, size_t raw_per_image) {
    const size_t per = chunk_images_for(n_images, raw_per_image);
    std::vector<size_t> bounds{0};
    const size_t floor_per = pipe_chunk_floor() / 2 / (raw_per_image ? raw_per_image : 1) + 1;
    std::vector<size_t> ramp;
    for (size_t r = std::max<size_t>(per / 8, 1); r < per; r *= 2)
        if (r >= floor_per) ramp.push_back(r);
    size_t ramp_sum = 0;
    for (size_t r : ramp) ramp_sum += r;
    if (n_images < 2 * ramp_sum + 2 * per) {
        ramp.clear();
        ramp_sum = 0;
    }
    for (size_t r : ramp) bounds.push_back(bounds.back() + r);
    const size_t middle = n_images - 2 * ramp_sum, n_mid = (middle + per - 1) / per;
    for (size_t k = 0; k < n_mid; k++) bounds.push_back(bounds.back() + middle / n_mid + (k < middle % n_mid ? 1 : 0));
    for (size_t k = ramp.size(); k-- > 0;) bounds.push_back(bounds.back() + ramp[k]);
    return bounds;
}

// Allocates every slot's staging (packed_cap bytes of payloads) and makes the copy streams and the slots' streams wait
// for everything queued on the caller's stream so far.
int pipe_begin(Pipe& pp, size_t packed_cap) {
    hoh_ctx* ctx = pp.ctx;
    TRY(pipe_init(ctx));
    const size_t units = pp.max_chunk * pp.units;
    for (int b = 0; b < pp.depth; b++) {
        PipeSlot& s = pp.slot[b];
        TRY(scratch_t(s.stage, S_IO_A, pp.max_chunk * pp.raw1, &s.rgb));
        TRY(scratch_t(s.stage, S_IO_B, packed_cap, &s.packed));
        TRY(scratch_t(s.stage, S_IO_C, units + 1, &s.off));
        TRY(scratch(s.stage, S_IO_D, pp.max_chunk * pp.recs * pp.rec_bytes, &s.rec));
        TRY(pinned_off(ctx, b, units + 1, &s.h_off));
    }
    CK(cudaEventRecord(ctx->ev_start, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->s_h2d, ctx->ev_start, 0));
    CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_start, 0));
    for (int b = 0; b < pp.depth; b++)
        if (pp.slot[b].run != ctx) CK(cudaStreamWaitEvent(pp.slot[b].run->stream, ctx->ev_start, 0));
    return HOH_OK;
}

// Whatever way a host-buffer call ends, nothing may still read or write the caller's buffers when it returns.  The
// slots' child contexts launch on the caller's behalf: their launches count as the caller's.
struct PipeGuard {
    const Pipe& pp;
    uint64_t launches[kPipeDepth];
    explicit PipeGuard(const Pipe& p) : pp(p) {
        for (int b = 0; b < pp.depth; b++) launches[b] = pp.slot[b].run->launches;
    }
    ~PipeGuard() {
        hoh_ctx* ctx = pp.ctx;
        cudaStreamSynchronize(ctx->s_h2d);
        cudaStreamSynchronize(ctx->s_d2h);
        cudaStreamSynchronize(ctx->stream);
        for (hoh_ctx* ch : ctx->child)
            if (ch) cudaStreamSynchronize(ch->stream);
        for (int b = 0; b < pp.depth; b++)
            if (pp.slot[b].run != ctx) ctx->launches += pp.slot[b].run->launches - launches[b];
    }
};

// Encodes the chunks of a host-buffer call.  code(b, n_images) codes the chunk in slot b on the slot's run context:
// pixels in rgb, payloads to packed (dev_cap bytes), chunk-relative offsets to off, records to rec.  Chunk c's H2D copy
// and kernels are queued depth - 1 chunks ahead of the fetch of its payloads.  off_host receives the offsets into
// packed_host, rec_host (may be NULL) the records, chunk_base (may be NULL) where each chunk starts in packed_host.
template <class Code>
int pipe_encode(Pipe& pp, size_t dev_cap, const uint8_t* rgb_host, uint8_t* packed_host, size_t packed_cap,
                uint64_t* off_host, void* rec_host, uint64_t* chunk_base, Code code) {
    hoh_ctx* ctx = pp.ctx;
    TRY(pipe_begin(pp, dev_cap));
    PipeGuard guard(pp);
    const size_t n_chunks = pp.chunks(), depth = pp.depth, units = pp.units;
    uint64_t base = 0;
    off_host[0] = 0;
    for (size_t c = 0; c + 1 < n_chunks + depth; c++) {
        if (c < n_chunks) {  // copy in and code chunk c
            const int b = (int)(c % depth);
            const PipeSlot& s = pp.slot[b];
            const size_t first = pp.bounds[c], n_c = pp.bounds[c + 1] - first;
            if (c >= depth) CK(cudaStreamWaitEvent(ctx->s_h2d, ctx->ev_comp[b], 0));  // s.rgb consumed
            CK(cudaMemcpyAsync(s.rgb, rgb_host + first * pp.raw1, n_c * pp.raw1, cudaMemcpyHostToDevice, ctx->s_h2d));
            CK(cudaEventRecord(ctx->ev_h2d[b], ctx->s_h2d));
            CK(cudaStreamWaitEvent(s.run->stream, ctx->ev_h2d[b], 0));
            if (c >= depth) CK(cudaStreamWaitEvent(s.run->stream, ctx->ev_d2h[b], 0));  // s.packed fetched
            TRY(code(b, n_c));
            CK(cudaEventRecord(ctx->ev_comp[b], s.run->stream));
            // its offset table follows on the run stream (tiny; must not queue behind big fetches)
            CK(cudaMemcpyAsync(s.h_off, s.off, (n_c * units + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.run->stream));
            CK(cudaEventRecord(ctx->ev_off[b], s.run->stream));
        }
        if (c + 1 >= depth) {  // fetch chunk p = c - (depth - 1)
            const size_t p = c + 1 - depth;
            const int b = (int)(p % depth);
            const PipeSlot& s = pp.slot[b];
            const size_t u0 = pp.bounds[p] * units, nu = pp.bounds[p + 1] * units - u0;
            CK(cudaEventSynchronize(ctx->ev_off[b]));
            const uint64_t total = s.h_off[nu];
            if (total > dev_cap || base + total > packed_cap) return HOH_E_CAPACITY;
            CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_comp[b], 0));
            CK(cudaMemcpyAsync(packed_host + base, s.packed, total, cudaMemcpyDeviceToHost, ctx->s_d2h));
            if (rec_host)
                CK(cudaMemcpyAsync(static_cast<uint8_t*>(rec_host) + u0 * pp.rec_bytes, s.rec, nu * pp.rec_bytes,
                                   cudaMemcpyDeviceToHost, ctx->s_d2h));
            CK(cudaEventRecord(ctx->ev_d2h[b], ctx->s_d2h));
            for (size_t i = 1; i <= nu; i++) off_host[u0 + i] = base + s.h_off[i];
            if (chunk_base) chunk_base[p] = base;
            base += total;
        }
    }
    CK(cudaStreamSynchronize(ctx->s_d2h));
    return HOH_OK;
}

// pipe_decode's copy-in hook: where a chunk's payloads come from and where they land in its staging.  This one, for the
// whole-image calls, stages one range of packed_host per chunk, from its first unit's start to its last unit's end.
struct RangeIn {
    // bytes chunk c stages; HOH_E_ARG when its offsets run backwards or past packed_bytes
    int bytes(const Pipe& pp, size_t c, const uint64_t* off_host, size_t packed_bytes, uint64_t* out) const {
        const uint64_t lo = off_host[pp.bounds[c] * pp.units], hi = off_host[pp.bounds[c + 1] * pp.units];
        if (hi < lo || hi > packed_bytes) return HOH_E_ARG;
        *out = hi - lo;
        return HOH_OK;
    }
    // chunk c's offset table (units of the chunk + 1 entries) rebased onto its staging
    void rebase(const Pipe& pp, size_t c, const uint64_t* off_host, uint64_t* h_off) const {
        const size_t u0 = pp.bounds[c] * pp.units, nu = (pp.bounds[c + 1] - pp.bounds[c]) * pp.units;
        for (size_t i = 0; i <= nu; i++) h_off[i] = off_host[u0 + i] - off_host[u0];
    }
    // queues the copies of chunk c's payloads (bytes of them) into dst on the H2D copy stream
    int copy(const Pipe& pp, size_t c, const uint8_t* packed_host, const uint64_t* off_host, uint64_t bytes,
             uint8_t* dst) const {
        hoh_ctx* ctx = pp.ctx;
        CK(cudaMemcpyAsync(dst, packed_host + off_host[pp.bounds[c] * pp.units], bytes, cudaMemcpyHostToDevice, ctx->s_h2d));
        return HOH_OK;
    }
};

// Decodes the chunks of a host-buffer call.  code(b, n_images, packed_bytes) decodes the chunk in slot b on the slot's
// run context: payloads in packed (packed_bytes, zero padding included), chunk-relative offsets in off, pixels to rgb,
// records (status) to rec.  Per chunk: rebase its offsets on the host, pad, H2D payloads (through the copy-in hook
// `in`) and offsets, code, D2H pixels and records.  The hook's HOH_E_ARG (offsets that run backwards or past
// packed_bytes) comes before anything is queued.
template <class Code, class In = RangeIn>
int pipe_decode(Pipe& pp, const uint8_t* packed_host, size_t packed_bytes, const uint64_t* off_host, uint8_t* rgb_host,
                int32_t* status_host, Code code, const In& in = In()) {
    hoh_ctx* ctx = pp.ctx;
    const size_t n_chunks = pp.chunks(), depth = pp.depth, units = pp.units;
    std::vector<uint64_t> chunk_bytes(n_chunks);
    size_t max_packed = 0;
    for (size_t c = 0; c < n_chunks; c++) {
        TRY(in.bytes(pp, c, off_host, packed_bytes, &chunk_bytes[c]));
        max_packed = std::max<size_t>(max_packed, chunk_bytes[c]);
    }
    // >= 32 zero bytes behind a chunk's last payload byte (the decode input contract, hohgpu.h)
    auto padded = [](size_t bytes) { return (bytes + 47) & ~(size_t)15; };
    TRY(pipe_begin(pp, padded(max_packed)));
    PipeGuard guard(pp);
    for (size_t c = 0; c < n_chunks; c++) {
        const int b = (int)(c % depth);
        const PipeSlot& s = pp.slot[b];
        const size_t first = pp.bounds[c], n_c = pp.bounds[c + 1] - first, nu = n_c * units;
        const uint64_t bytes = chunk_bytes[c];
        const size_t aligned = bytes & ~(size_t)15;
        if (c >= depth) CK(cudaEventSynchronize(ctx->ev_h2d[b]));  // s.h_off was read by chunk c-depth's copy
        in.rebase(pp, c, off_host, s.h_off);
        if (c >= depth) CK(cudaStreamWaitEvent(ctx->s_h2d, ctx->ev_comp[b], 0));  // s.packed / s.off consumed
        CK(cudaMemsetAsync(s.packed + aligned, 0, padded(bytes) - aligned, ctx->s_h2d));
        TRY(in.copy(pp, c, packed_host, off_host, bytes, s.packed));
        CK(cudaMemcpyAsync(s.off, s.h_off, (nu + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->s_h2d));
        CK(cudaEventRecord(ctx->ev_h2d[b], ctx->s_h2d));
        CK(cudaStreamWaitEvent(s.run->stream, ctx->ev_h2d[b], 0));
        if (c >= depth) CK(cudaStreamWaitEvent(s.run->stream, ctx->ev_d2h[b], 0));  // s.rgb fetched
        TRY(code(b, n_c, padded(bytes)));
        CK(cudaEventRecord(ctx->ev_comp[b], s.run->stream));
        CK(cudaStreamWaitEvent(ctx->s_d2h, ctx->ev_comp[b], 0));
        CK(cudaMemcpyAsync(rgb_host + first * pp.raw1, s.rgb, n_c * pp.raw1, cudaMemcpyDeviceToHost, ctx->s_d2h));
        if (status_host)
            CK(cudaMemcpyAsync(status_host + first * pp.recs, s.rec, n_c * pp.recs * pp.rec_bytes, cudaMemcpyDeviceToHost,
                               ctx->s_d2h));
        CK(cudaEventRecord(ctx->ev_d2h[b], ctx->s_d2h));
    }
    CK(cudaStreamSynchronize(ctx->s_d2h));
    return HOH_OK;
}
}  // namespace
extern "C" {

int hoh_encode_images_s0_host(hoh_ctx* ctx, const uint8_t* rgb_host, size_t n_images, uint32_t width,
                              uint32_t height, uint8_t* packed_host, size_t packed_cap, uint64_t* off_host,
                              hoh_stream_result* results_host) {
    DeviceGuard guard_(ctx);
    if (!ctx || !rgb_host || !packed_host || !off_host) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const size_t raw1 = (size_t)width * height * 3;
    Pipe pp(ctx, chunk_plan(n_images, raw1), kPipeDepth, raw1, hg.streams_per_image, sizeof(hoh_stream_result));
    const size_t per = pp.max_chunk, out_bytes = hoh_encode_images_out_bytes(&hg, per);
    const size_t dev_cap = per * raw1 + per * raw1 / 4 + 4096 * per * pp.units;
    uint8_t* d_out[kPipeDepth];  // the slabs hoh_encode_images_s0 codes into before it gathers the payloads
    for (int b = 0; b < pp.depth; b++) {  // slot b codes on child[b], from staging there
        TRY(child_of(ctx, b, &pp.slot[b].run));
        pp.slot[b].stage = pp.slot[b].run;
        TRY(scratch_t(pp.slot[b].stage, S_IO_E, out_bytes, &d_out[b]));
    }
    return pipe_encode(pp, dev_cap, rgb_host, packed_host, packed_cap, off_host, results_host, nullptr,
                       [&](int b, size_t n_c) {
                           const PipeSlot& s = pp.slot[b];
                           return hoh_encode_images_s0(s.run, s.rgb, n_c, width, height, nullptr, d_out[b], out_bytes,
                                                       static_cast<hoh_stream_result*>(s.rec), s.packed, dev_cap, s.off);
                       });
}

int hoh_decode_images_s0_host(hoh_ctx* ctx, const uint8_t* packed_host, size_t packed_bytes,
                              const uint64_t* off_host, size_t n_images, uint32_t width, uint32_t height,
                              uint8_t* rgb_host, int32_t* status_host) {
    DeviceGuard guard_(ctx);
    if (!ctx || !rgb_host || !packed_host || !off_host) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const size_t raw1 = (size_t)width * height * 3;
    Pipe pp(ctx, chunk_plan(n_images, raw1), kPipeDepth, raw1, hg.streams_per_image, sizeof(int32_t));
    for (int b = 0; b < pp.depth; b++) {  // slot b decodes on child[b], from staging there
        TRY(child_of(ctx, b, &pp.slot[b].run));
        pp.slot[b].stage = pp.slot[b].run;
    }
    return pipe_decode(pp, packed_host, packed_bytes, off_host, rgb_host, status_host,
                       [&](int b, size_t n_c, size_t padded) {
                           const PipeSlot& s = pp.slot[b];
                           return hoh_decode_images_s0(s.run, s.packed, padded, s.off, n_c, width, height, nullptr,
                                                       s.rgb, static_cast<int32_t*>(s.rec));
                       });
}

// =================================================================================================
// batched plane kernels
// =================================================================================================
int hoh_subtract_green_dev(hoh_ctx* ctx, const uint8_t* d_rgb, size_t pixels, uint16_t* d_g, uint16_t* d_rg,
                           uint16_t* d_bg) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_rgb || !d_g || !d_rg || !d_bg) return HOH_E_ARG;
    if (!pixels) return HOH_OK;
    k_subtract_green<<<grid_cap(pixels, 256), 256, 0, ctx->stream>>>(d_rgb, pixels, d_g, d_rg, d_bg);
    LAUNCHED("k_subtract_green");
    return HOH_OK;
}

int hoh_add_green_dev(hoh_ctx* ctx, const uint16_t* d_g, const uint16_t* d_rg, const uint16_t* d_bg, size_t pixels,
                      uint8_t* d_rgb) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_rgb || !d_g || !d_rg || !d_bg) return HOH_E_ARG;
    if (!pixels) return HOH_OK;
    k_add_green<<<grid_cap(pixels, 256), 256, 0, ctx->stream>>>(d_g, d_rg, d_bg, pixels, d_rgb);
    LAUNCHED("k_add_green");
    return HOH_OK;
}

int hoh_channel_picker_dev(hoh_ctx* ctx, const uint8_t* d_src, size_t n_px, int total, int target, uint16_t* d_out) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_src || !d_out || total <= 0 || target < 0 || target >= total) return HOH_E_ARG;
    if (n_px == 0) return HOH_OK;
    k_channel_picker<<<grid_cap(n_px, 256), 256, 0, ctx->stream>>>(d_src, n_px, (uint32_t)total, (uint32_t)target, d_out);
    LAUNCHED("k_channel_picker");
    return HOH_OK;
}

int hoh_predict_fastpath_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                             uint16_t* d_resid) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_planes || !d_resid || w <= 0 || h <= 0 || depth < 1 || depth > 9) return HOH_E_ARG;
    if (!n_planes) return HOH_OK;
    k_predict_fastpath<<<grid_cap((uint64_t)n_planes * ((h + kFastpathBand - 1) / kFastpathBand) * 256, 256, 148u * 64u), w >= 192 ? 256 : 64, 0, ctx->stream>>>(d_planes, n_planes, w, h,
                                                                                          depth, d_resid, (uint64_t)w * h);
    LAUNCHED("k_predict_fastpath");
    return HOH_OK;
}

int hoh_unpredict_fastpath_dev(hoh_ctx* ctx, const uint16_t* d_resid, size_t n_planes, int w, int h, int depth,
                               const uint16_t* d_backref, uint16_t* d_planes) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_planes || !d_resid || w <= 0 || h <= 0 || depth < 1 || depth > 9) return HOH_E_ARG;
    if (!n_planes) return HOH_OK;
    TRY(ensure_smem_opt_in(ctx));
    if (d_backref || (size_t)w * 2 * 4 > 200 * 1024) {
        k_unpredict_fastpath_serial<<<blocks_for(n_planes, 64), 64, 0, ctx->stream>>>(d_resid, n_planes, w, h, depth,
                                                                                      d_backref, d_planes);
        LAUNCHED("k_unpredict_fastpath_serial");
    } else {
        k_unpredict_fastpath_wave<<<blocks_for(n_planes, 4), 128, (size_t)w * 2 * 4, ctx->stream>>>(
            d_resid, n_planes, w, h, depth, d_planes);
        LAUNCHED("k_unpredict_fastpath_wave");
    }
    return HOH_OK;
}

int hoh_predict_all_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                        int x_tiles, int y_tiles, const uint16_t* d_tile_maps, uint16_t* d_resid) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_planes || !d_resid || !d_tile_maps || w <= 0 || h <= 0 || depth < 1 || depth > 9 || x_tiles <= 0 ||
        y_tiles <= 0)
        return HOH_E_ARG;
    if (!n_planes) return HOH_OK;
    return predict_all_parallel(ctx, d_planes, n_planes, w, h, depth, x_tiles, y_tiles, d_tile_maps, d_resid,
                                (uint64_t)w * h);
}

int hoh_unpredict_all_dev(hoh_ctx* ctx, const uint16_t* d_resid, size_t n_planes, int w, int h, int depth,
                          int x_tiles, int y_tiles, const uint16_t* d_tile_maps, const uint16_t* d_backref,
                          uint16_t* d_planes) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_planes || !d_resid || !d_tile_maps || w <= 0 || h <= 0 || depth < 1 || depth > 9 || x_tiles <= 0 ||
        y_tiles <= 0)
        return HOH_E_ARG;
    if (!n_planes) return HOH_OK;
    uint16_t* top;
    uint8_t* bp;
    TRY(scratch_t(ctx, S_TOP, n_planes * (size_t)w, &top));
    TRY(scratch_t(ctx, S_BP, n_planes * (size_t)w, &bp));
    k_raster_walk<true><<<blocks_for(n_planes, 64), 64, 0, ctx->stream>>>(d_resid, n_planes, w, h, depth, x_tiles,
                                                                         y_tiles, d_tile_maps, d_backref, d_planes, top, bp, (uint64_t)w * h);
    LAUNCHED("k_raster_walk<unpredict>");
    return HOH_OK;
}

int hoh_predict_section_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                            int x_tiles, int y_tiles, const uint16_t* d_masks, int n_masks, uint16_t* d_resid,
                            uint32_t cell_cap, uint32_t* d_counts) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_planes || !d_resid || !d_masks || !d_counts || w <= 0 || h <= 0 || depth < 1 || depth > 9 ||
        x_tiles <= 0 || y_tiles <= 0 || n_masks <= 0)
        return HOH_E_ARG;
    if (!n_planes) return HOH_OK;
    const uint64_t jobs = (uint64_t)n_planes * x_tiles * y_tiles * n_masks;
    const int tw = (w + x_tiles - 1) / x_tiles;
    uint16_t* wtop = nullptr;
    uint8_t* wbp = nullptr;
    if (tw > kMaxCellW) {
        TRY(scratch_t(ctx, S_WIDE_TOP, jobs * tw, &wtop));
        TRY(scratch_t(ctx, S_WIDE_BP, jobs * tw, &wbp));
    }
    k_section<false><<<blocks_for(jobs, 64), 64, 0, ctx->stream>>>(d_planes, n_planes, w, h, depth, x_tiles, y_tiles,
                                                                  d_masks, n_masks, d_resid, cell_cap, d_counts, nullptr,
                                                                  nullptr, wtop, wbp);
    LAUNCHED("k_section<resid>");
    return HOH_OK;
}

} // extern "C" (reopened below)
namespace {
// resid_stride: u16 elements between consecutive residual planes (>= w*h)
int predictor_search_impl(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                          int mode, uint16_t* d_tile_maps, uint8_t* d_index_lists, uint16_t* d_resid,
                          uint64_t resid_stride) {
    if (!ctx || !d_planes || !d_resid || !d_tile_maps || !d_index_lists || w <= 0 || h <= 0 || depth < 1 ||
        depth > 9 || mode < 1)
        return HOH_E_ARG;
    if (!n_planes) return HOH_OK;
    const int grid = 40;  // layer_encode.hpp:124
    const int xt = (w + grid - 1) / grid, yt = (h + grid - 1) / grid;
    const int cells = xt * yt;
    const int n_masks = mode * 5 < 14 ? mode * 5 : 14;  // layer_encode.hpp:178
    const int c = 1 << depth;
    const uint64_t per = (uint64_t)w * h;
    const uint64_t jobs = (uint64_t)n_planes * cells * n_masks;
    uint32_t* hist;
    double *cost, *sums, *e_tab;
    uint16_t* masks;
    uint16_t* top;
    uint8_t* bp;
    uint32_t e_len;
    TRY(scratch_t(ctx, S_HIST, n_planes * (size_t)c, &hist));
    TRY(scratch_t(ctx, S_COST, n_planes * (size_t)c, &cost));
    TRY(scratch_t(ctx, S_SUMS, jobs, &sums));
    TRY(scratch_t(ctx, S_MASKS, 16, &masks));
    TRY(scratch_t(ctx, S_TOP, n_planes * (size_t)w, &top));
    TRY(scratch_t(ctx, S_BP, n_planes * (size_t)w, &bp));
    TRY(cost_table_for(ctx, per, &e_tab, &e_len));
    CK(cudaMemcpyAsync(masks, kStockMasks, sizeof kStockMasks, cudaMemcpyHostToDevice, ctx->stream));
    k_predict_fastpath<<<grid_cap((uint64_t)n_planes * ((h + kFastpathBand - 1) / kFastpathBand) * 256, 256, 148u * 64u), w >= 192 ? 256 : 64, 0, ctx->stream>>>(d_planes, n_planes, w, h, depth, d_resid,
                                                                                resid_stride);
    LAUNCHED("k_predict_fastpath");
    const int passes = mode > 2 ? 2 : 1;  // layer_encode.hpp:215
    for (int pass = 0; pass < passes; pass++) {
        k_plane_histogram<<<(unsigned)n_planes, 256, 0, ctx->stream>>>(d_resid, (uint32_t)per, depth, hist, resid_stride);
        LAUNCHED("k_plane_histogram");
        k_cost_from_hist<<<blocks_for(n_planes * (uint64_t)c, 256), 256, 0, ctx->stream>>>(hist, n_planes * (uint64_t)c,
                                                                                          e_tab, e_len, cost);
        LAUNCHED("k_cost_from_hist");
        {  // all masks of a cell in one walk: one thread per (plane, cell)
            const uint64_t cell_jobs = (uint64_t)n_planes * cells;
            const unsigned blocks = blocks_for(cell_jobs, 64);
            // `masks` holds the reference's own list (kStockMasks): the STOCK instantiations have it compiled in
            if (n_masks == 5)
                k_section_costs<5, true><<<blocks, 64, 0, ctx->stream>>>(d_planes, n_planes, w, h, depth, xt, yt, masks, cost, sums);
            else if (n_masks == 10)
                k_section_costs<10, true><<<blocks, 64, 0, ctx->stream>>>(d_planes, n_planes, w, h, depth, xt, yt, masks, cost, sums);
            else
                k_section_costs<14, true><<<blocks, 64, 0, ctx->stream>>>(d_planes, n_planes, w, h, depth, xt, yt, masks, cost, sums);
            LAUNCHED("k_section_costs");
        }
        k_pick_masks<<<blocks_for(n_planes * (uint64_t)cells, 256), 256, 0, ctx->stream>>>(
            sums, n_planes * (uint64_t)cells, n_masks, masks, d_tile_maps, d_index_lists);
        LAUNCHED("k_pick_masks");
        TRY(predict_all_parallel(ctx, d_planes, n_planes, w, h, depth, xt, yt, d_tile_maps, d_resid, resid_stride));
    }
    return HOH_OK;
}
}  // namespace
extern "C" {

int hoh_predictor_search_dev(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                             int mode, uint16_t* d_tile_maps, uint8_t* d_index_lists, uint16_t* d_resid) {
    DeviceGuard guard_(ctx);
    return predictor_search_impl(ctx, d_planes, n_planes, w, h, depth, mode, d_tile_maps, d_index_lists, d_resid,
                                 (uint64_t)w * h);
}

// -------------------------------------------------------------------------------------------------
// layer_encode.hpp:11 for many planes
// -------------------------------------------------------------------------------------------------
static LayerGeom layer_geom(int w, int h, int depth, int mode) {
    LayerGeom lg;
    lg.per = (uint32_t)w * h;
    lg.per_pad = (lg.per + 7u) & ~7u;
    lg.xt = (w + 39) / 40;
    lg.yt = (h + 39) / 40;
    lg.cells = (mode >= 1 && (lg.xt > 1 || lg.yt > 1)) ? lg.xt * lg.yt : 0u;  // layer_encode.hpp:126-132
    lg.cells_pad = (lg.cells + 7u) & ~7u;
    lg.depth = depth;
    lg.mode = mode;
    lg.enc_flags = 0;
    // candidate slabs sized by what each is coded with: A 15 bits, B the index map at 8, C 16, D 15, E-G up to 19
    const uint32_t bits_of[kLayerSlots] = {15, 8, 16, 15, 17, 18, 19, 14, 13, 12};
    uint32_t at = 0, widest = 0;
    for (int k = 0; k < kLayerSlots; k++) {
        const bool used = k == 0 || (mode >= 1 && (k != 1 || lg.cells));
        lg.slot_cap[k] = used ? (uint32_t)hoh_enc_slab_bytes(k == 1 ? lg.cells : lg.per, bits_of[k]) : 0u;
        lg.slot_off[k] = at;
        at += lg.slot_cap[k];
        if (k != 1 && lg.slot_cap[k] > widest) widest = lg.slot_cap[k];
    }
    lg.plane_bytes = at;
    lg.out_cap = (kLayerHdrCap + lg.slot_cap[1] + widest + 15u) & ~15u;
    return lg;
}

size_t hoh_layer_encode_out_bytes(size_t n_planes, int w, int h, int depth, int mode) {
    const LayerGeom lg = layer_geom(w, h, depth, mode);
    return n_planes * ((size_t)lg.plane_bytes + lg.out_cap);
}

int hoh_layer_encode_batch(hoh_ctx* ctx, const uint16_t* d_planes, size_t n_planes, int w, int h, int depth,
                           int mode, unsigned flags, const uint8_t* d_nuke, size_t nuke_stride, uint32_t planes_per_map,
                           uint8_t* d_out, size_t out_bytes, hoh_stream_result* d_results,
                           uint8_t* d_packed, size_t packed_cap, uint64_t* d_packed_off) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_planes || !d_out || !d_results || w <= 0 || h <= 0 || depth < 1 || depth > 9 || mode < 0 || mode > 4)
        return HOH_E_ARG;
    if (d_nuke && (planes_per_map == 0 || nuke_stride < (size_t)w * h)) return HOH_E_ARG;
    if (n_planes == 0) return HOH_OK;
    if ((uint64_t)w * h >= (1u << 21)) return HOH_E_UNSUPPORTED;  // varint.hpp:39-45
    LayerGeom lg = layer_geom(w, h, depth, mode);
    lg.enc_flags = flags & HOH_FIX_LONE;
    if (lg.xt > 256 || lg.yt > 256) return HOH_E_UNSUPPORTED;    // grid size bytes (layer_encode.hpp:276-277)
    if (out_bytes < hoh_layer_encode_out_bytes(n_planes, w, h, depth, mode)) return HOH_E_CAPACITY;
    const size_t n = n_planes;
    uint16_t *syms, *maps;
    uint8_t *idx, *hdr;
    uint32_t *n_used, *hdr_len, *kept, *best, *kept_px = nullptr;
    int32_t* status;
    hoh_enc_stream* streams;
    hoh_stream_result *rr, *res;
    TRY(scratch_t(ctx, S_RESID, 2 * n * lg.per_pad + n * lg.cells_pad, &syms));
    TRY(scratch_t(ctx, S_L_MAPS, n * (lg.cells ? lg.cells : 1), &maps));
    TRY(scratch_t(ctx, S_L_IDX, n * (lg.cells ? lg.cells : 1), &idx));
    TRY(scratch_t(ctx, S_L_HDR, n * kLayerHdrCap, &hdr));
    uint32_t* with_idx;
    TRY(scratch_t(ctx, S_L_U32, 6 * n, &n_used));
    hdr_len = n_used + n;
    kept = hdr_len + n;
    best = kept + n;
    with_idx = best + n;
    if (d_nuke) kept_px = with_idx + n;
    TRY(scratch_t(ctx, S_L_STATUS, n, &status));
    TRY(scratch_t(ctx, S_STREAMS, 9 * n, &streams));
    TRY(scratch_t(ctx, S_L_RR, 9 * n, &rr));
    TRY(scratch_t(ctx, S_L_RES, (size_t)kLayerSlots * n, &res));
    CK(cudaMemsetAsync(res, 0, (size_t)kLayerSlots * n * sizeof(hoh_stream_result), ctx->stream));
    uint16_t* resid0 = syms;
    uint16_t* resid1 = syms + n * lg.per_pad;
    const uint32_t range = 1u << depth;
    auto run_round = [&](int round, uint32_t max_range, uint32_t max_pb) -> int {
        const uint32_t per_plane = round == 0 ? (mode >= 1 ? 9u : 1u) : (round == 1 ? 1u : 3u);
        const size_t count = n * per_plane;
        k_layer_streams<<<blocks_for(count, 256), 256, 0, ctx->stream>>>(lg, n, round, n_used, kept_px, res, streams);
        LAUNCHED("k_layer_streams");
        if (round != 1) {  // one histogram per residual array instead of one per stream
            uint32_t* freqs;
            TRY(scratch_t(ctx, S_FREQS, count * kFreqRow, &freqs));
            const uint32_t a = round == 3 ? 0u : 1u, b_first = round == 3 ? 0u : 1u;
            const uint32_t b = round == 0 ? (mode >= 1 ? 8u : 0u) : (round == 2 ? 2u : 3u);
            k_layer_histograms<<<(unsigned)(2 * n), 256, 0, ctx->stream>>>(n, per_plane, a, b_first, b, streams, syms, freqs);
            LAUNCHED("k_layer_histograms");
            TRY(encode_from_freqs(ctx, streams, count, syms, d_out, rr, freqs, max_range, max_pb, 0, true));
        } else {
            TRY(hoh_encode_entropy_batch(ctx, streams, count, syms, d_out, rr, max_range, max_pb, lg.per));
        }
        k_layer_scatter<<<blocks_for(count, 256), 256, 0, ctx->stream>>>(lg, n, round, rr, res);
        LAUNCHED("k_layer_scatter");
        return HOH_OK;
    };
    // layer_encode.hpp:63-120: fastpath residuals
    k_predict_fastpath<<<grid_cap((uint64_t)n * ((h + kFastpathBand - 1) / kFastpathBand) * 256, 256, 148u * 64u), w >= 192 ? 256 : 64, 0, ctx->stream>>>(d_planes, n, w, h, depth, resid0,
                                                                                  lg.per_pad);
    LAUNCHED("k_predict_fastpath");
    auto compact = [&](uint16_t* resid) -> int {  // :93-99, :328-333
        if (!d_nuke) return HOH_OK;
        k_compact_planes<<<blocks_for(n * 32, 128), 128, 0, ctx->stream>>>(n, lg.per, lg.per_pad, d_nuke, nuke_stride,
                                                                          planes_per_map, resid, kept_px);
        LAUNCHED("k_compact_planes");
        return HOH_OK;
    };
    TRY(compact(resid0));
    if (mode >= 1 && lg.cells) {  // :126-272
        TRY(predictor_search_impl(ctx, d_planes, n, w, h, depth, mode, maps, idx, resid1, lg.per_pad));
        TRY(compact(resid1));
    }
    k_layer_headers<<<blocks_for(n, 64), 64, 0, ctx->stream>>>(lg, n, idx, syms, n_used, hdr, hdr_len);
    LAUNCHED("k_layer_headers");
    if (mode >= 1 && lg.cells) TRY(run_round(1, 14, 8));  // the predictor-index maps (:308-317)
    // The candidates (:106, 334-392).  The reference codes six of them per plane and keeps one.  Here the tables of all
    // nine (both prob_bits directions) are built, which gives every candidate's size up to one word without coding it
    // (warp_estimate_words); k_layer_plan replays the decisions over those intervals and only the candidates whose bytes
    // or exact size the outcome needs go through the coder, as one dense list (typically one per plane).
    // HOH_LAYER_CODE_ALL=1 codes every candidate on the path (the previous behaviour, for tests and comparisons).
    if (mode == 0) {
        TRY(run_round(0, range, 15));
    } else {
        const size_t count = 9 * n;
        uint8_t* need;
        uint32_t* order;
        TRY(scratch_t(ctx, S_L_NEED, count, &need));
        TRY(scratch_t(ctx, S_L_ORDER, count + 1, &order));
        uint32_t* n_active = order + count;
        if (!ctx->d_layer_stats) {
            CK(cudaMalloc(&ctx->d_layer_stats, 4 * sizeof(uint32_t)));
            CK(cudaMemsetAsync(ctx->d_layer_stats, 0, 4 * sizeof(uint32_t), ctx->stream));
        }
        k_layer_streams<<<blocks_for(count, 256), 256, 0, ctx->stream>>>(lg, n, 0, n_used, kept_px, res, streams);
        LAUNCHED("k_layer_streams");
        uint32_t* freqs;
        TRY(scratch_t(ctx, S_FREQS, count * kFreqRow, &freqs));
        k_layer_histograms<<<(unsigned)(2 * n), 256, 0, ctx->stream>>>(n, 9u, 1u, 1u, 8u, streams, syms, freqs);
        LAUNCHED("k_layer_histograms");
        uint32_t* cum;
        uint8_t* heads;
        EncMeta* meta;
        TRY(build_tables(ctx, streams, count, freqs, &cum, &heads, &meta));
        const bool code_all = getenv("HOH_LAYER_CODE_ALL") != nullptr;
        k_layer_plan<<<blocks_for(n, 128), 128, 0, ctx->stream>>>(lg, n, streams, meta, res, hdr_len,
                                                                  (flags & HOH_FIX_STALE) ? 1u : 0u, code_all ? 1u : 0u, need,
                                                                  ctx->d_layer_stats);
        LAUNCHED("k_layer_plan");
        k_layer_order<<<1, 1024, 0, ctx->stream>>>(need, streams, (uint32_t)count, order, n_active);
        LAUNCHED("k_layer_order");
        k_layer_est_results<<<blocks_for(count, 256), 256, 0, ctx->stream>>>(count, streams, meta, rr);
        LAUNCHED("k_layer_est_results");
        TRY(encode_with_tables(ctx, streams, count, syms, d_out, rr, cum, heads, meta, range, 19, 0, true, order, n_active));
        k_layer_scatter<<<blocks_for(count, 256), 256, 0, ctx->stream>>>(lg, n, 0, rr, res);
        LAUNCHED("k_layer_scatter");
    }
    k_layer_decide<<<blocks_for(n, 128), 128, 0, ctx->stream>>>(lg, n, res, (flags & HOH_FIX_STALE) ? 1u : 0u, hdr, hdr_len,
                                                                kept, best, with_idx, status);
    LAUNCHED("k_layer_decide");
    const uint64_t out_base = (uint64_t)n * lg.plane_bytes;
    k_layer_assemble<<<(unsigned)n, 256, 0, ctx->stream>>>(lg, hdr, hdr_len, res, kept, best, with_idx, status, d_out, d_out,
                                                           out_base, d_results);
    LAUNCHED("k_layer_assemble");
    if (d_packed) {
        if (!d_packed_off) return HOH_E_ARG;
        k_scan_sizes<<<1, 1024, 0, ctx->stream>>>(d_results, (uint32_t)n, d_packed_off);
        LAUNCHED("k_scan_sizes");
        k_gather_streams<<<(unsigned)n, 256, 0, ctx->stream>>>(d_results, d_out, d_packed_off, d_packed, packed_cap);
        LAUNCHED("k_gather_streams");
    }
    return HOH_OK;
}

} // extern "C" (reopened below)
namespace {
// The tile shapes of an image (choh.cpp:459-474): the last column and the last row take what is left of the
// image, so there are up to four shapes, each a rectangular sub-grid of the tile grid.
struct TileClass {
    TileSel sel;
    int tw, th;
};
int tile_classes(const TileGeom& g, TileClass out[4]) {
    const uint32_t rw = g.width - (g.x_tiles - 1) * g.tile_w, bh = g.height - (g.y_tiles - 1) * g.tile_h;
    uint32_t xs[2][3], ys[2][3];  // {first, count, size}
    int nx = 0, ny = 0;
    if (rw == g.tile_w) {
        xs[nx][0] = 0, xs[nx][1] = g.x_tiles, xs[nx][2] = g.tile_w, nx++;
    } else {
        if (g.x_tiles > 1) xs[nx][0] = 0, xs[nx][1] = g.x_tiles - 1, xs[nx][2] = g.tile_w, nx++;
        xs[nx][0] = g.x_tiles - 1, xs[nx][1] = 1, xs[nx][2] = rw, nx++;
    }
    if (bh == g.tile_h) {
        ys[ny][0] = 0, ys[ny][1] = g.y_tiles, ys[ny][2] = g.tile_h, ny++;
    } else {
        if (g.y_tiles > 1) ys[ny][0] = 0, ys[ny][1] = g.y_tiles - 1, ys[ny][2] = g.tile_h, ny++;
        ys[ny][0] = g.y_tiles - 1, ys[ny][1] = 1, ys[ny][2] = bh, ny++;
    }
    int n = 0;
    for (int j = 0; j < ny; j++)
        for (int i = 0; i < nx; i++) {
            TileClass& c = out[n++];
            c.sel.g = g;
            c.sel.x_first = xs[i][0];
            c.sel.x_count = xs[i][1];
            c.sel.y_first = ys[j][0];
            c.sel.y_count = ys[j][1];
            c.sel.per_image = xs[i][1] * ys[j][1];
            c.tw = (int)xs[i][2];
            c.th = (int)ys[j][2];
        }
    return n;
}
TileSel whole_grid(const TileGeom& g) {
    TileSel s;
    s.g = g;
    s.x_first = s.y_first = 0;
    s.x_count = g.x_tiles;
    s.y_count = g.y_tiles;
    s.per_image = g.tiles_per_image;
    return s;
}
constexpr int kTSlots = 9;  // scratch buffers of one tile shape in hoh_encode_images (S_T_NUKE .. S_T_R9)
inline Slot tslot(int cls, Slot base) { return (Slot)(S_T_NUKE + cls * kTSlots + (base - S_T_NUKE)); }
}  // namespace
extern "C" {

// -------------------------------------------------------------------------------------------------
// lz.hpp:6 for many tiles
// -------------------------------------------------------------------------------------------------
static uint32_t lz_side_stride(size_t npx) { return (uint32_t)((npx / 3 + 1 + 7) & ~(size_t)7); }  // lz.hpp:23-26: size/9 entries

size_t hoh_find_lz_stride(int w, int h) {
    if (w <= 0 || h <= 0) return 0;
    const size_t npx = (size_t)w * h;
    // each side stream: 8 bytes of varints/metadata, a table of at most ~520 bytes, 10 bits per symbol
    return (1 + 4 * hoh_enc_slab_bytes(lz_side_stride(npx), 10) + 15) & ~(size_t)15;
}

} // extern "C" (reopened below)
namespace {
// shared body of the two LZ entry points; nuke_stride = elements per tile in d_nuke
int find_lz_impl(hoh_ctx* ctx, const uint8_t* d_rgb, LzShape sh, size_t n_tiles, size_t max_npx, int distance, unsigned flags,
                 const int32_t* d_bonus, uint8_t* d_nuke, uint32_t nuke_stride, uint8_t* d_lz, size_t lz_stride,
                 uint32_t* d_lz_size, int32_t* d_status, uint32_t* d_info = nullptr) {
    if (max_npx >= (1u << 21) * 3ull) return HOH_E_UNSUPPORTED;  // side streams must stay below 2^21 symbols (varint.hpp:39-45)
    const uint32_t stride = lz_side_stride(max_npx);
    const uint32_t slab = (uint32_t)hoh_enc_slab_bytes(stride, 10);
    if (lz_stride < (1 + 4 * (size_t)slab + 15) / 16 * 16 || lz_stride > 0xffffffffull) return HOH_E_CAPACITY;
    const uint32_t wide = distance > 8;
    const uint32_t row_limit = (flags & HOH_FIX_LONE) ? 65535u : 65536u;  // lz.hpp:54 / :88-89, see k_lz_match
    sh.pad = 1u << distance;
    sh.px_stride = sh.pad + (sh.stride + kLzSeg - 1) / kLzSeg * kLzSeg + 32 * kLzAhead;
    uint32_t *px, *state, *counts;
    uint16_t* side;
    uint8_t* slabs;
    int32_t* bonus = nullptr;
    hoh_enc_stream* streams;
    hoh_stream_result* res;
    TRY(scratch_t(ctx, S_LZ_PX, n_tiles * sh.px_stride, &px));
    TRY(scratch_t(ctx, S_LZ_STATE, n_tiles * sh.stride, &state));
    TRY(scratch_t(ctx, S_LZ_SIDE, n_tiles * 4 * stride, &side));
    TRY(scratch_t(ctx, S_LZ_COUNTS, n_tiles * 4, &counts));
    TRY(scratch_t(ctx, S_LZ_SLABS, n_tiles * 4 * slab, &slabs));
    TRY(scratch_t(ctx, S_LZ_RES, n_tiles * 4, &res));
    TRY(scratch_t(ctx, S_STREAMS, n_tiles * 4, &streams));
    k_lz_pack<<<(unsigned)n_tiles, 256, 0, ctx->stream>>>(d_rgb, sh, px);
    LAUNCHED("k_lz_pack");
    if (!d_bonus || d_info) {
        TRY(scratch_t(ctx, S_LZ_BONUS, n_tiles, &bonus));
        k_lz_bonus<<<(unsigned)n_tiles, 256, 0, ctx->stream>>>(px, sh, bonus, d_info);
        LAUNCHED("k_lz_bonus");
        if (!d_bonus) d_bonus = bonus;
    }
    const uint64_t segs = (sh.stride + kLzSeg - 1) / kLzSeg;
    uint32_t* flag = nullptr;
    if (distance >= 10 && !getenv("HOH_LZ_DENSE")) {
        // wide windows: candidates from chains of 4-pixel hashes; the dense scan only redoes flagged tiles
        uint32_t *heads, *next;
        TRY(scratch_t(ctx, S_LZ_KEYS, (size_t)n_tiles * kLzHeads, &heads));
        TRY(scratch_t(ctx, S_LZ_VALS, (size_t)n_tiles * sh.stride, &next));
        TRY(scratch_t(ctx, S_LZ_FLAG, n_tiles, &flag));
        CK(cudaMemsetAsync(flag, 0, n_tiles * sizeof(uint32_t), ctx->stream));
        CK(cudaMemsetAsync(heads, 0xff, (size_t)n_tiles * kLzHeads * sizeof(uint32_t), ctx->stream));
        const uint64_t bpt = (sh.stride + 255) / 256;
        k_lz_chains<<<(unsigned)(n_tiles * bpt), 256, 0, ctx->stream>>>(px, sh, n_tiles, heads, next);
        LAUNCHED("k_lz_chains");
        k_lz_match_sparse<<<(unsigned)(n_tiles * bpt), 256, 0, ctx->stream>>>(px, sh, n_tiles, 1u << distance, row_limit, heads, next, state,
                                                                             flag);
        LAUNCHED("k_lz_match_sparse");
    }
    k_lz_match<<<blocks_for(n_tiles * segs * 32, 128), 128, 0, ctx->stream>>>(px, sh, n_tiles, 1u << distance, wide ? row_limit : 0u, state,
                                                                             flag);
    LAUNCHED("k_lz_match");
    k_lz_walk<<<blocks_for(n_tiles * 32, 128), 128, 0, ctx->stream>>>(state, sh, n_tiles, d_bonus, 0, wide, d_nuke,
                                                                     nuke_stride, side, stride, counts);
    LAUNCHED("k_lz_walk");
    k_lz_streams<<<blocks_for(n_tiles * 4, 256), 256, 0, ctx->stream>>>(n_tiles, counts, stride, slab, flags & HOH_FIX_LONE,
                                                                        streams);
    LAUNCHED("k_lz_streams");
    TRY(hoh_encode_entropy_batch(ctx, streams, n_tiles * 4, side, slabs, res, 256, 10, stride));
    k_lz_assemble<<<(unsigned)n_tiles, 128, 0, ctx->stream>>>(res, slabs, wide, d_lz, (uint32_t)lz_stride, d_lz_size,
                                                             d_status);
    LAUNCHED("k_lz_assemble");
    return HOH_OK;
}
}  // namespace
extern "C" {

int hoh_find_lz_rgb_batch(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_tiles, int w, int h, int distance,
                          unsigned flags, const int32_t* d_bonus, uint8_t* d_nuke, uint8_t* d_lz, size_t lz_stride,
                          uint32_t* d_lz_size, int32_t* d_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_rgb || !d_nuke || !d_lz || !d_lz_size || w <= 0 || h <= 0 || distance < 0 || distance > 16)
        return HOH_E_ARG;
    if (n_tiles == 0) return HOH_OK;
    const size_t npx = (size_t)w * h;
    if (npx > 0xffffffffull) return HOH_E_UNSUPPORTED;
    LzShape sh;
    memset(&sh, 0, sizeof(sh));
    sh.tiled = 0;
    sh.npx = (uint32_t)npx;
    sh.width = (uint32_t)w;
    sh.stride = (uint32_t)npx;
    return find_lz_impl(ctx, d_rgb, sh, n_tiles, npx, distance, flags, d_bonus, d_nuke, (uint32_t)npx, d_lz, lz_stride, d_lz_size,
                        d_status);
}

int hoh_find_lz_images(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_images, uint32_t width, uint32_t height,
                       int distance, unsigned flags, const int32_t* d_bonus, uint8_t* d_nuke, uint8_t* d_lz, size_t lz_stride,
                       uint32_t* d_lz_size, int32_t* d_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_rgb || !d_nuke || !d_lz || !d_lz_size || distance < 0 || distance > 16) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    LzShape sh;
    memset(&sh, 0, sizeof(sh));
    sh.tiled = 1;
    sh.sel = whole_grid(to_geom(hg));
    sh.stride = sh.sel.g.plane_stride;
    return find_lz_impl(ctx, d_rgb, sh, n_images * sh.sel.g.tiles_per_image, (size_t)hg.tile_w * hg.tile_h, distance, flags, d_bonus,
                        d_nuke, sh.sel.g.plane_stride, d_lz, lz_stride, d_lz_size, d_status);
}

// -------------------------------------------------------------------------------------------------
// encode_tile for the tiles of whole images, any cruncher mode
// -------------------------------------------------------------------------------------------------
int hoh_encode_images(hoh_ctx* ctx, const uint8_t* d_rgb, size_t n_images, uint32_t width, uint32_t height,
                      int mode, unsigned flags, uint8_t* d_packed, size_t packed_cap, uint64_t* d_tile_off,
                      hoh_tile_result* d_tiles) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_rgb || !d_packed || !d_tile_off || !d_tiles || mode < 0 || mode > 4) return HOH_E_ARG;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    CK(cudaMemsetAsync(d_tile_off, 0, sizeof(uint64_t), ctx->stream));
    if (n_images == 0) return HOH_OK;
    const TileGeom g = to_geom(hg);
    TileClass cls[4];
    const int n_cls = tile_classes(g, cls);
    static const int dist_of_mode[5] = {6, 10, 11, 12, 14};  // choh.cpp:123-136
    const int distance = dist_of_mode[mode];
    const uint32_t per8 = mode > 2 ? 3u : 1u;
    // scratch per IMAGE: this function's buffers + what the LZ finder and layer_encode_batch allocate themselves.
    // The candidates of every shape stay alive until the image chunk's tiles have been emitted in tile order.
    size_t lz_stride[4], out8_tile[4], out9_tile[4], per_image = 0;
    for (int c = 0; c < n_cls; c++) {
        const size_t npx = (size_t)cls[c].tw * cls[c].th;
        lz_stride[c] = hoh_find_lz_stride(cls[c].tw, cls[c].th);
        out8_tile[c] = hoh_layer_encode_out_bytes(per8, cls[c].tw, cls[c].th, 8, mode);
        out9_tile[c] = hoh_layer_encode_out_bytes(2, cls[c].tw, cls[c].th, 9, mode);
        const size_t lz_words = (1u << distance) + (npx + kLzSeg) + 32 * kLzAhead;
        per_image += cls[c].sel.per_image *
                     ((per8 + 2) * npx * 2 + out8_tile[c] + out9_tile[c] + lz_stride[c] + g.plane_stride + lz_words * 4 +
                      npx * 4 + (distance >= 10 ? 4 * npx + 4 * (size_t)kLzHeads : 0) + 4 * (size_t)lz_side_stride(npx) * 2 +
                      4 * hoh_enc_slab_bytes(lz_side_stride(npx), 10) +
                      3 * (2 * npx * 2 + 8192) + 4096);
    }
    TRY(new_shape(ctx, ((uint64_t)width << 40) ^ ((uint64_t)height << 16) ^ ((uint64_t)mode << 8) ^ 1u, ctx->enc_key));
    const size_t budget = scratch_budget(ctx);
    size_t images_per_chunk = budget / per_image;
    if (images_per_chunk == 0) images_per_chunk = 1;
    if (images_per_chunk > n_images) images_per_chunk = n_images;
    uint8_t *nuke[4], *lz[4], *out8[4], *out9[4];
    uint32_t* u32[4];
    uint16_t *p8[4], *p9[4];
    hoh_stream_result *r8[4], *r9[4];
    for (int c = 0; c < n_cls; c++) {
        const size_t ct = images_per_chunk * cls[c].sel.per_image, npx = (size_t)cls[c].tw * cls[c].th;
        TRY(scratch_t(ctx, tslot(c, S_T_NUKE), ct * g.plane_stride, &nuke[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_LZ), ct * lz_stride[c], &lz[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_U32), ct * 3, &u32[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_P8), ct * per8 * npx, &p8[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_P9), ct * 2 * npx, &p9[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_O8), ct * out8_tile[c], &out8[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_O9), ct * out9_tile[c], &out9[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_R8), ct * per8, &r8[c]));
        TRY(scratch_t(ctx, tslot(c, S_T_R9), ct * 2, &r9[c]));
    }
    for (size_t img0 = 0; img0 < n_images; img0 += images_per_chunk) {
        const size_t ni = std::min(images_per_chunk, n_images - img0);
        const uint8_t* rgb = d_rgb + img0 * (size_t)width * height * 3;
        for (int c = 0; c < n_cls; c++) {
            const TileSel& sel = cls[c].sel;
            const int tw = cls[c].tw, th = cls[c].th;
            const size_t nt = ni * sel.per_image, npx = (size_t)tw * th;
            uint32_t* lz_size = u32[c];
            int32_t* lz_status = reinterpret_cast<int32_t*>(u32[c] + nt);
            uint32_t* info = u32[c] + 2 * nt;
            LzShape sh;
            memset(&sh, 0, sizeof(sh));
            sh.tiled = 1;
            sh.sel = sel;
            sh.stride = g.plane_stride;
            TRY(find_lz_impl(ctx, rgb, sh, nt, npx, distance, flags, nullptr, nuke[c], g.plane_stride, lz[c], lz_stride[c],
                             lz_size, lz_status, info));
            k_tile_planes<<<(unsigned)nt, 256, 0, ctx->stream>>>(rgb, sel, per8, p8[c], p9[c]);
            LAUNCHED("k_tile_planes");
            // the 8-bit planes and the 9-bit planes are two independent batches, each bound by stream length rather
            // than stream count: they run side by side in two child contexts (own stream, own scratch)
            hoh_ctx* c8 = ctx;
            hoh_ctx* c9 = ctx;
            if (!ctx->profiling) {
                TRY(child_of(ctx, 0, &c8));
                TRY(child_of(ctx, 1, &c9));
                TRY(aux_init(ctx));
                CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
                CK(cudaStreamWaitEvent(c8->stream, ctx->ev_fork, 0));
                CK(cudaStreamWaitEvent(c9->stream, ctx->ev_fork, 0));
            }
            TRY(hoh_layer_encode_batch(c8, p8[c], nt * per8, tw, th, 8, mode, flags, nuke[c], g.plane_stride, per8, out8[c],
                                       nt * out8_tile[c], r8[c], nullptr, 0, nullptr));
            TRY(hoh_layer_encode_batch(c9, p9[c], nt * 2, tw, th, 9, mode, flags, nuke[c], g.plane_stride, 2, out9[c],
                                       nt * out9_tile[c], r9[c], nullptr, 0, nullptr));
            if (c8 != ctx) {
                CK(cudaEventRecord(ctx->ev_join[0], c8->stream));
                CK(cudaEventRecord(ctx->ev_join[1], c9->stream));
                CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[0], 0));
                CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[1], 0));
            }
            k_tile_decide<<<blocks_for(nt, 128), 128, 0, ctx->stream>>>(nt, sel, img0, per8, r8[c], r9[c], lz_size, lz_status,
                                                                        info, d_tiles);
            LAUNCHED("k_tile_decide");
        }
        // offsets in tile order over the chunk's images, then every shape emits its tiles
        k_tile_scan<<<1, 1024, 0, ctx->stream>>>(d_tiles, img0 * g.tiles_per_image, (uint32_t)(ni * g.tiles_per_image),
                                                 d_tile_off);
        LAUNCHED("k_tile_scan");
        for (int c = 0; c < n_cls; c++) {
            const size_t nt = ni * cls[c].sel.per_image;
            k_tile_emit<<<(unsigned)nt, 256, 0, ctx->stream>>>(cls[c].sel, img0, per8, r8[c], r9[c], out8[c], out9[c], lz[c],
                                                              (uint32_t)lz_stride[c], d_tiles, d_packed, packed_cap);
            LAUNCHED("k_tile_emit");
        }
    }
    return HOH_OK;
}

// -------------------------------------------------------------------------------------------------
// tile decoder, any cruncher mode (inverse of hoh_encode_images)
// -------------------------------------------------------------------------------------------------
} // extern "C" (reopened below)
namespace {
// Scratch of the tile decoder's phases for up to `ct` tiles of one shape per pass (hoh_decode_images: every tile of a
// chunk's images; hoh_decode_regions: the slots of one shape).
struct DecScratch {
    uint32_t max_cells, max_side;
    size_t per_tile;  // scratch bytes per tile in a pass
    DTile* tiles;
    DPlane* planes;
    uint16_t *lz_sym, *idx_sym, *resid, *out, *backref, *maps, *top;
    uint8_t* bp;
    int32_t* pstatus;
    hoh_dec_stream* streams;
    hoh_dec_result *res_a, *res_b;
};
int dec_sizes(const hoh_tile_geometry& hg, const TileGeom& g, DecScratch* d) {
    d->max_cells = (((uint32_t)hg.tile_w + 39) / 40) * (((uint32_t)hg.tile_h + 39) / 40);
    if ((hg.tile_w + 39) / 40 > 256 || (hg.tile_h + 39) / 40 > 256) return HOH_E_UNSUPPORTED;
    d->max_side = lz_side_stride((size_t)hg.tile_w * hg.tile_h);
    d->per_tile = 4 * (size_t)d->max_side * 2 + 3 * (size_t)g.plane_stride * 2 * 2 + (size_t)g.plane_stride * 2 +
                  3 * (size_t)(kCumRow * 4 + kFreqRow * 4) + 3 * (size_t)hg.tile_w * 3 + 4096;
    return HOH_OK;
}
int dec_scratch(hoh_ctx* ctx, const hoh_tile_geometry& hg, const TileGeom& g, size_t ct, DecScratch* d) {
    const uint32_t max_cells_pad = (d->max_cells + 7u) & ~7u;
    TRY(scratch_t(ctx, S_D_TILES, ct, &d->tiles));
    TRY(scratch_t(ctx, S_D_PLANES, ct * 3, &d->planes));
    TRY(scratch_t(ctx, S_D_LZSYM, ct * 4 * d->max_side, &d->lz_sym));
    TRY(scratch_t(ctx, S_D_IDXSYM, ct * 3 * max_cells_pad, &d->idx_sym));
    TRY(scratch_t(ctx, S_D_RESID, ct * 3 * g.plane_stride, &d->resid));
    TRY(scratch_t(ctx, S_D_OUT, ct * 3 * g.plane_stride, &d->out));
    TRY(scratch_t(ctx, S_D_BACKREF, ct * g.plane_stride, &d->backref));
    TRY(scratch_t(ctx, S_D_MAPS, ct * 3 * d->max_cells, &d->maps));
    TRY(scratch_t(ctx, S_D_STREAMS, ct * 3, &d->streams));
    TRY(scratch_t(ctx, S_D_RES_A, ct * 3, &d->res_a));
    TRY(scratch_t(ctx, S_D_RES_B, ct * 3, &d->res_b));
    TRY(scratch_t(ctx, S_D_TOP, ct * 3 * (size_t)hg.tile_w, &d->top));
    TRY(scratch_t(ctx, S_D_BP, ct * 3 * (size_t)hg.tile_w, &d->bp));
    TRY(scratch_t(ctx, S_D_PSTATUS, ct * 3, &d->pstatus));
    return HOH_OK;
}
// One pass of the tile decoder over nt tiles of shape tw x th (choh.cpp:459-474).  begin() launches the phase that
// fills d.tiles / d.streams for local tiles 0 .. nt-1, store() the one that writes their pixels out; the phases in
// between only see local tile numbers.
template <class Begin, class Store>
int decode_pass(hoh_ctx* ctx, const DecScratch& d, size_t nt, int tw, int th, uint32_t plane_stride,
                const uint8_t* d_packed, size_t packed_bytes, Begin begin, Store store) {
    const uint32_t npx = (uint32_t)tw * th;
    const uint32_t xt = (tw + 39) / 40, yt = (th + 39) / 40, cells = xt * yt, cells_pad = (cells + 7u) & ~7u;
    const uint32_t side = lz_side_stride(npx);
    TRY(begin(side));
    for (uint32_t k = 0; k < 4; k++) {  // un_lz.hpp:100-145: the side streams follow one another
        TRY(decode_common(ctx, d.streams, nt, d_packed, packed_bytes, d.lz_sym, d.res_a));
        k_dt_lz_next<<<blocks_for(nt, 128), 128, 0, ctx->stream>>>(nt, k, d_packed, packed_bytes, d.res_a, side, d.tiles,
                                                                   d.streams);
        LAUNCHED("k_dt_lz_next");
    }
    k_dt_channels<<<blocks_for(nt, 128), 128, 0, ctx->stream>>>(nt, d_packed, packed_bytes, xt, yt, cells_pad, d.tiles,
                                                                d.planes, d.streams);
    LAUNCHED("k_dt_channels");
    TRY(decode_common(ctx, d.streams, nt * 3, d_packed, packed_bytes, d.idx_sym, d.res_a));
    k_dt_main<<<blocks_for(nt * 3, 128), 128, 0, ctx->stream>>>(nt * 3, cells, cells_pad, plane_stride, npx, d.res_a,
                                                                d.idx_sym, d.planes, d.maps, d.streams);
    LAUNCHED("k_dt_main");
    TRY(decode_common(ctx, d.streams, nt * 3, d_packed, packed_bytes, d.resid, d.res_b));
    k_dt_unlz<<<blocks_for(nt * 32, 128), 128, 0, ctx->stream>>>(nt, npx, plane_stride, d.lz_sym, side, d.tiles, d.backref);
    LAUNCHED("k_dt_unlz");
    // One thread per plane with its inputs prefetched in 8-pixel groups (tile widths that are multiples of
    // 8: 17 ms for 5 760 planes of 256x270, 37 ms for 46 080).  Other widths take the scalar walk, whose
    // loads sit on the pixel chain: there a half-warp per predictor-grid plane is faster while the launch is
    // bound by the length of one plane's walk (37 vs 55 ms for 5 760 planes; crossover near 20 000).
    const bool grouped = tw % 8 == 0 && tw >= 16 && plane_stride % 8 == 0;  // k_dt_unpredict's prefetched walk
    const bool wide_walk = !grouped && nt * 3 <= 16384;
    k_dt_unpredict<<<blocks_for(nt * 3, 64), 64, 0, ctx->stream>>>(nt * 3, tw, th, (int)xt, (int)yt, plane_stride,
                                                                   d.planes, d.tiles, d.res_b, d.resid, d.maps, d.backref,
                                                                   d.out, d.top, d.bp, d.pstatus, wide_walk ? 1u : 0u);
    LAUNCHED("k_dt_unpredict");
    if (wide_walk) {
        k_dt_unpredict16<<<blocks_for(nt * 3, kUp16Planes), kUp16Planes * 16,
                           (size_t)kUp16Planes * ((tw + 1) & ~1) * 3, ctx->stream>>>(
            nt * 3, tw, th, (int)xt, (int)yt, plane_stride, d.planes, d.tiles, d.res_b, d.resid, d.maps, d.backref, d.out,
            d.pstatus);
        LAUNCHED("k_dt_unpredict16");
    }
    return store();
}

// Slots per tile shape of a region decode (RoiPlan, hoh_kernels.cuh) and the shapes' sub-grids.
// Bound: a window covers pixel columns wx .. wx + crop_w - 1, and column x lies in tile column floor(x / tile_w).  For
// integers a, b >= 0, floor((a + b) / t) - floor(a / t) <= ceil(b / t), so the window touches at most
// ceil((crop_w - 1) / tile_w) + 1 = (crop_w + tile_w - 2) / tile_w + 1 tile columns, and no more than the x_count
// columns of a shape's sub-grid; the same holds for rows.  k_roi_select asserts it.
RoiPlan roi_plan(const TileGeom& g, const TileClass* cls, int n_cls, uint32_t crop_w, uint32_t crop_h) {
    RoiPlan p;
    memset(&p, 0, sizeof(p));
    p.g = g;
    p.crop_w = crop_w;
    p.crop_h = crop_h;
    p.n_cls = (uint32_t)n_cls;
    const uint32_t span_x = (crop_w + g.tile_w - 2) / g.tile_w + 1, span_y = (crop_h + g.tile_h - 2) / g.tile_h + 1;
    for (int c = 0; c < n_cls; c++) {
        const TileSel& s = cls[c].sel;
        p.x_first[c] = s.x_first;
        p.x_count[c] = s.x_count;
        p.y_first[c] = s.y_first;
        p.y_count[c] = s.y_count;
        p.cols[c] = std::min(s.x_count, span_x);
        p.rows[c] = std::min(s.y_count, span_y);
        p.first[c] = p.per_image;
        p.per_image += p.cols[c] * p.rows[c];
    }
    return p;
}
}  // namespace
extern "C" {

int hoh_decode_images(hoh_ctx* ctx, const uint8_t* d_packed, size_t packed_bytes, const uint64_t* d_tile_off,
                      size_t n_images, uint32_t width, uint32_t height, uint8_t* d_rgb, int32_t* d_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_packed || !d_tile_off || !d_rgb || !d_status) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    if (packed_bytes < 32) return HOH_E_ARG;  // input contract (hohgpu.h)
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const TileGeom g = to_geom(hg);
    TileClass cls[4];
    const int n_cls = tile_classes(g, cls);
    DecScratch d;
    TRY(dec_sizes(hg, g, &d));
    TRY(new_shape(ctx, ((uint64_t)width << 40) ^ ((uint64_t)height << 16) ^ 2u, ctx->dec_key));
    const size_t budget = scratch_budget(ctx);
    size_t images_per_chunk = budget / (d.per_tile * g.tiles_per_image);
    if (images_per_chunk == 0) images_per_chunk = 1;
    if (images_per_chunk > n_images) images_per_chunk = n_images;
    // upper bound for any one shape's tiles in a chunk
    TRY(dec_scratch(ctx, hg, g, images_per_chunk * g.tiles_per_image, &d));
    for (size_t img0 = 0; img0 < n_images; img0 += images_per_chunk) {
        const size_t ni = std::min(images_per_chunk, n_images - img0);
        for (int c = 0; c < n_cls; c++) {  // one pass per tile shape (choh.cpp:459-474)
            const TileSel& sel = cls[c].sel;
            const size_t nt = ni * sel.per_image;
            TRY(decode_pass(
                ctx, d, nt, cls[c].tw, cls[c].th, g.plane_stride, d_packed, packed_bytes,
                [&](uint32_t side) {
                    k_dt_begin<<<blocks_for(nt, 128), 128, 0, ctx->stream>>>(nt, sel, img0, d_packed, packed_bytes,
                                                                             d_tile_off, side, d.tiles, d.streams);
                    LAUNCHED("k_dt_begin");
                    return HOH_OK;
                },
                [&]() {
                    k_dt_store<<<(unsigned)nt, 256, 0, ctx->stream>>>(sel, img0, g.plane_stride, d.tiles, d.pstatus, d.out,
                                                                      d_rgb, d_status);
                    LAUNCHED("k_dt_store");
                    return HOH_OK;
                }));
        }
    }
    return HOH_OK;
}

// -------------------------------------------------------------------------------------------------
// region decoder: the tiles of each image's window only
// -------------------------------------------------------------------------------------------------
int hoh_decode_regions(hoh_ctx* ctx, const uint8_t* d_packed, size_t packed_bytes, const uint64_t* d_tile_off,
                       size_t n_images, uint32_t width, uint32_t height, const uint32_t* d_origin,
                       uint32_t crop_w, uint32_t crop_h, uint8_t* d_crops, int32_t* d_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !d_packed || !d_tile_off || !d_origin || !d_crops || !d_status) return HOH_E_ARG;
    if (crop_w == 0 || crop_h == 0 || crop_w > width || crop_h > height) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    if (packed_bytes < 32) return HOH_E_ARG;  // input contract (hohgpu.h)
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const TileGeom g = to_geom(hg);
    TileClass cls[4];
    const int n_cls = tile_classes(g, cls);
    const RoiPlan plan = roi_plan(g, cls, n_cls, crop_w, crop_h);
    DecScratch d;
    TRY(dec_sizes(hg, g, &d));
    TRY(new_shape(ctx, ((uint64_t)width << 40) ^ ((uint64_t)height << 16) ^ ((uint64_t)crop_w << 28) ^
                           ((uint64_t)crop_h << 4) ^ 3u,
                  ctx->roi_key));
    const size_t budget = scratch_budget(ctx);
    size_t images_per_chunk = budget / (d.per_tile * plan.per_image + 8 * plan.per_image);
    if (images_per_chunk == 0) images_per_chunk = 1;
    if (images_per_chunk > n_images) images_per_chunk = n_images;
    uint32_t max_cls = 0;  // slots of the largest shape: one pass's tiles per image
    for (int c = 0; c < n_cls; c++) max_cls = std::max(max_cls, plan.cols[c] * plan.rows[c]);
    TRY(dec_scratch(ctx, hg, g, images_per_chunk * max_cls, &d));
    uint32_t* slots;
    int32_t* slot_status;
    TRY(scratch_t(ctx, S_R_SLOTS, images_per_chunk * plan.per_image, &slots));
    TRY(scratch_t(ctx, S_R_STATUS, images_per_chunk * plan.per_image, &slot_status));
    for (size_t img0 = 0; img0 < n_images; img0 += images_per_chunk) {
        const size_t ni = std::min(images_per_chunk, n_images - img0);
        k_roi_select<<<blocks_for(ni, 128), 128, 0, ctx->stream>>>(ni, img0, d_origin, plan, slots);
        LAUNCHED("k_roi_select");
        for (int c = 0; c < n_cls; c++) {
            const uint32_t cls_slots = plan.cols[c] * plan.rows[c], first = plan.first[c];
            const size_t nt = ni * cls_slots;
            TRY(decode_pass(
                ctx, d, nt, cls[c].tw, cls[c].th, g.plane_stride, d_packed, packed_bytes,
                [&](uint32_t side) {
                    k_dt_begin_roi<<<blocks_for(nt, 128), 128, 0, ctx->stream>>>(
                        nt, cls_slots, first, plan.per_image, g.tiles_per_image, img0, d_packed, packed_bytes, d_tile_off,
                        side, slots, d.tiles, d.streams);
                    LAUNCHED("k_dt_begin_roi");
                    return HOH_OK;
                },
                [&]() {
                    k_dt_store_window<<<(unsigned)nt, 256, 0, ctx->stream>>>(cls_slots, first, img0, plan, g.plane_stride,
                                                                             d_origin, slots, d.tiles, d.pstatus, d.out,
                                                                             d_crops, slot_status);
                    LAUNCHED("k_dt_store_window");
                    return HOH_OK;
                }));
        }
        k_roi_fold<<<blocks_for(ni, 128), 128, 0, ctx->stream>>>(ni, img0, plan, slots, slot_status, d_status);
        LAUNCHED("k_roi_fold");
    }
    return HOH_OK;
}

// -------------------------------------------------------------------------------------------------
// host-buffer forms of the two whole-tile calls (what tools/choh_batch.cpp / dhoh_batch.cpp call)
// -------------------------------------------------------------------------------------------------
} // extern "C" (reopened below)
namespace {
// Chunk boundaries (image indices) of a whole-tile host call.  The mode >= 1 kernels (rANS candidates, the plane walks of
// the decoder) last as long as ONE stream's serial chain however few streams a launch holds, so cutting a batch into k
// chunks multiplies their time by almost k (BASELINE config 3, decode: 112 ms for 256 frames at once, 4 x ~100 ms in four
// chunks) while the copies it would hide are short (6.4 GB at 55 GB/s = 116 ms).  Two chunks: the second one's H2D and
// the first one's D2H overlap the kernels, and the chain is paid twice, not four times; one chunk when the batch is
// small.  The double-buffered staging (raw + packed, twice) must leave most of the device to the codec's own scratch.
// floor_bytes: the smallest chunk, in bytes of pixels.
std::vector<size_t> tile_chunk_plan(size_t n_images, size_t raw_per_image, size_t floor_bytes = (size_t)256 << 20) {
    size_t per = (n_images + 1) / 2;
    const size_t min_per = floor_bytes / (raw_per_image ? raw_per_image : 1) + 1;
    if (per < min_per) per = min_per;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
        const size_t cap = free_b / 4 / (raw_per_image * 5 + 1);  // 2 x (raw + 1.5 raw packed) within a quarter of what is free
        if (cap >= 1 && per > cap) per = cap;
    }
    if (per > n_images) per = n_images;
    if (per == 0) per = 1;
    std::vector<size_t> bounds{0};
    while (bounds.back() < n_images) bounds.push_back(std::min(bounds.back() + per, n_images));
    return bounds;
}
}  // namespace
extern "C" {

int hoh_encode_images_host(hoh_ctx* ctx, const uint8_t* rgb_host, size_t n_images, uint32_t width, uint32_t height,
                           int mode, unsigned flags, uint8_t* packed_host, size_t packed_cap, uint64_t* tile_off_host,
                           hoh_tile_result* tiles_host) {
    DeviceGuard guard_(ctx);
    if (!ctx || !rgb_host || !packed_host || !tile_off_host || !tiles_host || mode < 0 || mode > 4) return HOH_E_ARG;
    tile_off_host[0] = 0;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const size_t raw1 = (size_t)width * height * 3;
    Pipe pp(ctx, tile_chunk_plan(n_images, raw1), 2, raw1, hg.tiles_per_image, sizeof(hoh_tile_result));
    for (int b = 0; b < pp.depth; b++) {  // coded on ctx itself, staging out of new_shape's reach (hoh_ctx::child)
        pp.slot[b].run = ctx;
        TRY(child_of(ctx, 2 + b, &pp.slot[b].stage));
    }
    const size_t per = pp.max_chunk, dev_cap = per * raw1 + per * raw1 / 2 + 8192 * per * pp.units;
    std::vector<uint64_t> chunk_base(pp.chunks());
    TRY(pipe_encode(pp, dev_cap, rgb_host, packed_host, packed_cap, tile_off_host, tiles_host, chunk_base.data(),
                    [&](int b, size_t n_c) {
                        const PipeSlot& s = pp.slot[b];
                        return hoh_encode_images(ctx, s.rgb, n_c, width, height, mode, flags, s.packed, dev_cap, s.off,
                                                 static_cast<hoh_tile_result*>(s.rec));
                    }));
    for (size_t c = 0; c < pp.chunks(); c++)  // tile records carry chunk-relative offsets: rebase
        for (size_t t = pp.bounds[c] * pp.units; t < pp.bounds[c + 1] * pp.units; t++) tiles_host[t].start += chunk_base[c];
    return HOH_OK;
}

int hoh_decode_images_host(hoh_ctx* ctx, const uint8_t* packed_host, size_t packed_bytes, const uint64_t* tile_off_host,
                           size_t n_images, uint32_t width, uint32_t height, uint8_t* rgb_host, int32_t* status_host) {
    DeviceGuard guard_(ctx);
    if (!ctx || !packed_host || !tile_off_host || !rgb_host || !status_host) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const size_t raw1 = (size_t)width * height * 3;
    Pipe pp(ctx, tile_chunk_plan(n_images, raw1), 2, raw1, hg.tiles_per_image, sizeof(int32_t));
    for (int b = 0; b < pp.depth; b++) {  // decoded on ctx itself, staging out of new_shape's reach (hoh_ctx::child)
        pp.slot[b].run = ctx;
        TRY(child_of(ctx, 2 + b, &pp.slot[b].stage));
    }
    return pipe_decode(pp, packed_host, packed_bytes, tile_off_host, rgb_host, status_host,
                       [&](int b, size_t n_c, size_t padded) {
                           const PipeSlot& s = pp.slot[b];
                           // a tile that fails to decode leaves its pixels untouched: make "untouched" mean zero
                           CK(cudaMemsetAsync(s.rgb, 0, n_c * raw1, ctx->stream));
                           return hoh_decode_images(ctx, s.packed, padded, s.off, n_c, width, height, s.rgb,
                                                    static_cast<int32_t*>(s.rec));
                       });
}

} // extern "C" (reopened below)
namespace {
// pipe_decode's copy-in hook for hoh_decode_regions_host.  A run is one tile row of one image's window: tiles
// [a, b) of the offset table, contiguous in packed_host.  Only runs are staged, back to back; every tile of a run keeps
// its place in the run and every other tile gets an empty range at the current end of the staging, so the rebased table
// stays ascending.  The chunk's origins follow its payloads to the slot's device copy of them.
struct RegionIn {
    std::vector<std::vector<std::pair<size_t, size_t>>> runs;  // per image, ascending
    const uint32_t* origin_host;
    uint32_t* d_origin[kPipeDepth];
    // tile rows the window at (wx, wy) of image i touches; none for a window that does not lie inside the image
    RegionIn(const hoh_tile_geometry& hg, size_t n_images, const uint32_t* origin, uint32_t crop_w, uint32_t crop_h)
        : runs(n_images), origin_host(origin) {
        for (size_t i = 0; i < n_images; i++) {
            const uint64_t wx = origin[2 * i], wy = origin[2 * i + 1];
            if (wx + crop_w > hg.width || wy + crop_h > hg.height) continue;
            const size_t tx0 = wx / hg.tile_w, tx1 = (wx + crop_w - 1) / hg.tile_w;
            for (size_t ty = wy / hg.tile_h; ty <= (wy + crop_h - 1) / hg.tile_h; ty++) {
                const size_t row = i * hg.tiles_per_image + ty * hg.x_tiles;
                runs[i].emplace_back(row + tx0, row + tx1 + 1);
            }
        }
    }
    int bytes(const Pipe& pp, size_t c, const uint64_t* off_host, size_t packed_bytes, uint64_t* out) const {
        uint64_t sum = 0;
        for (size_t i = pp.bounds[c]; i < pp.bounds[c + 1]; i++)
            for (const auto& r : runs[i]) {
                for (size_t t = r.first; t < r.second; t++)
                    if (off_host[t + 1] < off_host[t]) return HOH_E_ARG;
                if (off_host[r.second] > packed_bytes) return HOH_E_ARG;
                sum += off_host[r.second] - off_host[r.first];
            }
        *out = sum;
        return HOH_OK;
    }
    void rebase(const Pipe& pp, size_t c, const uint64_t* off_host, uint64_t* h_off) const {
        const size_t u0 = pp.bounds[c] * pp.units, u1 = pp.bounds[c + 1] * pp.units;
        size_t u = u0;
        uint64_t at = 0;
        for (size_t i = pp.bounds[c]; i < pp.bounds[c + 1]; i++)
            for (const auto& r : runs[i]) {
                for (; u < r.first; u++) h_off[u - u0] = at;
                for (; u < r.second; u++) h_off[u - u0] = at + off_host[u] - off_host[r.first];
                at += off_host[r.second] - off_host[r.first];
            }
        for (; u <= u1; u++) h_off[u - u0] = at;
    }
    // one copy per run, straight from the caller's buffer (tools/bench_regions.py measures it against a host-side
    // gather into pinned staging followed by one copy)
    int copy(const Pipe& pp, size_t c, const uint8_t* packed_host, const uint64_t* off_host, uint64_t,
             uint8_t* dst) const {
        hoh_ctx* ctx = pp.ctx;
        uint64_t at = 0;
        for (size_t i = pp.bounds[c]; i < pp.bounds[c + 1]; i++)
            for (const auto& r : runs[i]) {
                const uint64_t len = off_host[r.second] - off_host[r.first];
                CK(cudaMemcpyAsync(dst + at, packed_host + off_host[r.first], len, cudaMemcpyHostToDevice, ctx->s_h2d));
                at += len;
            }
        const size_t n_c = pp.bounds[c + 1] - pp.bounds[c];
        CK(cudaMemcpyAsync(d_origin[c % pp.depth], origin_host + 2 * pp.bounds[c], n_c * 2 * sizeof(uint32_t),
                           cudaMemcpyHostToDevice, ctx->s_h2d));
        return HOH_OK;
    }
};
}  // namespace
extern "C" {

int hoh_decode_regions_host(hoh_ctx* ctx, const uint8_t* packed_host, size_t packed_bytes,
                            const uint64_t* tile_off_host, size_t n_images, uint32_t width, uint32_t height,
                            const uint32_t* origin_host, uint32_t crop_w, uint32_t crop_h,
                            uint8_t* crops_host, int32_t* status_host) {
    DeviceGuard guard_(ctx);
    if (!ctx || !packed_host || !tile_off_host || !origin_host || !crops_host || !status_host) return HOH_E_ARG;
    if (crop_w == 0 || crop_h == 0 || crop_w > width || crop_h > height) return HOH_E_ARG;
    if (n_images == 0) return HOH_OK;
    hoh_tile_geometry hg;
    TRY(hoh_tile_geometry_for(width, height, &hg));
    const TileGeom g = to_geom(hg);
    TileClass cls[4];
    const int n_cls = tile_classes(g, cls);
    const RoiPlan plan = roi_plan(g, cls, n_cls, crop_w, crop_h);
    size_t touched = 0;  // bytes of pixels of the tiles an image's slots decode: what a chunk is planned by
    for (int c = 0; c < n_cls; c++) touched += (size_t)plan.cols[c] * plan.rows[c] * cls[c].tw * cls[c].th * 3;
    // HOH_PIPE_CHUNK_KB lowers the floor (tests: two chunks of a small batch)
    const size_t floor_bytes = getenv("HOH_PIPE_CHUNK_KB") ? std::min(pipe_chunk_floor(), (size_t)256 << 20) : (size_t)256 << 20;
    const size_t crop1 = (size_t)crop_w * crop_h * 3;
    Pipe pp(ctx, tile_chunk_plan(n_images, touched, floor_bytes), 2, crop1, hg.tiles_per_image, sizeof(int32_t));
    pp.recs = 1;
    RegionIn in(hg, n_images, origin_host, crop_w, crop_h);
    for (int b = 0; b < pp.depth; b++) {  // decoded on ctx itself, staging out of new_shape's reach (hoh_ctx::child)
        pp.slot[b].run = ctx;
        TRY(child_of(ctx, 2 + b, &pp.slot[b].stage));
        TRY(scratch_t(pp.slot[b].stage, S_IO_E, pp.max_chunk * 2, &in.d_origin[b]));
    }
    return pipe_decode(
        pp, packed_host, packed_bytes, tile_off_host, crops_host, status_host,
        [&](int b, size_t n_c, size_t padded) {
            const PipeSlot& s = pp.slot[b];
            // a failing tile or a bad window leaves its pixels untouched: make "untouched" mean zero
            CK(cudaMemsetAsync(s.rgb, 0, n_c * crop1, ctx->stream));
            return hoh_decode_regions(ctx, s.packed, padded, s.off, n_c, width, height, in.d_origin[b], crop_w, crop_h,
                                      s.rgb, static_cast<int32_t*>(s.rec));
        },
        in);
}

// =================================================================================================
// compat shims (host pointers)
// =================================================================================================

int hoh_encode_entropy(hoh_ctx* ctx, const uint16_t* symbols, size_t n, size_t range, uint8_t* out, size_t out_cap,
                       uint32_t prob_bits, size_t* out_size, int* stream_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || (!symbols && n) || !out || !out_size) return HOH_E_ARG;
    if (range == 0 || range > HOH_MAX_RANGE || prob_bits == 0 || prob_bits > HOH_MAX_PROB_BITS || n > 0xfffffff0ull)
        return HOH_E_UNSUPPORTED;
    uint16_t* d_sym;
    TRY(stage_in(ctx, S_IO_A, symbols, n, &d_sym));
    hoh_enc_stream st;
    memset(&st, 0, sizeof st);
    st.n = (uint32_t)n;
    st.range = (uint32_t)range;
    st.prob_bits = prob_bits;
    st.out_cap = (uint32_t)hoh_enc_slab_bytes(n, prob_bits);
    hoh_enc_stream* d_st;
    TRY(stage_in(ctx, S_IO_B, &st, 1, &d_st));
    uint8_t* d_out;
    hoh_stream_result* d_res;
    TRY(scratch_t(ctx, S_IO_C, st.out_cap, &d_out));
    TRY(scratch_t(ctx, S_RESULTS, 1, &d_res));
    TRY(hoh_encode_entropy_batch(ctx, d_st, 1, d_sym, d_out, d_res, (uint32_t)range, prob_bits, (uint32_t)n));
    hoh_stream_result res;
    TRY(stage_out(ctx, &res, d_res, 1));
    if (stream_status) *stream_status = res.status;
    *out_size = 0;
    if (res.status != HOH_S_OK) return HOH_E_STREAM;
    if (res.size > out_cap) return HOH_E_CAPACITY;
    TRY(stage_out(ctx, out, d_out + res.start, res.size));
    *out_size = res.size;
    return HOH_OK;
}

int hoh_encode_entropy_8bit(hoh_ctx* ctx, const uint8_t* symbols, size_t n, size_t range, uint8_t* out,
                            size_t out_cap, uint32_t prob_bits, size_t* out_size, int* stream_status) {
    DeviceGuard guard_(ctx);
    // entropy_encoding.hpp:283-303 widens to u16 and calls the 16-bit form
    std::vector<uint16_t> wide(n);
    for (size_t i = 0; i < n; i++) wide[i] = symbols[i];
    return hoh_encode_entropy(ctx, wide.data(), n, range, out, out_cap, prob_bits, out_size, stream_status);
}

int hoh_decode_entropy(hoh_ctx* ctx, const uint8_t* in, size_t in_size, size_t* byte_pointer, uint16_t* symbols,
                       size_t symbols_cap, size_t* symbol_size, unsigned flags, int* stream_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !in || !byte_pointer || !symbol_size || (!symbols && symbols_cap)) return HOH_E_ARG;
    uint8_t* d_in;
    const size_t padded = (in_size + 47) & ~(size_t)15;
    TRY(scratch_t(ctx, S_IO_A, padded, &d_in));
    CK(cudaMemsetAsync(d_in + (in_size & ~(size_t)15), 0, padded - (in_size & ~(size_t)15), ctx->stream));
    CK(cudaMemcpyAsync(d_in, in, in_size, cudaMemcpyHostToDevice, ctx->stream));
    hoh_dec_stream st;
    memset(&st, 0, sizeof st);
    st.in_off = *byte_pointer;
    st.sym_cap = (uint32_t)(symbols_cap > 0xfffffff0ull ? 0xfffffff0ull : symbols_cap);
    st.flags = flags;
    hoh_dec_stream* d_st;
    TRY(stage_in(ctx, S_IO_B, &st, 1, &d_st));
    uint16_t* d_sym;
    hoh_dec_result* d_res;
    TRY(scratch_t(ctx, S_IO_C, symbols_cap + 64, &d_sym));
    TRY(scratch_t(ctx, S_DRESULTS, 1, &d_res));
    TRY(hoh_decode_entropy_batch(ctx, d_st, 1, d_in, padded, d_sym, d_res, (uint32_t)st.sym_cap));
    hoh_dec_result res;
    TRY(stage_out(ctx, &res, d_res, 1));
    if (stream_status) *stream_status = res.status;
    *symbol_size = res.n;
    *byte_pointer = res.end_off;
    size_t take = res.n < symbols_cap ? res.n : symbols_cap;
    if (res.status != HOH_S_OK && res.status != HOH_S_OVERFLOW && res.status != HOH_S_BAD_STATE) return HOH_E_STREAM;
    TRY(stage_out(ctx, symbols, d_sym, take));  // a stream that fails the final-state check still hands its symbols out
    return res.status == HOH_S_OK ? HOH_OK : res.status == HOH_S_OVERFLOW ? HOH_E_CAPACITY : HOH_E_STREAM;
}

int hoh_normalize_freqs(hoh_ctx* ctx, uint32_t* freqs, uint32_t* cum_freqs, size_t size, uint32_t target_total,
                        int* stream_status) {
    DeviceGuard guard_(ctx);
    if (!ctx || !freqs || !cum_freqs || size == 0) return HOH_E_ARG;
    if (size > HOH_MAX_RANGE) return HOH_E_UNSUPPORTED;
    uint32_t *d_f, *d_c;
    int32_t* d_s;
    TRY(stage_in(ctx, S_IO_A, freqs, size, &d_f));
    TRY(scratch_t(ctx, S_IO_B, size + 1, &d_c));
    TRY(scratch_t(ctx, S_IO_C, 1, &d_s));
    k_normalize_only<<<1, 32, 0, ctx->stream>>>(d_f, d_c, (uint32_t)size, target_total, d_s);
    LAUNCHED("k_normalize_only");
    int32_t st;
    TRY(stage_out(ctx, &st, d_s, 1));
    if (stream_status) *stream_status = st;
    if (st != HOH_S_OK) return HOH_E_STREAM;
    TRY(stage_out(ctx, freqs, d_f, size));
    TRY(stage_out(ctx, cum_freqs, d_c, size + 1));
    return HOH_OK;
}

int hoh_subtract_green(hoh_ctx* ctx, const uint8_t* rgb, size_t size, uint16_t* green, uint16_t* red_g,
                       uint16_t* blue_g) {
    DeviceGuard guard_(ctx);
    if (!ctx || !rgb || !green || !red_g || !blue_g) return HOH_E_ARG;
    const size_t px = size / 3;
    uint8_t* d_rgb;
    uint16_t* d_pl;
    TRY(stage_in(ctx, S_IO_A, rgb, px * 3, &d_rgb));
    TRY(scratch_t(ctx, S_IO_B, px * 3, &d_pl));
    TRY(hoh_subtract_green_dev(ctx, d_rgb, px, d_pl, d_pl + px, d_pl + 2 * px));
    TRY(stage_out(ctx, green, d_pl, px));
    TRY(stage_out(ctx, red_g, d_pl + px, px));
    TRY(stage_out(ctx, blue_g, d_pl + 2 * px, px));
    return HOH_OK;
}

int hoh_add_green(hoh_ctx* ctx, const uint16_t* green, const uint16_t* red_g, const uint16_t* blue_g, size_t pixels,
                  uint8_t* rgb) {
    DeviceGuard guard_(ctx);
    if (!ctx || !rgb || !green || !red_g || !blue_g) return HOH_E_ARG;
    uint16_t* d_pl;
    uint8_t* d_rgb;
    TRY(scratch_t(ctx, S_IO_B, pixels * 3, &d_pl));
    TRY(scratch_t(ctx, S_IO_A, pixels * 3, &d_rgb));
    CK(cudaMemcpyAsync(d_pl, green, pixels * 2, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_pl + pixels, red_g, pixels * 2, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_pl + 2 * pixels, blue_g, pixels * 2, cudaMemcpyHostToDevice, ctx->stream));
    TRY(hoh_add_green_dev(ctx, d_pl, d_pl + pixels, d_pl + 2 * pixels, pixels, d_rgb));
    TRY(stage_out(ctx, rgb, d_rgb, pixels * 3));
    return HOH_OK;
}

int hoh_channelpredict_fastpath(hoh_ctx* ctx, const uint16_t* data, int w, int h, int depth, uint16_t* out) {
    DeviceGuard guard_(ctx);
    if (!ctx || !data || !out || w <= 0 || h <= 0) return HOH_E_ARG;
    const size_t px = (size_t)w * h;
    uint16_t *d_in, *d_out;
    TRY(stage_in(ctx, S_IO_A, data, px, &d_in));
    TRY(scratch_t(ctx, S_IO_B, px, &d_out));
    TRY(hoh_predict_fastpath_dev(ctx, d_in, 1, w, h, depth, d_out));
    return stage_out(ctx, out, d_out, px);
}

int hoh_channelpredict_section(hoh_ctx* ctx, const uint16_t* data, int w, int h, int depth, int x_tiles, int y_tiles,
                               int x, int y, uint16_t predictor, uint16_t* out, size_t out_cap, size_t* out_count) {
    DeviceGuard guard_(ctx);
    if (!ctx || !data || !out || !out_count || w <= 0 || h <= 0 || x_tiles <= 0 || y_tiles <= 0 || x < 0 || y < 0 ||
        x >= x_tiles || y >= y_tiles)
        return HOH_E_ARG;
    const size_t px = (size_t)w * h;
    const int tw = (w + x_tiles - 1) / x_tiles, th = (h + y_tiles - 1) / y_tiles;
    const uint32_t cell_cap = (uint32_t)tw * th;
    const size_t cells = (size_t)x_tiles * y_tiles;
    uint16_t *d_in, *d_mask, *d_res;
    uint32_t* d_cnt;
    TRY(stage_in(ctx, S_IO_A, data, px, &d_in));
    TRY(stage_in(ctx, S_IO_B, &predictor, 1, &d_mask));
    TRY(scratch_t(ctx, S_IO_C, cells * cell_cap, &d_res));
    TRY(scratch_t(ctx, S_IO_D, cells, &d_cnt));
    TRY(hoh_predict_section_dev(ctx, d_in, 1, w, h, depth, x_tiles, y_tiles, d_mask, 1, d_res, cell_cap, d_cnt));
    const size_t cell = (size_t)y * x_tiles + x;
    uint32_t cnt;
    TRY(stage_out(ctx, &cnt, d_cnt + cell, 1));
    *out_count = cnt;
    if (cnt > out_cap) return HOH_E_CAPACITY;
    return stage_out(ctx, out, d_res + cell * cell_cap, cnt);
}

int hoh_channelpredict_all(hoh_ctx* ctx, const uint16_t* data, int w, int h, int depth, int x_tiles, int y_tiles,
                           const uint16_t* tile_map, uint16_t* out) {
    DeviceGuard guard_(ctx);
    if (!ctx || !data || !out || !tile_map || w <= 0 || h <= 0 || x_tiles <= 0 || y_tiles <= 0) return HOH_E_ARG;
    const size_t px = (size_t)w * h;
    uint16_t *d_in, *d_map, *d_out;
    TRY(stage_in(ctx, S_IO_A, data, px, &d_in));
    TRY(stage_in(ctx, S_IO_B, tile_map, (size_t)x_tiles * y_tiles, &d_map));
    TRY(scratch_t(ctx, S_IO_C, px, &d_out));
    TRY(hoh_predict_all_dev(ctx, d_in, 1, w, h, depth, x_tiles, y_tiles, d_map, d_out));
    return stage_out(ctx, out, d_out, px);
}

int hoh_unpredict_all(hoh_ctx* ctx, const uint16_t* resid, size_t n_resid, int w, int h, int depth, int x_tiles,
                      int y_tiles, const uint16_t* tile_map, const uint16_t* backref, uint16_t* out) {
    DeviceGuard guard_(ctx);
    if (!ctx || !resid || !out || !tile_map || w <= 0 || h <= 0 || x_tiles <= 0 || y_tiles <= 0) return HOH_E_ARG;
    const size_t px = (size_t)w * h;
    if (n_resid > px) n_resid = px;
    uint16_t *d_in, *d_map, *d_out, *d_br = nullptr;
    TRY(scratch_t(ctx, S_IO_A, px, &d_in));
    CK(cudaMemsetAsync(d_in, 0, px * 2, ctx->stream));
    CK(cudaMemcpyAsync(d_in, resid, n_resid * 2, cudaMemcpyHostToDevice, ctx->stream));
    TRY(stage_in(ctx, S_IO_B, tile_map, (size_t)x_tiles * y_tiles, &d_map));
    TRY(scratch_t(ctx, S_IO_C, px, &d_out));
    if (backref) TRY(stage_in(ctx, S_IO_D, backref, px, &d_br));
    TRY(hoh_unpredict_all_dev(ctx, d_in, 1, w, h, depth, x_tiles, y_tiles, d_map, d_br, d_out));
    return stage_out(ctx, out, d_out, px);
}

int hoh_unpredict_fastpath(hoh_ctx* ctx, const uint16_t* resid, size_t n_resid, int w, int h, int depth,
                           const uint16_t* backref, uint16_t* out) {
    DeviceGuard guard_(ctx);
    if (!ctx || !resid || !out || w <= 0 || h <= 0) return HOH_E_ARG;
    const size_t px = (size_t)w * h;
    if (n_resid > px) n_resid = px;
    uint16_t *d_in, *d_out, *d_br = nullptr;
    TRY(scratch_t(ctx, S_IO_A, px, &d_in));
    CK(cudaMemsetAsync(d_in, 0, px * 2, ctx->stream));
    CK(cudaMemcpyAsync(d_in, resid, n_resid * 2, cudaMemcpyHostToDevice, ctx->stream));
    TRY(scratch_t(ctx, S_IO_C, px, &d_out));
    if (backref) TRY(stage_in(ctx, S_IO_D, backref, px, &d_br));
    TRY(hoh_unpredict_fastpath_dev(ctx, d_in, 1, w, h, depth, d_br, d_out));
    return stage_out(ctx, out, d_out, px);
}

int hoh_predictor_search(hoh_ctx* ctx, const uint16_t* plane, int w, int h, int depth, int mode, uint16_t* tile_map,
                         uint8_t* index_list, uint16_t* final_resid) {
    DeviceGuard guard_(ctx);
    if (!ctx || !plane || !tile_map || !index_list || w <= 0 || h <= 0) return HOH_E_ARG;
    const size_t px = (size_t)w * h;
    const size_t cells = (size_t)((w + 39) / 40) * ((h + 39) / 40);
    uint16_t *d_in, *d_map, *d_res;
    uint8_t* d_idx;
    TRY(stage_in(ctx, S_IO_A, plane, px, &d_in));
    TRY(scratch_t(ctx, S_IO_B, cells, &d_map));
    TRY(scratch_t(ctx, S_IO_C, px, &d_res));
    TRY(scratch_t(ctx, S_IO_D, cells, &d_idx));
    TRY(hoh_predictor_search_dev(ctx, d_in, 1, w, h, depth, mode, d_map, d_idx, d_res));
    TRY(stage_out(ctx, tile_map, d_map, cells));
    TRY(stage_out(ctx, index_list, d_idx, cells));
    if (final_resid) TRY(stage_out(ctx, final_resid, d_res, px));
    return HOH_OK;
}

int hoh_find_lz_rgb(hoh_ctx* ctx, const uint8_t* source, size_t size, int width, int height, uint8_t* lz_symbols,
                    size_t lz_cap, uint8_t* nukemap, int distance, int break_even_bonus, size_t* lz_size) {
    DeviceGuard guard_(ctx);
    if (!ctx || !source || !lz_symbols || !nukemap || !lz_size || width <= 0 || height <= 0) return HOH_E_ARG;
    const size_t npx = (size_t)width * height;
    if (size != npx * 3) return HOH_E_ARG;
    const size_t stride = hoh_find_lz_stride(width, height);
    uint8_t *d_rgb, *d_nuke, *d_lz;
    uint32_t* d_size;
    int32_t* d_bonus;
    TRY(stage_in(ctx, S_IO_A, source, size, &d_rgb));
    TRY(scratch_t(ctx, S_IO_B, npx, &d_nuke));
    TRY(scratch_t(ctx, S_IO_C, stride, &d_lz));
    TRY(scratch_t(ctx, S_IO_D, 2, &d_size));
    d_bonus = reinterpret_cast<int32_t*>(d_size + 1);
    CK(cudaMemcpyAsync(d_bonus, &break_even_bonus, sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    TRY(hoh_find_lz_rgb_batch(ctx, d_rgb, 1, width, height, distance, 0, d_bonus, d_nuke, d_lz, stride, d_size, nullptr));
    uint32_t n = 0;
    TRY(stage_out(ctx, &n, d_size, 1));
    if (n > lz_cap) return HOH_E_CAPACITY;
    TRY(stage_out(ctx, lz_symbols, d_lz, n));
    std::vector<uint8_t> nk(npx);
    TRY(stage_out(ctx, nk.data(), d_nuke, npx));
    for (size_t i = 0; i < npx; i++) nukemap[i] |= nk[i];
    *lz_size = n;
    return HOH_OK;
}

int hoh_channel_picker(hoh_ctx* ctx, const uint8_t* src, size_t size, int total, int target, uint16_t* out) {
    DeviceGuard guard_(ctx);
    if (!ctx || !src || !out || total <= 0 || size % (size_t)total) return HOH_E_ARG;
    uint8_t* d_in;
    uint16_t* d_out;
    TRY(stage_in(ctx, S_IO_A, src, size, &d_in));
    TRY(scratch_t(ctx, S_IO_B, size / total, &d_out));
    TRY(hoh_channel_picker_dev(ctx, d_in, size / total, total, target, d_out));
    return stage_out(ctx, out, d_out, size / total);
}

}  // extern "C"
