// hoh_kernels.cuh — sm_100a kernels of the hoh-ANS hot path (included once, by hoh_api.cu).
//
// Parallelisation (SURVEY.md section 7): the format gives every entropy stream ONE Rans64 state, so
// a stream is a serial chain and throughput comes from running one stream per warp lane over many
// independent streams (channel x tile x image).  Per-stream frequency tables live in shared memory
// laid out [symbol][lane] so that 32 lanes indexing 32 different tables never collide on a bank;
// symbols are moved between HBM and the lanes through a padded shared-memory transpose so that
// every global access is a coalesced row; renormalisation words go straight to / from each lane's
// own slab (L2 merges the sectors).  Prediction kernels are per-pixel data parallel on the encode
// side and an anti-diagonal wavefront (one row per lane, skewed by one column) on the decode side.
//
// Reference functions restated (file:line into the reference tree) are named at each kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cassert>
#include <type_traits>

#include "../../include/hohgpu.h"
#include "hoh_format.cuh"

namespace hohk {

constexpr int kFreqRow = 512;   // u32 per stream in the histogram / frequency scratch
constexpr int kCumRow = 520;    // u32 per stream in the cumulative-table scratch (range+1 used)
constexpr int kChunk = 64;      // symbols per lane between two shared-memory refills
static_assert(true, "");
constexpr int kGroup = 8;       // encoder: symbols whose lookups + reciprocals are hoisted ahead of the serial part
constexpr int kSymStride = 66;  // u16 per staged row (64 + 2 pad -> 33 words: conflict-free transpose)
constexpr uint64_t kRansL = 1ull << 31;  // rans64.hpp:59
constexpr int kDecChunk = 32;   // decoder: symbols per lane between two coalesced flushes
constexpr int kDecStride = 34;  // u16 per staged row (32 + 2 pad -> 17 words: conflict-free transpose)
constexpr uint32_t kSymBits = 9;  // dense decode table entry = cum << 9 | symbol (symbols < 512)
constexpr uint32_t kSymMask = (1u << kSymBits) - 1u;

// Per-stream scratch the encode pipeline threads through its kernels.
struct EncMeta {
    uint64_t payload_start;  // byte offset of the first payload word in the output buffer
    uint32_t payload_bytes;
    uint32_t head_len;     // varints + metadata + table
    uint32_t stored_size;  // entropy_encoding.hpp:45
    int32_t status;
    uint32_t table_u16;  // 1 if prob_bits <= 15 (every cumulative count fits a 16-bit lane)
    uint32_t win_lo;     // lowest symbol with a non-zero frequency
    uint32_t win_rows;   // (highest - lowest + 1) + 1: rows of cum[] the encoder needs for this stream
    uint32_t est;        // payload words known without coding: low 24 bits = lower bound, top 8 = upper - lower (255: unknown)
};

// Per-stream scratch of the decode pipeline.
struct DecMeta {
    uint64_t payload_off;  // byte offset of the rANS payload (or of the stored symbols)
    uint32_t n;
    uint32_t range;
    uint32_t prob_bits;
    uint32_t kind;  // 0 nothing to do, 1 stored, 2 rANS
    uint32_t maxbits;
    int32_t status;
    uint32_t used;  // symbols with non-zero frequency = rows of the dense decode table (+1 sentinel)
    uint32_t pad;
};

// Bounds-clamped byte view of the input buffer: malformed streams read zeros, never fault.
struct ByteView {
    const uint8_t* base;
    uint64_t size;
    __host__ __device__ __forceinline__ uint8_t operator[](uint64_t i) const { return i < size ? base[i] : (uint8_t)0; }
};

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
        if ((int)lane_id() >= d) v += o;
    }
    return v;
}

__device__ __forceinline__ uint32_t warp_min(uint32_t v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}

// =================================================================================================
// Symbol histogram — entropy_encoding.hpp:32-39.  One CTA per stream, shared-memory atomics.
// =================================================================================================
__global__ void __launch_bounds__(256) k_histogram(const hoh_enc_stream* __restrict__ streams,
                                                   const uint16_t* __restrict__ symbols,
                                                   uint32_t* __restrict__ freqs) {
    __shared__ uint32_t hist[kFreqRow];
    const hoh_enc_stream st = streams[blockIdx.x];
    for (int i = threadIdx.x; i < kFreqRow; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const uint16_t* src = symbols + st.sym_off;
    for (uint32_t i = threadIdx.x; i < st.n; i += blockDim.x) {
        uint32_t s = src[i];
        if (s < st.range) atomicAdd(&hist[s], 1u);
    }
    __syncthreads();
    uint32_t* dst = freqs + (size_t)blockIdx.x * kFreqRow;
    for (int i = threadIdx.x; i < kFreqRow; i += blockDim.x) dst[i] = hist[i];
}

// =================================================================================================
// Table build — stattools.hpp:6-70 (calc_cum_freqs, normalize_freqs) + entropy_encoding.hpp:43-203
// (header, clamp search, table serialisation).  One warp per stream.
// =================================================================================================
// Exclusive prefix sum of v[0..count) into out[0..count], each lane owning a contiguous run.
__device__ __forceinline__ void warp_cumsum(const uint32_t* v, uint32_t* out, uint32_t count) {
    const uint32_t lane = lane_id();
    const uint32_t per = (count + 31u) / 32u;
    const uint32_t lo = min(lane * per, count), hi = min(lo + per, count);
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += v[i];
    uint32_t run = warp_incl_scan(sum) - sum;
    for (uint32_t i = lo; i < hi; i++) {
        out[i] = run;
        run += v[i];
    }
    __syncwarp();
    // total = last exclusive + last value; computed by lane 0 to keep it simple and race free
    if (lane == 0) out[count] = count ? out[count - 1] + v[count - 1] : 0u;
    __syncwarp();
}

// Rescales raw counts `f` (range entries, in shared memory) to sum to 2^prob_bits with every used
// symbol kept non-zero — stattools.hpp:13-70.  `sc` is a second shared array.  On return f holds the
// normalised frequencies and cum[0..range] their prefix sums.  Returns HOH_S_*.
__device__ int warp_normalize(uint32_t* f, uint32_t* sc, uint32_t* cum, uint32_t range, uint32_t target) {
    const uint32_t lane = lane_id();
    if (target < range) return HOH_S_RANGE_GT_TOTAL;  // stattools.hpp:14
    warp_cumsum(f, cum, range);
    const uint32_t total = cum[range];
    __syncwarp();
    // stattools.hpp:20-24: cum[i] = target * cum[i] / total, then scaled freq = difference
    for (uint32_t i = lane; i < range; i += 32) {
        uint32_t a = (uint32_t)(((uint64_t)target * cum[i]) / total);
        uint32_t b = (uint32_t)(((uint64_t)target * cum[i + 1]) / total);
        sc[i] = b - a;
    }
    __syncwarp();
    // stattools.hpp:28-57: every used symbol that rounded to zero takes one count from the
    // lowest-index symbol of smallest frequency > 1, in ascending thief order.
    int status = HOH_S_OK;
    uint32_t thieves = 0, capacity = 0;
    for (uint32_t i = lane; i < range; i += 32) {
        thieves += (f[i] != 0 && sc[i] == 0) ? 1u : 0u;
        capacity += sc[i] > 1u ? sc[i] - 1u : 0u;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        thieves += __shfl_xor_sync(0xffffffffu, thieves, d);
        capacity += __shfl_xor_sync(0xffffffffu, capacity, d);
    }
    if (thieves > 16u) {
        // Many thieves (small prob_bits against a wide alphabet).  The order of the donors never changes: a steal
        // makes the current donor even smaller, so it stays the minimum until it is down to 1, and nobody else
        // moves.  Donors are therefore drained in ascending (frequency, index) order, each giving frequency - 1
        // counts, the last one partially — found by a binary search on that key instead of one search per thief.
        if (capacity < thieves) return HOH_S_NO_DONOR;  // stattools.hpp:42 fires at the first thief left without donor
        uint32_t lo = 0, hi = 1u << 30;  // largest key K with cap(K) = sum over donors with key < K of (freq - 1) <= thieves
        while (hi - lo > 1u) {
            const uint32_t mid = lo + (hi - lo) / 2u;
            uint32_t cap = 0;
            for (uint32_t j = lane; j < range; j += 32) {
                const uint32_t v = sc[j];
                cap += (v > 1u && ((v << 10) | j) < mid) ? v - 1u : 0u;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) cap += __shfl_xor_sync(0xffffffffu, cap, d);
            if (cap <= thieves) lo = mid;
            else hi = mid;
        }
        uint32_t cap = 0;
        for (uint32_t j = lane; j < range; j += 32) {
            const uint32_t v = sc[j];
            cap += (v > 1u && ((v << 10) | j) < lo) ? v - 1u : 0u;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) cap += __shfl_xor_sync(0xffffffffu, cap, d);
        const uint32_t rest = thieves - cap;  // taken from the donor whose key is exactly lo
        __syncwarp();
        for (uint32_t j = lane; j < range; j += 32) {
            const uint32_t v = sc[j];
            if (v > 1u) {
                const uint32_t key = (v << 10) | j;
                if (key < lo) sc[j] = 1;
                else if (key == lo) sc[j] = v - rest;
            } else if (f[j] != 0 && v == 0) {
                sc[j] = 1;
            }
        }
        __syncwarp();
    } else
    for (uint32_t base = 0; base < range; base += 32) {
        uint32_t i = base + lane;
        bool thief = i < range && f[i] != 0 && sc[i] == 0;
        uint32_t pending = __ballot_sync(0xffffffffu, thief);
        while (pending) {
            uint32_t who = base + (uint32_t)__ffs((int)pending) - 1u;
            pending &= pending - 1u;
            uint32_t key = 0xffffffffu;
            for (uint32_t j = lane; j < range; j += 32) {
                uint32_t v = sc[j];
                if (v > 1u) key = min(key, (v << 10) | j);
            }
            key = warp_min(key);
            if (key == 0xffffffffu) {
                status = HOH_S_NO_DONOR;  // stattools.hpp:42
                pending = 0;
                base = range;
                break;
            }
            if (lane == 0) {
                sc[key & 1023u]--;
                sc[who] = 1;
            }
            __syncwarp();
        }
    }
    if (status != HOH_S_OK) return status;
    for (uint32_t i = lane; i < range; i += 32) f[i] = sc[i];
    __syncwarp();
    warp_cumsum(f, cum, range);
    return HOH_S_OK;
}

// Warp-parallel form of hohfmt::build_head.  Lane 0 makes the (short, data-dependent) decisions —
// varints, clamp search, table mode — then every lane packs its contiguous run of frequencies: field
// widths are computed per symbol, their bit offsets come from a prefix sum (warp shuffles), and each
// field is OR-ed MSB-first into a zeroed big-endian word buffer with shared-memory atomics.  OR equals
// the reference packer's ADD as long as no field is wider than its width; a table with such a field
// (D6: table mode 1 with a frequency >= 2^maxbits, or one symbol owning all of 2^prob_bits) is detected
// with a ballot and handed to the bit-serial builder, which reproduces the reference's carries.
// `buf` = HOH_HEAD_CAP bytes of shared memory; on return it holds the head bytes in memory order.
__device__ __forceinline__ void bits_or(uint32_t* words, uint32_t bit, uint32_t value, uint32_t width) {
    if (width == 0u) return;
    const uint64_t win = (uint64_t)value << (64u - (bit & 31u) - width);  // width <= 19: fits
    const uint32_t k = bit >> 5;
    atomicOr(&words[k], (uint32_t)(win >> 32));
    if ((uint32_t)win) atomicOr(&words[k + 1u], (uint32_t)win);
}

// hohfmt::plan_head with the two clamp walks (entropy_encoding.hpp:53-122) done by the whole warp.  A walk visits
// the symbols from one end, its field width is the running maximum of the width each frequency needs on the ladder
// 0, 1, 4, 8, 12, ..., it stops at the first symbol whose running width reaches prob_bits, records where each rung
// was first needed and adds up the running widths: a prefix maximum.  Every lane owns a contiguous run of symbols:
// run maxima are combined by shuffles, each lane then walks its own run from the width it inherits.
// Results in scratch as warp_build_head expects: [0] = bytes of varints + metadata, [1] = table mode,
// [2] = stored-mode size, [3] = clamp count, [4 + j] = lo | hi << 16, [20 + k] = the head bytes.
__device__ __forceinline__ uint32_t ladder_need(uint32_t v) {  // smallest ladder width w with v < 2^w
    return v == 0u ? 0u : (v < 2u ? 1u : ((32u - (uint32_t)__clz((int)v) + 3u) & ~3u));
}
__device__ __forceinline__ uint32_t ladder_rung(uint32_t w) { return w == 0u ? 0u : (w == 1u ? 1u : w / 4u + 1u); }

__device__ void warp_plan_head(const uint32_t* f, uint32_t range, uint32_t n, uint32_t prob_bits, uint32_t* scratch,
                               uint32_t representable) {
    const uint32_t lane = lane_id();
    const uint32_t maxbits = hohfmt::bit_length(range - 1);
    const uint32_t count = (prob_bits - 1u) / 4u + 2u;  // :51
    const uint32_t per = (range + 31u) / 32u;
    const uint32_t lo = min(lane * per, range), hi = min(lo + per, range);
    uint32_t run_max = 0;
    bool wide = false;  // a frequency that does not fit a maxbits-wide field (table mode 1, D6)
    for (uint32_t i = lo; i < hi; i++) {
        run_max = max(run_max, ladder_need(f[i]));
        wide = wide || (f[i] >> maxbits) != 0u;
    }
    const bool any_wide = __any_sync(0xffffffffu, wide);
    // inclusive maxima over the lanes up to / from this one, then the widths a lane inherits
    uint32_t upto = run_max, from = run_max;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t b = __shfl_up_sync(0xffffffffu, upto, d), a = __shfl_down_sync(0xffffffffu, from, d);
        if ((int)lane >= d) upto = max(upto, b);
        if ((int)lane + d < 32) from = max(from, a);
    }
    uint32_t w_in_up = __shfl_up_sync(0xffffffffu, upto, 1), w_in_down = __shfl_down_sync(0xffffffffu, from, 1);
    if (lane == 0) w_in_up = 0;
    if (lane == 31) w_in_down = 0;
    const uint32_t w_all = __shfl_sync(0xffffffffu, from, 0);  // the running width after a walk over every symbol
    // pass 1: where does each walk stop, and the sum of the running widths before that
    uint64_t bits_up = 0, bits_down = 0;
    uint32_t stop_up = 0xffffffffu, stop_down = 0xffffffffu;
    {
        uint32_t w = w_in_up;
        for (uint32_t i = lo; i < hi; i++) {
            w = max(w, ladder_need(f[i]));
            if (w >= prob_bits) {
                stop_up = i;
                break;
            }
            bits_up += w;
        }
        w = w_in_down;
        for (uint32_t i = hi; i-- > lo;) {
            w = max(w, ladder_need(f[i]));
            if (w >= prob_bits) {
                stop_down = i;
                break;
            }
            bits_down += w;
        }
    }
    const uint32_t found_up = __ballot_sync(0xffffffffu, stop_up != 0xffffffffu);
    const uint32_t found_down = __ballot_sync(0xffffffffu, stop_down != 0xffffffffu);
    const int lane_up = found_up ? __ffs((int)found_up) - 1 : 32;          // the ascending walk visits lanes <= lane_up
    const int lane_down = found_down ? 31 - __clz((int)found_down) : -1;  // the descending walk visits lanes >= lane_down
    const bool seen_up = (int)lane <= lane_up, seen_down = (int)lane >= lane_down;
    uint64_t total = (seen_up ? bits_up : 0ull) + (seen_down ? bits_down : 0ull);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
    const uint32_t s_up = found_up ? __shfl_sync(0xffffffffu, stop_up, lane_up & 31) : range;       // :53-88 ends past the last symbol
    const uint32_t s_down = found_down ? __shfl_sync(0xffffffffu, stop_down, lane_down & 31) : 0u;  // :90-120 ends on symbol 0
    // pass 2: the marks — where each rung of the ladder was first needed — by the lanes the walks visited
    if (lane < 16) scratch[4 + lane] = (range - 1u) | (0u << 16);  // unused: lo = range - 1, hi = 0
    __syncwarp();
    if (seen_up) {
        uint32_t w = w_in_up;
        for (uint32_t i = lo; i < hi; i++) {
            const uint32_t need = ladder_need(f[i]);
            if (need > w) {
                for (uint32_t r = ladder_rung(w); r < ladder_rung(need) && r < count; r++)
                    atomicAnd(&scratch[4 + r], 0xffff0000u), atomicOr(&scratch[4 + r], i);
                w = need;
            }
            if (w >= prob_bits) break;
        }
    }
    if (seen_down) {
        uint32_t w = w_in_down;
        for (uint32_t i = hi; i-- > lo;) {
            const uint32_t need = ladder_need(f[i]);
            if (need > w) {
                for (uint32_t r = ladder_rung(w); r < ladder_rung(need) && r < count; r++)
                    atomicOr(&scratch[4 + r], i << 16);
                w = need;
            }
            if (w >= prob_bits) break;
        }
    }
    __syncwarp();
    if (lane == 0) {
        uint8_t tmp[8];
        uint32_t at = 0;
        at = hohfmt::put_varint(tmp, at, range - 1);
        at = hohfmt::put_varint(tmp, at, n);
        const uint32_t stored = at + 1 + (uint32_t)(((uint64_t)maxbits * n + 7) / 8);
        const uint64_t raw_table_bytes = ((uint64_t)prob_bits * range + 7) / 8;  // :47
        uint64_t clamped_bits = (uint64_t)((uint32_t)(2 * ((int)maxbits - 1)) * count) + 2ull * prob_bits;  // :48-49
        clamped_bits += total + (found_up ? prob_bits : 0u) + (found_down ? prob_bits : 0u);
        const uint32_t last_down = found_down ? prob_bits : w_all;
        clamped_bits += (uint64_t)last_down * ((uint64_t)s_down - (uint64_t)s_up - 1ull);  // :121, size_t arithmetic: wraps
        const uint64_t clamped_bytes = (clamped_bits + 7) / 8;
        uint32_t mode = raw_table_bytes < clamped_bytes ? 1u : 2u;  // :135 / :148
        if (representable && mode == 1u && any_wide) mode = 2u;
        tmp[at++] = (uint8_t)((1u << 7) + (prob_bits << 2) + mode);
        scratch[0] = at;
        scratch[1] = mode;
        scratch[2] = stored;
        scratch[3] = count;
        for (uint32_t k = 0; k < 8; k++) scratch[20 + k] = tmp[k];
    }
    __syncwarp();
}

__device__ uint32_t warp_build_head(const uint32_t* f, uint32_t range, uint32_t n, uint32_t prob_bits,
                                    uint8_t* buf, uint32_t* scratch /* >= 40 words */, uint32_t* stored_size,
                                    uint32_t representable = 0) {
    const uint32_t lane = lane_id();
    uint32_t* words = reinterpret_cast<uint32_t*>(buf);
    const uint32_t maxbits = hohfmt::bit_length(range - 1);
    // scratch: [0] = bytes of varints+metadata, [1] = mode, [2] = stored size, [3] = clamp count, [4..] = lo/hi
    warp_plan_head(f, range, n, prob_bits, scratch, representable);
    for (uint32_t k = lane; k < HOH_HEAD_CAP / 4; k += 32) words[k] = 0u;
    __syncwarp();
    const uint32_t at = scratch[0], mode = scratch[1], count = scratch[3];
    *stored_size = scratch[2];
    // field widths of this lane's run of symbols, and whether every value fits
    const uint32_t per = (range + 31u) / 32u;
    const uint32_t lo = min(lane * per, range), hi = min(lo + per, range);
    uint32_t my_bits = 0;
    bool fits = true;
    for (uint32_t i = lo; i < hi; i++) {
        uint32_t w;
        if (mode == 1u) {
            w = maxbits;
        } else {  // hohfmt::clamp_width_of
            w = 0;
            for (uint32_t j = 0; j < count; j++) {
                const uint32_t c = scratch[4 + j];
                if ((c & 0xffffu) <= i && (c >> 16) >= i) w = j == 0 ? 1u : 4u * j;
            }
            w = min(w, prob_bits);
        }
        fits = fits && (w >= 32u || f[i] < (1u << w));
        my_bits += w;
    }
    if (!__all_sync(0xffffffffu, fits)) {  // over-wide field somewhere: exact bit-serial path
        uint32_t len = 0;
        if (lane == 0) len = hohfmt::build_head(f, range, n, prob_bits, buf, stored_size);
        len = __shfl_sync(0xffffffffu, len, 0);
        *stored_size = __shfl_sync(0xffffffffu, *stored_size, 0);
        __syncwarp();
        return len;
    }
    const uint32_t pair_bits = mode == 2u ? 2u * count * maxbits : 0u;
    uint32_t bit = warp_incl_scan(my_bits) - my_bits + 8u * at + pair_bits;
    const uint32_t total_bits = __shfl_sync(0xffffffffu, bit + my_bits, 31);
    if (lane == 0) {
        for (uint32_t k = 0; k < at; k++) bits_or(words, 8u * k, scratch[20 + k], 8u);
        if (mode == 2u)
            for (uint32_t j = 0; j < count; j++) {
                const uint32_t c = scratch[4 + j];
                bits_or(words, 8u * at + 2u * j * maxbits, c & 0xffffu, maxbits);
                bits_or(words, 8u * at + (2u * j + 1u) * maxbits, c >> 16, maxbits);
            }
    }
    for (uint32_t i = lo; i < hi; i++) {
        uint32_t w;
        if (mode == 1u) {
            w = maxbits;
        } else {
            w = 0;
            for (uint32_t j = 0; j < count; j++) {
                const uint32_t c = scratch[4 + j];
                if ((c & 0xffffu) <= i && (c >> 16) >= i) w = j == 0 ? 1u : 4u * j;
            }
            w = min(w, prob_bits);
        }
        bits_or(words, bit, f[i], w);
        bit += w;
    }
    __syncwarp();
    // big-endian bit order -> bytes in memory order
    const uint32_t len = (total_bits + 7u) / 8u;
    for (uint32_t k = lane; k < (len + 3u) / 4u; k += 32) words[k] = __byte_perm(words[k], 0u, 0x0123);
    __syncwarp();
    return len;
}

constexpr int kTableWarps = 4;

// -------------------------------------------------------------------------------------------------
// How many 32-bit words the Rans64 coder will emit for a stream, from its histogram and its table alone.
// -------------------------------------------------------------------------------------------------
// The state starts at 2^31 (rans64.hpp:65) and ends in [2^31, 2^63); every step multiplies it by M / f (M = 2^prob_bits)
// up to a small relative error, every renormalisation (rans64.hpp:82-86) divides it by 2^32 up to a truncation.  With
// W emitted words:   log2(x_end) + 32 W = 31 + S + E,   S = sum over the symbols of (prob_bits - log2 f),
// hence W = floor((S + E) / 32) exactly.  E is bounded from the same data:
//   a step turns x = q f + r into q M + r + start = x M / f + d with |d| <= M - f, a relative error below f / x:
//     x >= 2^31 when the step did not renormalise      -> |e| <= 1.45 f / 2^31
//     x >= 2^(31 - prob_bits) f when it did (<= W steps) -> |e| <= 1.45 * 2^(prob_bits - 31)
//   a renormalisation drops the low word of an x >= 2^(63 - prob_bits) f: -1.45 * 2^(prob_bits - 31) <= e <= 0.
// So E lies in [-(B + 2 W k), B + W k] with B = 1.45 / 2^31 * sum(count f), k = 1.45 * 2^(prob_bits - 31): a fraction of a
// bit for 15-bit tables, a few bits at 19, and floor((S + E) / 32) is the same number at both ends of the interval
// for most streams.  layer_encode's candidates (layer_encode.hpp:334-392: the same residuals under six tables) are
// compared through these intervals, and only a candidate whose bytes or exact size the outcome needs is coded.
// k_finish_streams checks every coded stream against its interval (HOH_S_BAD_ESTIMATE).
// Returns EncMeta::est.  Warp-cooperative; `counts` = the raw histogram, `f` = the normalised frequencies.
__device__ __forceinline__ uint32_t warp_estimate_words(const uint32_t* __restrict__ counts, const uint32_t* f,
                                                        uint32_t range, uint32_t n, uint32_t bits) {
    const uint32_t lane = lane_id();
    double S = 0.0, B = 0.0;
    uint32_t seen = 0;
    for (uint32_t i = lane; i < range; i += 32) {
        const uint32_t c = counts[i];
        if (c != 0u) {
            const double fi = (double)f[i];
            S += (double)c * ((double)bits - log2(fi));
            B += (double)c * fi;
            seen += c;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        S += __shfl_xor_sync(0xffffffffu, S, d);
        B += __shfl_xor_sync(0xffffffffu, B, d);
        seen += __shfl_xor_sync(0xffffffffu, seen, d);
    }
    if (seen != n) return 0xff000000u;  // symbols outside the alphabet: the coder clamps them, the histogram skipped them
    B *= 1.45 / 2147483648.0;
    const double k = 1.45 * exp2((double)bits - 31.0);
    const double w_cap = floor((S + B + 1.0) / 32.0) + 1.0;
    const double slack = 1e-4 + 1e-12 * S;  // evaluation error of S (log2: 1 ulp, <= 512 terms)
    const double e_hi = B + w_cap * k + slack, e_lo = -(B + 2.0 * w_cap * k + slack);
    const double lo = fmax(0.0, floor((S + e_lo) / 32.0)), hi = floor((S + e_hi) / 32.0);
    if (hi - lo > 254.0 || hi >= 16777216.0) return 0xff000000u;
    return (uint32_t)lo | ((uint32_t)(hi - lo) << 24);
}
// What k_finish_streams will report as the stream's size if the coder emits `words` words (entropy_encoding.hpp:232-267).
__device__ __forceinline__ uint32_t stream_size_for(const hoh_enc_stream& st, const EncMeta& m, uint32_t words) {
    if (m.status != HOH_S_OK) return 0u;
    if (st.n == 0u) return st.prefix_len + m.head_len;
    const uint32_t payload = 4u * words + 8u;  // rans64.hpp:96-103: the flush writes the 64-bit state
    const uint32_t coded = m.head_len + hohfmt::varint_len(payload) + payload;
    return st.prefix_len + (m.stored_size < coded ? m.stored_size : coded);
}

__global__ void __launch_bounds__(kTableWarps * 32) k_build_tables(
    const hoh_enc_stream* __restrict__ streams, uint32_t n_streams, const uint32_t* __restrict__ freqs,
    uint32_t* __restrict__ cumtab, uint8_t* __restrict__ heads, EncMeta* __restrict__ meta) {
    __shared__ uint32_t s_f[kTableWarps][kFreqRow];
    __shared__ uint32_t s_sc[kTableWarps][kFreqRow];
    __shared__ uint32_t s_cum[kTableWarps][kFreqRow + 8];
    __shared__ __align__(16) uint8_t s_head[kTableWarps][HOH_HEAD_CAP];
    const uint32_t w = threadIdx.x >> 5, lane = lane_id();
    const uint32_t s = blockIdx.x * kTableWarps + w;
    if (s >= n_streams) return;
    const hoh_enc_stream st = streams[s];
    EncMeta m;
    m.payload_start = 0;
    m.payload_bytes = 0;
    m.head_len = 0;
    m.stored_size = 0;
    m.status = HOH_S_OK;
    m.table_u16 = st.prob_bits <= 15 ? 1u : 0u;
    m.win_lo = 0;
    m.win_rows = 0;
    m.est = 0xff000000u;
    uint8_t* head = heads + (size_t)s * HOH_HEAD_CAP;
    if (st.n == 0) {  // entropy_encoding.hpp:19-23: two varints and nothing else (D2)
        if (lane == 0) {
            uint32_t at = hohfmt::put_varint(s_head[w], 0, st.range - 1);
            at = hohfmt::put_varint(s_head[w], at, 0);
            for (uint32_t k = 0; k < at; k++) head[k] = s_head[w][k];
            m.head_len = at;
            meta[s] = m;
        }
        return;
    }
    uint32_t* f = s_f[w];
    uint32_t* sc = s_sc[w];
    uint32_t* cum = s_cum[w];
    const uint32_t* src = freqs + (size_t)s * kFreqRow;
    for (uint32_t i = lane; i < st.range; i += 32) f[i] = src[i];
    __syncwarp();
    int status = warp_normalize(f, sc, cum, st.range, 1u << st.prob_bits);
    if (status != HOH_S_OK) {
        if (lane == 0) {
            m.status = status;
            meta[s] = m;
        }
        return;
    }
    if ((st.reserved & HOH_FIX_LONE) && st.range > 1u) {
        // A stream with ONE distinct symbol gives it the whole 2^prob_bits, which the table format cannot
        // hold (the field is prob_bits wide: SURVEY D6) — no decoder can read such a stream back.  Decodable
        // variant: one count goes to a neighbouring symbol that never occurs.
        uint32_t lone = 0xffffffffu;
        for (uint32_t i = lane; i < st.range; i += 32)
            if (f[i] == (1u << st.prob_bits)) lone = i;
        lone = warp_min(lone);
        if (lone != 0xffffffffu) {
            if (lane == 0) {
                f[lone] -= 1u;
                f[lone + 1u < st.range ? lone + 1u : lone - 1u] = 1u;
            }
            __syncwarp();
            warp_cumsum(f, cum, st.range);
        }
    }
    uint32_t* ct = cumtab + (size_t)s * kCumRow;
    for (uint32_t i = lane; i <= st.range; i += 32) ct[i] = cum[i];
    {  // window of symbols that actually occur: the encoder stages only cum[win_lo .. win_lo + win_rows)
        uint32_t lo = 0xffffffffu, hi = 0u;
        for (uint32_t i = lane; i < st.range; i += 32)
            if (f[i] != 0u) {
                lo = min(lo, i);
                hi = max(hi, i);
            }
        lo = warp_min(lo);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, d));
        m.win_lo = lo;
        m.win_rows = hi - lo + 2u;
    }
    m.head_len = warp_build_head(f, st.range, st.n, st.prob_bits, s_head[w], sc, &m.stored_size, st.reserved & HOH_FIX_LONE);
    __syncwarp();
    m.est = warp_estimate_words(src, f, st.range, st.n, st.prob_bits);
    const uint32_t words = (m.head_len + 3u) / 4u;
    for (uint32_t k = lane; k < words; k += 32)
        reinterpret_cast<uint32_t*>(head)[k] = reinterpret_cast<const uint32_t*>(s_head[w])[k];
    if (lane == 0) meta[s] = m;
}

// =================================================================================================
// Rans64 core — rans64.hpp.  One state per lane.
// =================================================================================================
// rans64.hpp:262-278 (Rans64EncPutSymbol) == rans64.hpp:77-94 (Rans64EncPut) for every reachable
// state (SURVEY H2): x' = ((x / f) << bits) + x % f + start after the optional 32-bit renormalisation.
// The reference multiplies by a precomputed 64-bit reciprocal per symbol (24 B/symbol = 12 KB per
// stream — 32 per-lane tables of that size do not fit in shared memory).  Here the only per-symbol
// state in shared memory is the cumulative count.  A stream is one serial chain of steps, so what
// bounds the kernel is the LENGTH OF THE DEPENDENT CHAIN per symbol, not the instruction count:
// the reciprocal 1/f is computed in fp64 off the chain (it does not depend on x: MUFU.RCP64H + two
// Newton steps, biased low), and the chain itself is  u64 -> f64, one DFMA.RZ whose mantissa is the quotient
// (prob_bits >= 14; DMUL + f64 -> u64 below that), one IMAD for the remainder, one correction.  The estimate never exceeds the true quotient (operand truncated, the
// reciprocal biased by 2^-50, checked on the CPU over 2*10^8 cases) and is at most 1 short for
// prob_bits >= 14 (3 for 12..13), so the corrections below make the result exact for every input.

// 1/f biased low: inv <= (1/f)(1 - 2^-51), relative error < 2^-49.
__device__ __forceinline__ double recip_low(uint32_t f) {
    const double fd = (double)f;
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(fd));  // 20-bit seed
    double e = fma(-fd, r, 1.0);
    r = fma(r, e, r);
    e = fma(-fd, r, 1.0);
    r = fma(r, e, r);
    return r * 0.99999999999999911182;  // 1 - 2^-50
}

// One encoder step.  `words` is the stream's slab viewed as u32, `widx` the index of the lowest word
// written so far (words are emitted downwards).  The caller has checked the slab capacity up front
// (at most (n * bits + 32) / 32 + 3 words are ever written), so there is no per-symbol bounds test.
// A step with freq == 2^bits, start == 0 is an exact no-op (x / 2^bits, x mod 2^bits recombine to x and
// the renormalisation test x >= 2^63 never fires): lanes whose stream is shorter use it as padding.
// LOW_BITS: prob_bits below 14 may occur (the quotient estimate can then be short by more than one).
// `inv` = recip_low(freq) is passed in: it does not depend on the state, so callers compute it for a
// group of symbols ahead of the serial part (those computations overlap each other) and the serial
// part is only the short dependent chain.
// DIV selects how x / freq is taken:
//   0  prob_bits >= 14: the quotient is the mantissa of ONE fused multiply-add (below), short by at most 1
//   2  prob_bits >= 12: the same estimate, short by at most 3 (x / freq < 2^51 still fits the mantissa)
//   1  any prob_bits:   DMUL + F2I.U64.F64 (the conversion unit again, but such streams are short and few)
template <int DIV>
__device__ __forceinline__ uint64_t rans_put(uint64_t x, uint32_t start, uint32_t freq, double inv, uint32_t bits,
                                             uint32_t* __restrict__ words, uint32_t& widx) {
    // x >= ((L >> bits) << 32) * freq  <=>  (x >> (63 - bits)) >= freq, and 63 - bits >= 32
    const uint32_t xh = (uint32_t)(x >> 32), xl = (uint32_t)x;
    const bool emit = (xh >> (31u - bits)) >= freq;
    if (emit) words[--widx] = xl;
    // The state as a double (truncated), for BOTH outcomes of the renormalisation test, converted while the test is
    // still being evaluated: the select then picks a finished double and the test leaves the chain.  Same values as
    // converting the selected state, so the exactness argument below is untouched.  (Opaque to the compiler, which
    // otherwise branches around the 64-bit conversion.  Building the double on the FP64 pipe instead - two magic-number
    // additions, no conversion unit - was measured: 9.30 against 8.89 ms, the extra register moves cost more.)
    double d_full, d_hi;
    asm("cvt.rz.f64.u64 %0, %1;" : "=d"(d_full) : "l"(x));
    asm("cvt.rn.f64.u32 %0, %1;" : "=d"(d_hi) : "r"(xh));
    const double xd = emit ? d_hi : d_full;
    x = emit ? (uint64_t)xh : x;
    uint64_t q;  // q <= floor(x / freq), short by <= 1 (bits >= 14)
    if (DIV == 1) {
        q = __double2ull_rz(xd * inv);
    } else {
        // x / freq < 2^(63 - bits) <= 2^51: the product is added to 2^52 in the SAME fused operation, rounding
        // towards zero, so the mantissa of the sum IS floor(x_d * inv) — one DFMA instead of DMUL + F2I.U64.F64
        // (8 instead of 34 cycles on the chain).  Same bound as before (the product is not even rounded before
        // the floor); modelled on the CPU in tests/hostfmt (fmt_div_model) over the boundaries of every quotient.
        q = (uint64_t)__double_as_longlong(__fma_rz(xd, inv, 0x1p+52)) & 0x000fffffffffffffull;
    }
    uint32_t r = (uint32_t)x - (uint32_t)q * freq;           // true remainder < 2^32: exact mod 2^32
    if (r >= freq) {
        r -= freq;
        q++;
    }
    if (DIV != 0) {
        while (r >= freq) {
            r -= freq;
            q++;
        }
    }
    // r + start < 2^bits, so the sum cannot carry into the shifted quotient
    return (q << bits) | (uint64_t)(r + start);
}

// Words a stream of n symbols can emit at most, flush included, plus slack.
__device__ __host__ __forceinline__ uint64_t rans_words_bound(uint64_t n, uint32_t bits) {
    return (n * bits + 32u) / 32u + 4u;
}

// Table accessors.  PerLane: tab[(symbol * 32 + lane)] — 32 independent tables, bank == lane.
template <typename CumT>
struct PerLaneTable {
    const CumT* tab;
    uint32_t lane;
    __device__ __forceinline__ uint32_t cum(uint32_t s) const { return tab[s * 32u + lane]; }
};
// Shared: one table for every lane (static-table sweep).
template <typename CumT>
struct SharedTable {
    const CumT* tab;
    __device__ __forceinline__ uint32_t cum(uint32_t s) const { return tab[s]; }
};

// Cooperative, asynchronous load of one 64-symbol chunk for the 32 streams of a warp into the padded
// transpose: row r of `stage` receives symbols [64*chunk, 64*chunk+64) of stream r, zero-filled beyond
// its n.  cp.async (LDGSTS) writes shared memory directly, so the copy of the next chunk overlaps the
// coding of the current one; complete it with stage_wait().
__device__ __forceinline__ void cp_async4(uint32_t smem_addr, const void* gptr, uint32_t src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_addr), "l"(gptr), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void stage_wait() {
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();
}
template <int STRIDE = kSymStride>
__device__ __forceinline__ void stage_load_chunk(uint16_t* stage, const uint16_t* __restrict__ symbols,
                                                 const uint64_t* s_off, const uint32_t* s_n, uint32_t chunk) {
    const uint32_t lane = lane_id(), half = lane >> 4, q = lane & 15u;
    const uint32_t stage_addr = (uint32_t)__cvta_generic_to_shared(stage);
#pragma unroll 4
    for (uint32_t jj = 0; jj < 16; jj++) {
        const uint32_t r = 2u * jj + half;
        const uint32_t first = chunk * kChunk + 4u * q;
        const uint32_t n = s_n[r];
        const uint32_t left = n > first ? min(n - first, 4u) : 0u;  // symbols of this quad that exist
        // never form an address past the stream: clamp the source to its start when nothing is read
        const uint16_t* src = symbols + s_off[r] + (left ? first : 0u);
        const uint32_t dst = stage_addr + (r * (STRIDE / 2) + 2u * q) * 4u;
        cp_async4(dst, src, min(left, 2u) * 2u);
        cp_async4(dst + 4u, src + (left > 2u ? 2 : 0), left > 2u ? (left - 2u) * 2u : 0u);
    }
}

// The same chunk moved by the copy engine: when every stream of the warp has the whole chunk (all but the ragged last
// chunk of a stream), each lane issues ONE 128-byte cp.async.bulk for its own row (UBLKCP: source and destination
// 16-byte aligned, completion counted in bytes on an mbarrier) instead of the warp walking 16 x 2 four-byte LDGSTS with
// their address arithmetic (about 8.5 warp instructions per symbol of a ~67-instruction step).  Rows are 144 bytes
// apart (kBulkStride): 16-byte aligned for the copy engine, and a lane's 8 symbols of a group come out with one
// conflict-free LDS.128 (36 r mod 32 = 4 r: eight lanes x four words cover the 32 banks).
constexpr int kBulkStride = 72;  // u16 per staged row
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"((uint32_t)__cvta_generic_to_shared(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Decode side: rows of `stage` (32 symbols per stream, row stride kDecStride) -> global symbol arrays.
// Eight lanes cover one row with 8-byte stores, four rows per instruction.
__device__ __forceinline__ void stage_store_chunk(const uint16_t* stage, uint16_t* __restrict__ symbols,
                                                  const uint64_t* s_off, const uint32_t* s_n, uint32_t chunk) {
    const uint32_t lane = lane_id(), sub = lane >> 3, q = lane & 7u;
    const uint32_t* stage32 = reinterpret_cast<const uint32_t*>(stage);
#pragma unroll
    for (uint32_t jj = 0; jj < 8; jj++) {
        const uint32_t r = 4u * jj + sub;
        const uint32_t first = chunk * kDecChunk + 4u * q;
        const uint32_t n = s_n[r];
        const uint32_t a = stage32[r * (kDecStride / 2) + 2u * q];
        const uint32_t b = stage32[r * (kDecStride / 2) + 2u * q + 1u];
        if (first + 3u < n) {
            *reinterpret_cast<uint2*>(symbols + s_off[r] + first) = make_uint2(a, b);
        } else if (first < n) {
            uint16_t* p = symbols + s_off[r] + first;
            p[0] = (uint16_t)a;
            if (first + 1u < n) p[1] = (uint16_t)(a >> 16);
            if (first + 2u < n) p[2] = (uint16_t)b;
        }
    }
}

// One warp per CTA, one stream per lane.  Each lane's table holds only the window of symbols that occur
// in its stream (cum[win_lo .. win_lo + win_rows)); `rows_lo < need <= rows` selects the warps of this
// launch's table-size class (need = widest window among the warp's streams), one launch per class.
// Dynamic shared memory: rows * 32 CumT + 2 * 32 * kSymStride u16 (double-buffered symbol staging).
template <typename CumT, bool LOW_BITS>
__global__ void __launch_bounds__(32) k_rans_encode(const hoh_enc_stream* __restrict__ streams,
                                                    uint32_t n_streams, const uint16_t* __restrict__ symbols,
                                                    const uint32_t* __restrict__ cumtab, uint8_t* __restrict__ out,
                                                    EncMeta* __restrict__ meta, uint32_t rows_lo, uint32_t rows,
                                                    uint32_t want_u16) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    CumT* tab = reinterpret_cast<CumT*>(smem_raw);
    uint16_t* stage0 = reinterpret_cast<uint16_t*>(smem_raw + (size_t)rows * 32u * sizeof(CumT));
    __shared__ uint64_t s_off[32];
    __shared__ uint32_t s_n[32];
    __shared__ __align__(8) uint64_t s_bar[2];  // one per staging buffer: bytes of its bulk copies still in flight

    const uint32_t lane = lane_id();
    const uint32_t s = blockIdx.x * 32u + lane;
    const bool exists = s < n_streams;
    hoh_enc_stream st;
    EncMeta m;
    if (exists) {
        st = streams[s];
        m = meta[s];
    } else {
        st.n = 0;
        st.range = 1;
        st.prob_bits = 1;
        st.sym_off = 0;
        st.out_off = 0;
        st.out_cap = 0;
        m.status = HOH_S_OK;
        m.table_u16 = want_u16;
        m.win_lo = 0;
        m.win_rows = 0;
    }
    // a stream takes part if it has symbols, its table was built, and it belongs to this launch's
    // table width (16-bit lanes for prob_bits <= 15, 32-bit otherwise)
    bool live = exists && st.n > 0 && m.status == HOH_S_OK && m.table_u16 == want_u16;
    uint32_t need = live ? m.win_rows : 0u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) need = max(need, __shfl_xor_sync(0xffffffffu, need, d));
    if (need <= rows_lo || need > rows) return;  // another class's launch (or nothing to do)
    // ... and of the two instantiations the one that fits the warp: the short division chain (LOW_BITS = false) is
    // exact for prob_bits >= 14 only, so a warp with a narrower stream belongs to the LOW_BITS launch (the host issues
    // that launch only when such streams may exist)
    uint32_t low = live ? st.prob_bits : 32u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) low = min(low, __shfl_xor_sync(0xffffffffu, low, d));
    if ((low < 14u) != LOW_BITS) return;
    if (live && (uint64_t)st.out_cap < rans_words_bound(st.n, st.prob_bits) * 4u + HOH_HEAD_CAP + 32u) {
        m.status = HOH_S_OVERFLOW;  // slab too small for the worst case: refuse rather than test per symbol
        meta[s] = m;
        live = false;
    }
    s_off[lane] = st.sym_off;
    s_n[lane] = live ? st.n : 0u;
    if (lane == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        mbar_fence_init();
    }
    __syncwarp();

    // tables: row i of stream j's window -> tab[i*32 + j]
    for (uint32_t j = 0; j < 32; j++) {
        const uint32_t sj = blockIdx.x * 32u + j;
        const bool lj = __shfl_sync(0xffffffffu, (int)live, j) != 0;
        const uint32_t wj = __shfl_sync(0xffffffffu, m.win_rows, j);
        const uint32_t oj = __shfl_sync(0xffffffffu, m.win_lo, j);
        if (!lj) continue;
        const uint32_t* src = cumtab + (size_t)sj * kCumRow + oj;
        for (uint32_t i = lane; i < wj; i += 32) tab[i * 32u + j] = (CumT)src[i];
    }

    const PerLaneTable<CumT> T{tab, lane};
    const uint32_t bits = st.prob_bits;
    uint32_t* words = reinterpret_cast<uint32_t*>(out + st.out_off);
    const uint32_t cap_words = st.out_cap / 4u;
    uint32_t widx = cap_words;
    uint64_t x = kRansL;  // rans64.hpp:65

    uint32_t n_max = s_n[lane];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, d));
    const uint32_t my_n = live ? st.n : 0u;
    const uint32_t full = 1u << bits;
    const uint32_t win_lo = m.win_lo;
    const uint32_t sym_max = live ? m.win_rows - 2u : 0u;  // index of the last window row that is a symbol

    // entropy_encoding.hpp:222-225, last symbol first, as a software pipeline over groups of kGroup
    // symbols: while the serial state updates of group g run, the table lookups and reciprocals of group
    // g-1 (independent of the state) are computed, so they are ready long before the chain needs them
    // and their instructions fill the chain's dependency stalls.  Groups are numbered across chunks:
    // group g covers symbols [kGroup*g, kGroup*g + kGroup).
    const int n_chunks = (int)((n_max + kChunk - 1) / kChunk);
    constexpr int kGroupsPerChunk = kChunk / kGroup;
    const uint16_t* my_sym = symbols + st.sym_off;
    uint32_t bar_parity = 0;   // bit b: parity of the next completion of s_bar[b]
    uint32_t bulk_loaded = 0;  // bit b: the chunk in buffer b came through the copy engine (else cp.async)
    // chunk -> buffer (chunk & 1).  Warp-uniform choice of mechanism: the copy engine when no stream has a ragged chunk.
    auto load_chunk = [&](int chunk) {
        const uint32_t b = (uint32_t)chunk & 1u, first = (uint32_t)chunk * kChunk;
        const uint32_t left = my_n > first ? my_n - first : 0u;
        uint16_t* buf = stage0 + b * 32 * kBulkStride;
        if (__any_sync(0xffffffffu, left > 0u && left < (uint32_t)kChunk)) {
            stage_load_chunk<kBulkStride>(buf, symbols, s_off, s_n, (uint32_t)chunk);
            bulk_loaded &= ~(1u << b);
        } else {
            const uint32_t rows_in = __popc(__ballot_sync(0xffffffffu, left != 0u));
            fence_proxy_async();  // the buffer's previous contents were read through the generic proxy
            if (left) bulk_g2s(buf + lane * kBulkStride, my_sym + first, kChunk * 2u, &s_bar[b]);
            if (lane == 0) mbar_expect_tx(&s_bar[b], rows_in * kChunk * 2u);
            bulk_loaded |= 1u << b;
        }
    };
    auto wait_chunk = [&](int chunk) {
        const uint32_t b = (uint32_t)chunk & 1u;
        if (bulk_loaded & (1u << b)) {
            mbar_wait(&s_bar[b], (bar_parity >> b) & 1u);
            bar_parity ^= 1u << b;
            __syncwarp();
        } else {
            stage_wait();
        }
    };
    auto group_words = [&](int g) -> uint4 {  // the 8 symbols of group g from the staging buffer (one LDS.128)
        const int chunk = g / kGroupsPerChunk, k0 = (g % kGroupsPerChunk) * kGroup;
        return *reinterpret_cast<const uint4*>(stage0 + (chunk & 1) * 32 * kBulkStride + lane * kBulkStride + k0);
    };
    // start / freq / reciprocal of symbol j of group g (independent of the coder's state)
    auto prepare_one = [&](int g, int j, const uint4& v, uint32_t& o_start, uint32_t& o_freq, double& o_inv) {
        const uint32_t w = j < 2 ? v.x : (j < 4 ? v.y : (j < 6 ? v.z : v.w));
        const bool on = (uint32_t)g * kGroup + (uint32_t)j < my_n;
        const uint32_t raw = (j & 1) ? (w >> 16) : (w & 0xffffu);
        // window-relative index; out-of-alphabet input must not index past the lane's table
        const uint32_t sym = on ? min(raw - win_lo, sym_max) : 0u;
        const uint32_t c0 = T.cum(sym), c1 = T.cum(sym + 1u);
        o_start = on ? c0 : 0u;  // padding step: freq = 2^bits, start = 0 leaves x untouched
        o_freq = on ? c1 - c0 : full;
        o_inv = recip_low(o_freq);
    };
    auto prepare = [&](int g, uint32_t(&g_start)[kGroup], uint32_t(&g_freq)[kGroup], double(&g_inv)[kGroup]) {
        const uint4 v = group_words(g);
#pragma unroll
        for (int j = 0; j < kGroup; j++) prepare_one(g, j, v, g_start[j], g_freq[j], g_inv[j]);
    };
    auto run = [&](const uint32_t(&g_start)[kGroup], const uint32_t(&g_freq)[kGroup], const double(&g_inv)[kGroup]) {
#pragma unroll
        for (int j = kGroup - 1; j >= 0; j--)
            x = rans_put<LOW_BITS ? 1 : 0>(x, g_start[j], g_freq[j], g_inv[j], bits, words, widx);
    };
    if (n_chunks > 0) {
        uint32_t a_start[kGroup], a_freq[kGroup], b_start[kGroup], b_freq[kGroup];
        double a_inv[kGroup], b_inv[kGroup];
        load_chunk(n_chunks - 1);
        wait_chunk(n_chunks - 1);
        if (n_chunks > 1) load_chunk(n_chunks - 2);
        const int n_groups = n_chunks * kGroupsPerChunk;  // even
        prepare(n_groups - 1, a_start, a_freq, a_inv);
        // (Weaving the preparation of group g-1 into the steps of group g by hand - symbol by symbol, held in place by
        // false dependencies - was tried: ptxas then does interleave the two streams, and the kernel takes the same 8.9 ms.)
        for (int g = n_groups - 1; g >= 1; g -= 2) {
            prepare(g - 1, b_start, b_freq, b_inv);  // g odd: g-1 is in the same chunk
            run(a_start, a_freq, a_inv);
            if (g - 1 >= 1) {
                if (((g - 1) % kGroupsPerChunk) == 0) {  // group g-2 is the last of the previous chunk
                    const int chunk = (g - 1) / kGroupsPerChunk;
                    wait_chunk(chunk - 1);  // chunk-1 has landed; this chunk's buffer is free (its last group is in b_*)
                    if (chunk >= 2) load_chunk(chunk - 2);
                }
                prepare(g - 2, a_start, a_freq, a_inv);
            }
            run(b_start, b_freq, b_inv);
        }
    }
    if (live) {
        // rans64.hpp:96-103 flush: low word at the lower address
        widx -= 2;
        words[widx] = (uint32_t)x;
        words[widx + 1] = (uint32_t)(x >> 32);
        m.payload_start = st.out_off + (uint64_t)widx * 4u;
        m.payload_bytes = (cap_words - widx) * 4u;
        meta[s] = m;
    }
}

// -------------------------------------------------------------------------------------------------
// The same encoder, warp-specialised: two warps per CTA share 32 streams (lane = stream in both).
// -------------------------------------------------------------------------------------------------
// A stream's step is a chain of ~20 dependent instructions (~80 cycles) and the preparation of a symbol (two table
// rows, an fp64 reciprocal) is ~35 instructions of which a group of eight overlap each other.  In ONE warp the two
// run one after the other whatever the source says — a warp issues in order and ptxas does not weave a second
// dependent chain into the stalls of the first (ncu source view of k_rans_encode with the weaving forced by false
// dependencies: the reciprocal's DFMA chain simply sits between two steps, 237 cycles per symbol all the same).
// In TWO warps the hardware scheduler does the weaving: the FEEDER warp reads the symbols (16 bytes = 8 symbols per lane
// straight from global memory, two groups ahead: no staging buffer, no copy loop), looks up start / freq, computes the
// reciprocal and hands (start, freq, 1/freq) over through shared memory, 8 symbols per lane at a time, double
// buffered; the CODER warp runs nothing but the serial steps and the renormalisation stores.  Hand-over by named
// barriers (bar.sync / bar.arrive, 64 threads): buffer b is "empty" on barrier b and "full" on barrier 2 + b (four
// barriers per CTA: an SM has 64, and they must not be what limits the CTAs it holds).
// Requires every stream's symbols 16-byte aligned and readable up to the next multiple of 8 symbols (the tile codec's
// and layer_encode's planes are); other callers keep k_rans_encode.
constexpr int kWsGroup = 8;
template <int ID>
__device__ __forceinline__ void bar_sync_named() { asm volatile("bar.sync %0, 64;" ::"n"(ID) : "memory"); }
template <int ID>
__device__ __forceinline__ void bar_arrive_named() { asm volatile("bar.arrive %0, 64;" ::"n"(ID) : "memory"); }

template <typename CumT, int DIV>
__global__ void __launch_bounds__(64) k_rans_encode_ws(const hoh_enc_stream* __restrict__ streams, uint32_t n_streams,
                                                       const uint16_t* __restrict__ symbols,
                                                       const uint32_t* __restrict__ cumtab, uint8_t* __restrict__ out,
                                                       EncMeta* __restrict__ meta, uint32_t rows_lo, uint32_t rows,
                                                       uint32_t want_u16, const uint32_t* __restrict__ order,
                                                       const uint32_t* __restrict__ n_active) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    CumT* tab = reinterpret_cast<CumT*>(smem_raw);
    uint4* hand = reinterpret_cast<uint4*>(smem_raw + (size_t)rows * 32u * sizeof(CumT));  // [2][kWsGroup][32]

    const uint32_t lane = lane_id();
    const bool feeder = threadIdx.x >= 32u;
    // `order` (optional): the streams to code, as a dense list of *n_active indices into `streams` - a caller that
    // wants a subset coded keeps the warps full this way (hoh_layer_encode_batch codes one candidate in six)
    const uint32_t slot = blockIdx.x * 32u + lane;
    const uint32_t n_slots = order ? *n_active : n_streams;
    if (blockIdx.x * 32u >= n_slots) return;
    const bool exists = slot < n_slots;
    const uint32_t s = exists ? (order ? order[slot] : slot) : 0u;
    hoh_enc_stream st;
    EncMeta m;
    if (exists) {
        st = streams[s];
        m = meta[s];
    } else {
        st.n = 0;
        st.range = 1;
        st.prob_bits = 1;
        st.sym_off = 0;
        st.out_off = 0;
        st.out_cap = 0;
        m.status = HOH_S_OK;
        m.table_u16 = want_u16;
        m.win_lo = 0;
        m.win_rows = 0;
    }
    // (both warps evaluate the same streams, so every decision below is the same in both)
    bool live = exists && st.n > 0 && m.status == HOH_S_OK && m.table_u16 == want_u16;
    uint32_t need = live ? m.win_rows : 0u;
    uint32_t low = live ? st.prob_bits : 32u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        need = max(need, __shfl_xor_sync(0xffffffffu, need, d));
        low = min(low, __shfl_xor_sync(0xffffffffu, low, d));
    }
    if (need <= rows_lo || need > rows) return;  // another class's launch (or nothing to do)
    // the instantiation that fits the warp's narrowest stream (rans_put): every warp runs in exactly one of the three
    if ((low >= 14u ? 0 : (low >= 12u ? 2 : 1)) != DIV) return;
    if (live && (uint64_t)st.out_cap < rans_words_bound(st.n, st.prob_bits) * 4u + HOH_HEAD_CAP + 32u) {
        m.status = HOH_S_OVERFLOW;  // slab too small for the worst case: refuse rather than test per symbol
        if (!feeder) meta[s] = m;
        live = false;
    }
    // tables: row i of stream j's window -> tab[i*32 + j], filled by all 64 threads
    for (uint32_t j = 0; j < 32; j++) {
        const uint32_t sj = __shfl_sync(0xffffffffu, s, j);
        const bool lj = __shfl_sync(0xffffffffu, (int)live, j) != 0;
        const uint32_t wj = __shfl_sync(0xffffffffu, m.win_rows, j);
        const uint32_t oj = __shfl_sync(0xffffffffu, m.win_lo, j);
        if (!lj) continue;
        const uint32_t* src = cumtab + (size_t)sj * kCumRow + oj;
        for (uint32_t i = threadIdx.x; i < wj; i += 64) tab[i * 32u + j] = (CumT)src[i];
    }
    __syncthreads();

    const uint32_t bits = st.prob_bits;
    const uint32_t my_n = live ? st.n : 0u;
    uint32_t n_max = my_n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, d));
    const int n_groups = (int)((n_max + kWsGroup - 1) / kWsGroup);

    if (feeder) {
        const PerLaneTable<CumT> T{tab, lane};
        const uint32_t full = 1u << bits;
        const uint32_t win_lo = m.win_lo;
        const uint32_t sym_max = live ? m.win_rows - 2u : 0u;  // index of the last window row that is a symbol
        const uint16_t* my_sym = symbols + st.sym_off;
        auto load = [&](int g) -> uint4 {  // the 8 symbols of group g (never past the stream's last group)
            if (g >= 0 && (uint32_t)g * kWsGroup < my_n) return __ldg(reinterpret_cast<const uint4*>(my_sym + (size_t)g * kWsGroup));
            return make_uint4(0u, 0u, 0u, 0u);
        };
        // entropy_encoding.hpp:222-225: last symbol first.  Two groups per trip: the barrier numbers are literals, and each
        // half owns a register set that it reloads (for the group two further on) as soon as it has unpacked it - a
        // rotation by register moves would wait for the load it moves (ncu: 36 % of the feeder's time, long scoreboard)
        uint4 set0 = load(n_groups - 1), set1 = load(n_groups - 2);
        auto feed = [&](int g, auto buf, uint4& mine) {
            constexpr int b = decltype(buf)::value;
            const uint4 cur = mine;
            uint32_t o_start[kWsGroup], o_freq[kWsGroup];
            double o_inv[kWsGroup];
#pragma unroll
            for (int j = 0; j < kWsGroup; j++) {
                const uint32_t w = j < 2 ? cur.x : (j < 4 ? cur.y : (j < 6 ? cur.z : cur.w));
                const bool on = (uint32_t)g * kWsGroup + (uint32_t)j < my_n;
                const uint32_t raw = (j & 1) ? (w >> 16) : (w & 0xffffu);
                // window-relative index; out-of-alphabet input must not index past the lane's table
                const uint32_t sym = on ? min(raw - win_lo, sym_max) : 0u;
                const uint32_t c0 = T.cum(sym), c1 = T.cum(sym + 1u);
                o_start[j] = on ? c0 : 0u;  // padding step: freq = 2^bits, start = 0 leaves x untouched
                o_freq[j] = on ? c1 - c0 : full;
                o_inv[j] = recip_low(o_freq[j]);
            }
            mine = load(g - 2);  // in flight while two groups are prepared
            bar_sync_named<b>();  // the coder has taken the buffer's previous contents
            uint4* dst = hand + (b * kWsGroup) * 32 + lane;
#pragma unroll
            for (int j = 0; j < kWsGroup; j++)
                dst[j * 32] = make_uint4(o_start[j], o_freq[j], (uint32_t)__double2loint(o_inv[j]), (uint32_t)__double2hiint(o_inv[j]));
            bar_arrive_named<2 + b>();  // full
        };
        for (int g = n_groups - 1; g >= 0; g -= 2) {
            feed(g, std::integral_constant<int, 0>{}, set0);
            if (g >= 1) feed(g - 1, std::integral_constant<int, 1>{}, set1);
        }
        return;
    }

    uint32_t* words = reinterpret_cast<uint32_t*>(out + st.out_off);
    const uint32_t cap_words = st.out_cap / 4u;
    uint32_t widx = cap_words;
    uint64_t x = kRansL;  // rans64.hpp:65
    bar_arrive_named<0>();  // both buffers start empty
    bar_arrive_named<1>();
    auto code = [&](auto buf) {
        constexpr int b = decltype(buf)::value;
        bar_sync_named<2 + b>();
        const uint4* src = hand + (b * kWsGroup) * 32 + lane;
        uint4 h[kWsGroup];
#pragma unroll
        for (int j = 0; j < kWsGroup; j++) h[j] = src[j * 32];
        bar_arrive_named<b>();  // everything is in registers: the feeder may refill
#pragma unroll
        for (int j = kWsGroup - 1; j >= 0; j--)
            x = rans_put<DIV>(x, h[j].x, h[j].y, __hiloint2double((int)h[j].w, (int)h[j].z), bits, words, widx);
    };
    for (int it = 0; it < n_groups; it += 2) {
        code(std::integral_constant<int, 0>{});
        if (it + 1 < n_groups) code(std::integral_constant<int, 1>{});
    }
    if (live) {
        // rans64.hpp:96-103 flush: low word at the lower address
        widx -= 2;
        words[widx] = (uint32_t)x;
        words[widx + 1] = (uint32_t)(x >> 32);
        m.payload_start = st.out_off + (uint64_t)widx * 4u;
        m.payload_bytes = (cap_words - widx) * 4u;
        meta[s] = m;
    }
}

// -------------------------------------------------------------------------------------------------
// Finish — entropy_encoding.hpp:232-267: length varint in front of the payload, or the stored-mode
// rewrite when that is smaller.  One warp per stream.  The header is written immediately in front
// of the payload (which already sits at the END of the stream's slab), so the payload never moves.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_finish_streams(const hoh_enc_stream* __restrict__ streams,
                                                        uint32_t n_streams, const uint16_t* __restrict__ symbols,
                                                        const uint8_t* __restrict__ heads,
                                                        const EncMeta* __restrict__ meta, uint8_t* __restrict__ out,
                                                        hoh_stream_result* __restrict__ results,
                                                        const uint32_t* __restrict__ order,
                                                        const uint32_t* __restrict__ n_active) {
    const uint32_t slot = blockIdx.x * 4u + (threadIdx.x >> 5), lane = lane_id();
    if (slot >= (order ? *n_active : n_streams)) return;
    const uint32_t s = order ? order[slot] : slot;  // as in k_rans_encode_ws
    const hoh_enc_stream st = streams[s];
    const EncMeta m = meta[s];
    const uint8_t* head = heads + (size_t)s * HOH_HEAD_CAP;
    hoh_stream_result res;
    res.status = m.status;
    res.payload_bytes = 0;
    res.stored = 0;
    res.start = st.out_off;
    res.size = 0;
    if (m.status != HOH_S_OK) {
        if (lane == 0) results[s] = res;
        return;
    }
    if (st.n == 0) {
        uint8_t* dst = out + st.out_off;
        if (lane == 0) {
            for (uint32_t k = 0; k < st.prefix_len; k++) dst[k] = st.prefix[k];
            for (uint32_t k = 0; k < m.head_len; k++) dst[st.prefix_len + k] = head[k];
            res.size = st.prefix_len + m.head_len;
            results[s] = res;
        }
        return;
    }
    {  // the coded length against what k_build_tables derived from the histogram (warp_estimate_words)
        const uint32_t w = (m.payload_bytes - 8u) / 4u, lo = m.est & 0xffffffu, span = m.est >> 24;
        if (span != 255u && (w < lo || w > lo + span)) res.status = HOH_S_BAD_ESTIMATE;
    }
    const uint32_t vlen = hohfmt::varint_len(m.payload_bytes);
    const uint32_t coded = m.head_len + vlen + m.payload_bytes;  // what encode_entropy returns
    if (m.stored_size < coded) {  // entropy_encoding.hpp:244-267
        uint8_t* dst = out + st.out_off;
        const uint32_t maxbits = hohfmt::bit_length(st.range - 1);
        uint32_t at = st.prefix_len;
        if (lane == 0) {
            for (uint32_t k = 0; k < st.prefix_len; k++) dst[k] = st.prefix[k];
            uint32_t a = hohfmt::put_varint(dst, at, st.range - 1);
            a = hohfmt::put_varint(dst, a, st.n);
            dst[a] = 0;
        }
        at += hohfmt::varint_len(st.range - 1) + hohfmt::varint_len(st.n) + 1u;
        const uint32_t body = (uint32_t)(((uint64_t)maxbits * st.n + 7) / 8);
        const uint16_t* sym = symbols + st.sym_off;
        for (uint32_t b = lane; b < body; b += 32) {  // MSB-first packing, symbol i at bit i*maxbits
            uint32_t byte = 0;
            for (uint32_t k = 0; k < 8; k++) {
                const uint64_t bit = (uint64_t)b * 8u + k;
                const uint64_t i = bit / maxbits;
                uint32_t v = 0;
                if (i < st.n) v = (sym[i] >> (maxbits - 1u - (uint32_t)(bit % maxbits))) & 1u;
                byte = (byte << 1) | v;
            }
            dst[at + b] = (uint8_t)byte;
        }
        res.size = st.prefix_len + m.stored_size;
        res.stored = 1;
        if (lane == 0) results[s] = res;
        return;
    }
    const uint32_t front = st.prefix_len + m.head_len + vlen;
    uint8_t* dst = out + m.payload_start - front;
    for (uint32_t k = lane; k < st.prefix_len; k += 32) dst[k] = st.prefix[k];
    for (uint32_t k = lane; k < m.head_len; k += 32) dst[st.prefix_len + k] = head[k];
    if (lane == 0) {
        hohfmt::put_varint(dst, st.prefix_len + m.head_len, m.payload_bytes);
        res.start = m.payload_start - front;
        res.size = front + m.payload_bytes;
        res.payload_bytes = m.payload_bytes;
        results[s] = res;
    }
}

// =================================================================================================
// Decode: header + table parse — entropy_decoding.hpp:143-253.  One warp per stream.
// =================================================================================================
__global__ void __launch_bounds__(kTableWarps * 32) k_parse_streams(
    const hoh_dec_stream* __restrict__ streams, uint32_t n_streams, const uint8_t* __restrict__ in,
    uint64_t in_bytes, uint32_t* __restrict__ cumtab, DecMeta* __restrict__ meta,
    hoh_dec_result* __restrict__ results) {
    __shared__ uint32_t s_f[kTableWarps][kFreqRow];
    __shared__ uint32_t s_cum[kTableWarps][kFreqRow + 8];
    const uint32_t w = threadIdx.x >> 5, lane = lane_id();
    const uint32_t s = blockIdx.x * kTableWarps + w;
    if (s >= n_streams) return;
    const hoh_dec_stream st = streams[s];
    const ByteView bytes{in, in_bytes};
    uint32_t* f = s_f[w];
    uint32_t* cum = s_cum[w];

    // lane 0 reads the header (varints, metadata byte) and, for table mode 2, the clamp pairs; the
    // frequency fields themselves are read by all lanes below
    hohfmt::StreamHead h;
    uint64_t after_table = 0;
    int status = HOH_S_OK;
    uint32_t* clamps = s_cum[w];  // [0] = count, [1..] = lo | hi << 16 (the cumulative counts come later)
    uint64_t field_bit = 0;       // absolute bit position (from byte 0 of the buffer) of the first frequency
    if (lane == 0) {
        h = hohfmt::parse_head(bytes, st.in_off, st.flags);
        after_table = h.body;
        field_bit = h.body * 8u;
        if (!h.empty && h.rans) {
            if (h.range > HOH_MAX_RANGE) {
                status = HOH_S_BAD_TABLE;
            } else if (h.table_mode == 2) {  // entropy_decoding.hpp:196-213: clamp pairs on maxbits bits each
                hohfmt::BitSource<ByteView> bits{bytes, h.body, 0, 0};
                uint32_t count = (uint32_t)(((int)h.prob_bits - 1) / 4 + 2);  // :197, int arithmetic
                if (count > 16u) count = 16u;
                clamps[0] = count;
                for (uint32_t j = 0; j < count; j++) {
                    const uint32_t lo = bits.get(h.maxbits) & 0xffffu;
                    const uint32_t hi = bits.get(h.maxbits) & 0xffffu;
                    clamps[1 + j] = lo | (hi << 16);
                }
                field_bit += 2ull * count * h.maxbits;
            } else if (h.table_mode == 3) {
                status = HOH_S_BAD_TABLE;
            }
            // HOH_FIX_CARRY.  A stream with ONE distinct symbol s writes the value 2^prob_bits into a prob_bits-wide
            // field.  The reference's bit packer ADDS fields into its pending byte (varint.hpp:47-77), so the field
            // itself reads 0 and the extra bit increments the bits already written in that byte (mod 2^k, k = bits
            // of the clamp pairs that share the field's first byte; k = 0: the bit is simply lost).  A valid table
            // never has frequency 0 for the first symbol inside its clamps, so the pattern is unambiguous: when the
            // field reads 0 and, with the increment undone, every clamp value is the same symbol, that symbol owns
            // the whole range.
            if ((st.flags & HOH_FIX_CARRY) && h.table_mode == 2u && status == HOH_S_OK && h.prob_bits >= 1u &&
                h.prob_bits <= HOH_MAX_PROB_BITS) {
                const uint32_t count = clamps[0];
                uint32_t v[32];
                for (uint32_t j = 0; j < count; j++) {
                    v[2u * j] = clamps[1 + j] & 0xffffu;
                    v[2u * j + 1u] = clamps[1 + j] >> 16;
                }
                hohfmt::BitSource<ByteView> bits{bytes, h.body, 0, 0};
                for (uint32_t j = 0; j < 2u * count; j++) bits.get(h.maxbits);
                const uint32_t field = bits.get(h.prob_bits);
                uint32_t rem = (2u * count * h.maxbits) & 7u;  // k
                bool borrow = true;
                for (int j = (int)(2u * count) - 1; j >= 0 && rem && borrow; j--) {
                    const uint32_t t = min(rem, h.maxbits), mask = (1u << t) - 1u;
                    uint32_t part = v[j] & mask;
                    if (part == 0u) part = mask;
                    else {
                        part--;
                        borrow = false;
                    }
                    v[j] = (v[j] & ~mask) | part;
                    rem -= t;
                }
                bool lone = field == 0u && count > 0u;
                for (uint32_t j = 1; j < 2u * count; j++) lone = lone && v[j] == v[0];
                if (lone && v[0] < h.range) {
                    clamps[0] = 0xffffffffu;  // marks the recovered table
                    clamps[1] = v[0];
                    field_bit = h.body * 8u + 2ull * count * h.maxbits + h.prob_bits;
                }
            }
        }
    }
    h.range = __shfl_sync(0xffffffffu, h.range, 0);
    h.n = __shfl_sync(0xffffffffu, h.n, 0);
    h.maxbits = __shfl_sync(0xffffffffu, h.maxbits, 0);
    h.rans = __shfl_sync(0xffffffffu, h.rans, 0);
    h.prob_bits = __shfl_sync(0xffffffffu, h.prob_bits, 0);
    h.table_mode = __shfl_sync(0xffffffffu, h.table_mode, 0);
    h.empty = __shfl_sync(0xffffffffu, h.empty, 0);
    h.body = __shfl_sync(0xffffffffu, h.body, 0);
    after_table = __shfl_sync(0xffffffffu, after_table, 0);
    field_bit = __shfl_sync(0xffffffffu, field_bit, 0);
    status = __shfl_sync(0xffffffffu, status, 0);
    __syncwarp();

    // table modes 1 and 2 (entropy_decoding.hpp:180-244): every lane reads the fields of its contiguous
    // run of symbols; widths per symbol, then bit offsets by prefix sum, then the reference's bit reader
    // positioned at the run's first bit
    if (!h.empty && h.rans && status == HOH_S_OK && h.table_mode == 2u && clamps[0] == 0xffffffffu) {
        const uint32_t lone = clamps[1];  // recovered lone-symbol table (HOH_FIX_CARRY)
        __syncwarp();
        for (uint32_t i = lane; i < h.range; i += 32) f[i] = i == lone ? (1u << h.prob_bits) : 0u;
        after_table = (field_bit + 7u) >> 3;
        __syncwarp();
    } else if (!h.empty && h.rans && status == HOH_S_OK && (h.table_mode == 1u || h.table_mode == 2u)) {
        const uint32_t count = h.table_mode == 2u ? clamps[0] : 0u;
        const uint32_t per = (h.range + 31u) / 32u;
        const uint32_t lo = min(lane * per, h.range), hi = min(lo + per, h.range);
        auto width_of = [&](uint32_t i) -> uint32_t {
            if (h.table_mode == 1u) return h.maxbits;
            uint32_t wd = 0;  // hohfmt::clamp_width_of
            for (uint32_t j = 0; j < count; j++) {
                const uint32_t c = clamps[1 + j];
                if ((c & 0xffffu) <= i && (c >> 16) >= i) wd = j == 0 ? 1u : 4u * j;
            }
            return min(wd, h.prob_bits);
        };
        uint32_t my_bits = 0;
        for (uint32_t i = lo; i < hi; i++) my_bits += width_of(i);
        const uint32_t incl = warp_incl_scan(my_bits);
        const uint64_t my_bit = field_bit + (incl - my_bits);
        const uint64_t end_bit = field_bit + __shfl_sync(0xffffffffu, incl, 31);
        hohfmt::BitSource<ByteView> bits{bytes, my_bit >> 3, 0, 0};
        if (my_bit & 7u) {  // start inside a byte: its low bits are the first ones of this run
            bits.have = 8u - (uint32_t)(my_bit & 7u);
            bits.held = bytes[bits.at++] & ((1u << bits.have) - 1u);
        }
        for (uint32_t i = lo; i < hi; i++) f[i] = bits.get(width_of(i));
        after_table = (end_bit + 7u) >> 3;
        __syncwarp();
    }

    DecMeta m;
    m.payload_off = h.body;
    m.n = h.n;
    m.range = h.range;
    m.prob_bits = h.prob_bits;
    m.kind = 0;
    m.maxbits = h.maxbits;
    m.status = status;
    m.used = 0;
    m.pad = 0;
    hoh_dec_result res;
    res.end_off = h.body;
    res.n = h.n;
    res.status = status;
    res.range = h.range;
    res.prob_bits = h.prob_bits;
    res.stored = 0;
    res.table_mode = h.table_mode;

    if (h.empty) {
        // nothing
    } else if (!h.rans) {  // entropy_decoding.hpp:278-290
        m.kind = 1;
        res.stored = 1;
        res.end_off = h.body + ((uint64_t)h.maxbits * h.n + 7) / 8;
    } else if (status == HOH_S_OK) {
        const uint32_t target = h.prob_bits < 32 ? (1u << h.prob_bits) : 0u;
        if (h.table_mode == 0) {  // entropy_decoding.hpp:174-179: flat counts through normalize_freqs
            if (target < h.range) {
                status = HOH_S_RANGE_GT_TOTAL;
            } else {
                for (uint32_t i = lane; i < h.range; i += 32) {
                    uint32_t a = (uint32_t)(((uint64_t)target * i) / h.range);
                    uint32_t b = (uint32_t)(((uint64_t)target * (i + 1)) / h.range);
                    f[i] = b - a;
                }
            }
        }
        __syncwarp();
        if (status == HOH_S_OK) {
            warp_cumsum(f, cum, h.range);  // stattools.hpp:6-11
            // Dense decode table: one packed entry (cum << 9 | symbol) per symbol that has a non-zero
            // frequency, in symbol order (so the packed words are strictly increasing).  Dropping the empty symbols changes nothing for a valid table
            // (a slot never falls on one) and keeps the lookup's neighbourhood search short.  Physical
            // rows: [0] = leading sentinel (0), [1 .. used] = entries, [used+1] = the total, [used+2] = all ones
            // (a row no slot can reach: the lookup needs no bounds tests).
            uint32_t* ct = cumtab + (size_t)s * kCumRow;
            {
                const uint32_t per = (h.range + 31u) / 32u;
                const uint32_t lo = min(lane * per, h.range), hi = min(lo + per, h.range);
                uint32_t cnt = 0;
                for (uint32_t i = lo; i < hi; i++) cnt += f[i] != 0u;
                const uint32_t incl = warp_incl_scan(cnt);
                uint32_t d = incl - cnt;
                for (uint32_t i = lo; i < hi; i++)
                    if (f[i] != 0u) ct[1u + d++] = (cum[i] << kSymBits) | i;
                m.used = __shfl_sync(0xffffffffu, incl, 31);
                if (lane == 0) {
                    ct[0] = 0u;
                    ct[m.used + 1u] = cum[h.range] << kSymBits;
                    ct[m.used + 2u] = 0xffffffffu;
                }
            }
            if (m.used == 0u || cum[h.range] >= (1u << 22) || h.prob_bits > HOH_MAX_PROB_BITS || h.prob_bits == 0u)
                status = HOH_S_BAD_TABLE;
            uint64_t at = after_table;
            const uint32_t payload = hohfmt::get_varint(bytes, &at);  // entropy_decoding.hpp:256
            m.payload_off = at;
            m.kind = status == HOH_S_OK ? 2u : 0u;
            res.end_off = (st.flags & HOH_FIX_ADVANCE) ? at + payload : at;  // D8
        }
        m.status = status;
        res.status = status;
    }
    if (m.n > st.sym_cap) {
        m.status = m.status == HOH_S_OK ? HOH_S_OVERFLOW : m.status;
        res.status = m.status;
    }
    if (lane == 0) {
        meta[s] = m;
        results[s] = res;
    }
}

// Stored-mode symbols — entropy_decoding.hpp:278-290.  One CTA per stream, exits unless stored.
__global__ void __launch_bounds__(256) k_unpack_stored(const hoh_dec_stream* __restrict__ streams,
                                                       const uint8_t* __restrict__ in, uint64_t in_bytes,
                                                       const DecMeta* __restrict__ meta,
                                                       uint16_t* __restrict__ symbols) {
    const DecMeta m = meta[blockIdx.x];
    if (m.kind != 1) return;
    const hoh_dec_stream st = streams[blockIdx.x];
    const ByteView bytes{in, in_bytes};
    const uint32_t n = min(m.n, st.sym_cap);
    uint16_t* dst = symbols + st.sym_off;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        uint64_t bit = (uint64_t)i * m.maxbits;
        uint32_t v = 0;
        for (uint32_t k = 0; k < m.maxbits; k++, bit++)
            v = (v << 1) | ((bytes[m.payload_off + (bit >> 3)] >> (7u - (uint32_t)(bit & 7u))) & 1u);
        dst[i] = (uint16_t)v;
    }
}

// -------------------------------------------------------------------------------------------------
// rANS decode, per-stream tables — entropy_decoding.hpp:254-276 with rans64.hpp:107-142.
// -------------------------------------------------------------------------------------------------
// Payload words.  Every lane reads its own stream, at its own data-dependent pace, starting at an
// arbitrary byte offset (SURVEY H3).  Words are staged in a per-lane ring in shared memory filled by
// cp.async in aligned 16-byte blocks: nothing in the decode loop ever names a register with a load in
// flight (a register look-ahead queue stalls on exactly that), and the ring is topped up at uniform
// points (every kTopUp symbols) far enough ahead that a whole period of consumption is always resident:
// a symbol consumes at most one word and a top-up requests words up to position + kAhead, so whatever
// is read during one period was requested by the previous top-up at the latest, whose copies are
// complete (cp.async.wait_group 1) before the period starts.
constexpr int kRingWords = 32;  // per lane, power of two (>= kAhead + 3 + 4: requests never overwrite unread words)
constexpr int kTopUp = 8;       // symbols between two top-ups (<= 8 words consumed)
constexpr int kAhead = 20;      // words requested ahead of the read position (>= 2 * kTopUp + 2)

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
// the same under a predicate of the instruction itself (no branch around it; the address is not touched when off)
__device__ __forceinline__ void cp_async16_if(uint32_t smem_addr, const void* gptr, bool on) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.u32 p, %2, 0;\n"
        "@p cp.async.cg.shared.global [%0], [%1], 16;\n"
        "}\n" ::"r"(smem_addr),
        "l"(gptr), "r"((uint32_t)on)
        : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

struct WordRing {
    const uint32_t* base16;  // 16-byte aligned word pointer at or below the first payload byte
    uint32_t* ring;          // this lane's kRingWords words of shared memory
    uint32_t ring_addr;      // the same, as a shared-window address
    uint32_t pos;            // aligned-word index (from base16) holding the first byte of `next`
    uint32_t end;            // aligned-word index up to which blocks have been requested (multiple of 4)
    uint32_t limit;          // first aligned-word index that must not be read (multiple of 4, inside the buffer)
    uint32_t shift;          // 8 * byte misalignment of the payload
    uint32_t next;           // the next payload word, assembled
    uint32_t wa, wb;         // ring[pos + 1], ring[pos + 2]: the aligned words the word after `next` is cut from

    __device__ __forceinline__ void request(uint32_t want) {  // blocks up to word index `want`
        while (end < want) {
            if (end < limit) cp_async16(ring_addr + (end & (kRingWords - 1)) * 4u, base16 + end);
            end += 4u;
        }
    }
    // in / in_bytes: the whole input buffer (16-byte aligned base; reads stay inside it)
    __device__ __forceinline__ void open(const uint8_t* in, uint64_t in_bytes, uint64_t off, uint32_t* lane_ring) {
        ring = lane_ring;
        ring_addr = (uint32_t)__cvta_generic_to_shared(lane_ring);
        const uint64_t buf_end = (reinterpret_cast<uint64_t>(in) + in_bytes) & ~15ull;
        uint64_t addr = reinterpret_cast<uint64_t>(in) + off;
        if (addr + 16u > buf_end) addr = buf_end - 16u;  // a malformed offset must not leave the buffer
        base16 = reinterpret_cast<const uint32_t*>(addr & ~15ull);
        pos = (uint32_t)((addr & 15ull) >> 2);
        shift = (uint32_t)(addr & 3ull) * 8u;
        const uint64_t words_left = (buf_end - (addr & ~15ull)) / 4u;
        limit = (uint32_t)min(words_left, (uint64_t)0xfffffff0u);
        end = 0;
        request(pos + kAhead);
        cp_async_commit();
        cp_async_wait_group<0>();
        next = __funnelshift_r(ring[pos & (kRingWords - 1)], ring[(pos + 1u) & (kRingWords - 1)], shift);
        wa = ring[(pos + 1u) & (kRingWords - 1)];
        wb = ring[(pos + 2u) & (kRingWords - 1)];
    }
    // uniform point, every kTopUp symbols: request ahead, and make everything but that request resident.
    // Straight-line: the previous top-up left end >= pos_then + kAhead and at most kTopUp words were consumed since, so
    // at most two 4-word blocks are missing; each is one PREDICATED cp.async (the request() loop compiled to a chain of
    // ~8 branches, ~330 cycles per top-up in the ncu source view of the fused decoder — a tenth of the kernel).
    __device__ __forceinline__ void top_up() {
        const uint32_t want = pos + kAhead;
#pragma unroll
        for (int k = 0; k < (kTopUp + 3) / 4; k++) {
            const bool need = end < want;
            cp_async16_if(ring_addr + (end & (kRingWords - 1)) * 4u, base16 + end, need && end < limit);
            end += need ? 4u : 0u;
        }
        cp_async_commit();
        cp_async_wait_group<1>();
    }
    // Consume `next` if `take`.  Branch-free: the following word is cut from two registers that were
    // loaded when the previous word was taken (at least one whole step ago), and the only memory access
    // is one predicated shared-memory load whose result is not looked at before the next take.
    __device__ __forceinline__ void take_if(bool take) {
        const uint32_t following = __funnelshift_r(wa, wb, shift);
        next = take ? following : next;
        pos += take ? 1u : 0u;
        wa = take ? wb : wa;
        if (take) wb = ring[(pos + 2u) & (kRingWords - 1)];
    }
};

// Symbol lookup, the equivalent of cum2sym[slot] (entropy_decoding.hpp:262-267), over the dense table
// (physical rows: see k_parse_streams).  A 128-entry table indexed by the top 7 bits of the slot holds
// the row whose interval contains the MIDDLE of that 1/128th of the range, so the wanted row is that
// one or a direct neighbour unless several symbols share the bucket; the four rows around it are
// fetched together (independent loads: one shared-memory round trip on the dependent chain) and the
// answer is selected without a branch; only a slot further away takes the scan loops.  The result is
// the largest row with cum <= slot, i.e. the symbol the reference's 2^prob_bits-entry table holds.
constexpr int kLutSize = 128;

// Dense table accessors: PerLane = 32 independent tables interleaved [row][lane]; Shared = one table.
struct PerLaneDense {
    const uint32_t* tab;
    uint32_t lane;
    __device__ __forceinline__ uint32_t at(uint32_t p) const { return tab[p * 32u + lane]; }
    // A load the compiler may not predicate on the outcome of the other rows' comparisons: the four rows of a
    // lookup must leave together (one shared-memory round trip on the dependent chain, not two).
    __device__ __forceinline__ uint32_t at_eager(uint32_t p) const {
        uint32_t v;
        asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(tab + p * 32u + lane)));
        return v;
    }
};
struct SharedDense {
    const uint32_t* tab;
    __device__ __forceinline__ uint32_t at(uint32_t p) const { return tab[p]; }
    __device__ __forceinline__ uint32_t at_eager(uint32_t p) const { return tab[p]; }
};

// The same table addressed by a 32-bit shared-window address computed ONCE (base = address of tab[lane]): the loads
// are LDS [R + imm] with no uniform-register window base.  With generic pointers into the dynamic shared array the
// compiler rebuilds that base (S2UR SR_CgaCtaId / UMOV / ULEA) in every decode step of the fused kernel, because the
// out-of-line far walk clobbers the uniform registers, and the step waits ~10 cycles for it.
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
struct PerLaneDenseS {
    uint32_t base;  // shared address of row 0 of this lane's table
    __device__ __forceinline__ uint32_t at(uint32_t p) const { return lds_u32(base + p * 128u); }
    __device__ __forceinline__ uint32_t at_eager(uint32_t p) const { return lds_u32(base + p * 128u); }
    // rows p-1 .. p+2 from one address register (four independent loads: one round trip on the chain)
    __device__ __forceinline__ void at4(uint32_t p, uint32_t& em, uint32_t& e0, uint32_t& e1, uint32_t& e2) const {
        const uint32_t a = base + p * 128u;
        asm("ld.shared.u32 %0, [%4+-128];\n\tld.shared.u32 %1, [%4];\n\tld.shared.u32 %2, [%4+128];\n\tld.shared.u32 %3, [%4+256];"
            : "=r"(em), "=r"(e0), "=r"(e1), "=r"(e2)
            : "r"(a));
    }
};

template <typename Table, typename LutT>
__device__ __forceinline__ void lut_build(const Table& T, LutT* lut, uint32_t lut_stride, uint32_t lut_shift,
                                          uint32_t used) {
    uint32_t p = 1;
    const uint32_t half = lut_shift ? (1u << (lut_shift - 1u)) : 0u;
    for (uint32_t j = 0; j < (uint32_t)kLutSize; j++) {
        const uint32_t target = (j << lut_shift) + half;
        while (p < used && (T.at(p + 1u) >> kSymBits) <= target) p++;
        lut[j * lut_stride] = (LutT)p;
    }
}

// The lookup proper: (e, hi) = the packed rows around the slot, assuming the wanted row is the midpoint row or a
// direct neighbour.  With key = (slot + 1) << 9, "cum(row) <= slot" is simply "row < key" on the packed words.
// Returns false when that assumption does not hold for this lane (several symbols inside 1/128th of the range).
template <typename Table, typename LutT>
__device__ __forceinline__ bool rans_lookup_near(const Table& T, const LutT* lut, uint32_t lut_stride,
                                                 uint32_t lut_shift, uint32_t slot, uint32_t key, uint32_t& p,
                                                 uint32_t& e, uint32_t& hi) {
    p = lut[(slot >> lut_shift) * lut_stride];
    const uint32_t em = T.at(p - 1u), e0 = T.at(p), e1 = T.at(p + 1u), e2 = T.at_eager(p + 2u);
    const bool down = e0 >= key;  // the row holding the bucket's middle starts after the slot
    const bool up = e1 < key;     // ... or ends before it
    e = down ? em : (up ? e1 : e0);
    // e2 enters arithmetically: written as a select the compiler predicates its load on `up`, which puts a
    // second shared-memory round trip on the chain whenever any lane of the warp needs the upper neighbour
    uint32_t up_ones;  // all ones when e1 < key; produced where the compiler cannot turn it back into a select
    asm("set.lt.u32.u32 %0, %1, %2;" : "=r"(up_ones) : "r"(e1), "r"(key));
    hi = down ? e0 : e1 + ((e2 - e1) & up_ones);
    return e < key && hi >= key;
}

// Walks to the row that holds the slot from where the near lookup ended (p = the midpoint row it started from;
// rare: only lanes for which rans_lookup_near said no move).
template <typename Table>
__device__ __forceinline__ void rans_lookup_far(const Table& T, uint32_t key, uint32_t p, uint32_t& e, uint32_t& hi) {
    p = T.at(p) >= key ? p - 1u : (T.at(p + 1u) < key ? p + 1u : p);  // the row `e` came from
    while (e >= key) {
        p--;
        hi = e;
        e = T.at(p);
    }
    while (hi < key) {
        p++;
        e = hi;
        hi = T.at(p + 1u);
    }
}

template <typename Table>
__device__ __noinline__ ulonglong2 rans_far_step(const Table T, uint32_t key, uint32_t p, uint32_t e, uint32_t hi,
                                                 uint64_t top, uint32_t slot) {
    rans_lookup_far(T, key, p, e, hi);
    ulonglong2 r;
    r.x = (uint64_t)((hi >> kSymBits) - (e >> kSymBits)) * top + (slot - (e >> kSymBits));
    r.y = e;
    return r;
}

// One decode step (rans64.hpp:118-142).  There is no "past the end of this stream" case: a lane whose
// stream is shorter than its neighbours' keeps decoding (its table lookups and word reads stay in
// bounds whatever the state is) and the surplus symbols are simply not stored.
// The state update is computed from the near lookup straight away; whether some lane needs the far walk is
// voted on meanwhile, and only then (rare, warp-uniform) is the update redone — the vote's latency overlaps
// the multiply instead of preceding it.
template <typename Table, typename LutT>
__device__ __forceinline__ uint32_t rans_get(uint64_t& x, WordRing& rd, const Table& T, const LutT* lut,
                                             uint32_t lut_stride, uint32_t lut_shift, uint32_t bits, uint32_t mask) {
    const uint32_t slot = (uint32_t)x & mask;  // rans64.hpp:118-121
    const uint32_t key = (slot + 1u) << kSymBits;
    uint32_t p, e, hi;
    const bool near = rans_lookup_near(T, lut, lut_stride, lut_shift, slot, key, p, e, hi);
    const uint64_t top = x >> bits;
    uint64_t next = (uint64_t)((hi >> kSymBits) - (e >> kSymBits)) * top + (slot - (e >> kSymBits));  // rans64.hpp:126-134
    if (__builtin_expect(__any_sync(0xffffffffu, !near), 0)) {
        // out of line: inlined, the walk sat in the middle of the step and the common case jumped over it — a taken
        // branch and an instruction-fetch bubble (~20 cycles of a ~315-cycle step, ncu source view) on every symbol
        const ulonglong2 fixed = rans_far_step(T, key, p, e, hi, top, slot);
        next = fixed.x;
        e = (uint32_t)fixed.y;
    }
    x = next;
    // rans64.hpp:137-141: x < 2^31, written on the two halves so that ONE predicate serves the state update and
    // the word ring (the 64-bit comparison was being evaluated twice, as >= and as >)
    const bool refill = ((uint32_t)(x >> 32) | ((uint32_t)x >> 31)) == 0u;
    x = refill ? ((x << 32) | rd.next) : x;
    rd.take_if(refill);
    return e & kSymMask;
}

// rans_get for kernels that address their tables by shared-window addresses (PerLaneDenseS; lut_s = address of this
// lane's entry 0 of the midpoint table, entries 32 * sizeof(LutT) bytes apart): same lookup, same step.
template <typename LutT>
__device__ __forceinline__ uint32_t rans_get_s(uint64_t& x, WordRing& rd, const PerLaneDenseS& T, uint32_t lut_s,
                                               uint32_t lut_shift, uint32_t bits, uint32_t mask) {
    const uint32_t slot = (uint32_t)x & mask;  // rans64.hpp:118-121
    const uint32_t key = (slot + 1u) << kSymBits;
    uint32_t p;
    if (sizeof(LutT) == 1) {
        asm("ld.shared.u8 %0, [%1];" : "=r"(p) : "r"(lut_s + (slot >> lut_shift) * 32u));
    } else {
        asm("ld.shared.u16 %0, [%1];" : "=r"(p) : "r"(lut_s + (slot >> lut_shift) * 64u));
    }
    uint32_t em, e0, e1, e2;
    T.at4(p, em, e0, e1, e2);
    const bool down = e0 >= key;  // see rans_lookup_near
    const bool up = e1 < key;
    uint32_t e = down ? em : (up ? e1 : e0);
    uint32_t up_ones;
    asm("set.lt.u32.u32 %0, %1, %2;" : "=r"(up_ones) : "r"(e1), "r"(key));
    uint32_t hi = down ? e0 : e1 + ((e2 - e1) & up_ones);
    const bool near = e < key && hi >= key;
    const uint64_t top = x >> bits;
    uint64_t next = (uint64_t)((hi >> kSymBits) - (e >> kSymBits)) * top + (slot - (e >> kSymBits));  // rans64.hpp:126-134
    if (__builtin_expect(__any_sync(0xffffffffu, !near), 0)) {
        const ulonglong2 fixed = rans_far_step(T, key, p, e, hi, top, slot);
        next = fixed.x;
        e = (uint32_t)fixed.y;
    }
    x = next;
    const bool refill = ((uint32_t)(x >> 32) | ((uint32_t)x >> 31)) == 0u;
    x = refill ? ((x << 32) | rd.next) : x;
    rd.take_if(refill);
    return e & kSymMask;
}

// One warp per CTA, one stream per lane.  `rows_lo < need <= rows` selects the warps of this launch's
// table-size class (need = rows of the largest dense table among the warp's streams): the host
// launches one grid per class with the matching shared-memory size and every warp runs in exactly one.
// LutT = u8 when rows <= 256.  Dynamic shared memory: rows * 32 u32 (tables) + 32 * kRingWords u32 (word
// rings) + 32 * kDecStride u16 (symbol staging) + 128 * 32 LutT.
template <typename LutT>
__global__ void __launch_bounds__(32) k_rans_decode(const hoh_dec_stream* __restrict__ streams,
                                                    uint32_t n_streams, const uint8_t* __restrict__ in,
                                                    uint64_t in_bytes, const uint32_t* __restrict__ cumtab,
                                                    const DecMeta* __restrict__ meta,
                                                    uint16_t* __restrict__ symbols,
                                                    hoh_dec_result* __restrict__ results, uint32_t rows_lo,
                                                    uint32_t rows) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint32_t* tab = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* rings = tab + (size_t)rows * 32u;
    uint16_t* stage = reinterpret_cast<uint16_t*>(rings + 32 * kRingWords);
    LutT* lut = reinterpret_cast<LutT*>(stage + 32 * kDecStride);
    __shared__ uint64_t s_off[32];
    __shared__ uint32_t s_n[32];

    const uint32_t lane = lane_id();
    const uint32_t s = blockIdx.x * 32u + lane;
    const bool exists = s < n_streams;
    hoh_dec_stream st;
    DecMeta m;
    st.sym_off = 0;
    st.sym_cap = 0;
    m.kind = 0;
    m.n = 0;
    m.range = 1;
    m.prob_bits = 1;
    m.payload_off = 0;
    m.status = HOH_S_OK;
    m.used = 0;
    if (exists) {
        st = streams[s];
        m = meta[s];
    }
    const bool live = exists && m.kind == 2u && m.n > 0u;
    uint32_t need = live ? m.used + 3u : 0u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) need = max(need, __shfl_xor_sync(0xffffffffu, need, d));
    if (need <= rows_lo || need > rows) return;  // another class's launch (or nothing to do)
    const uint32_t my_n = live ? min(m.n, st.sym_cap) : 0u;
    s_off[lane] = st.sym_off;
    s_n[lane] = my_n;

    for (uint32_t j = 0; j < 32; j++) {
        const uint32_t sj = blockIdx.x * 32u + j;
        const bool lj = __shfl_sync(0xffffffffu, (int)live, j) != 0;
        const uint32_t uj = __shfl_sync(0xffffffffu, m.used, j);
        if (!lj) continue;
        const uint32_t* src = cumtab + (size_t)sj * kCumRow;
        for (uint32_t i = lane; i < uj + 3u; i += 32) tab[i * 32u + j] = src[i];
    }
    __syncwarp();

    const PerLaneDense T{tab, lane};
    const uint32_t bits = m.prob_bits;
    const uint32_t mask = (1u << bits) - 1u;
    const uint32_t full = 1u << bits;
    const uint32_t lut_shift = bits > 7u ? bits - 7u : 0u;
    if (live) {
        lut_build(T, lut + lane, 32u, lut_shift, m.used);
    } else {  // idle lane of a working warp: a one-entry table so that its (discarded) lookups stay in bounds
        tab[lane] = 0u;
        tab[32u + lane] = 0u;
        tab[64u + lane] = full << kSymBits;
        tab[96u + lane] = 0xffffffffu;
        for (uint32_t j = 0; j < (uint32_t)kLutSize; j++) lut[j * 32u + lane] = (LutT)1;
    }
    __syncwarp();
    uint32_t n_max = my_n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, d));

    WordRing rd;
    rd.open(in, in_bytes, live ? m.payload_off : 0ull, rings + lane * kRingWords);
    uint64_t x;
    {  // rans64.hpp:107-116: state = first two payload words, low word first
        const uint32_t lo = rd.next;
        rd.take_if(true);
        const uint32_t hi = rd.next;
        rd.take_if(true);
        x = live ? ((uint64_t)lo | ((uint64_t)hi << 32)) : kRansL;
    }
    uint16_t* my_row = stage + lane * kDecStride;
    const PerLaneDenseS TS{(uint32_t)__cvta_generic_to_shared(tab + lane)};  // the loop's view of the table: see PerLaneDenseS
    const uint32_t lut_s = (uint32_t)__cvta_generic_to_shared(lut + lane);
    const uint32_t chunks = (n_max + kDecChunk - 1) / kDecChunk;
    // The encoder starts from 2^31 (rans64.hpp:65) and decoding undoes its steps one by one, so after the last
    // symbol of a sound stream the state is 2^31 again: the only integrity check the format offers (it carries no
    // checksum).  The state is sampled in the chunk where the lane's stream ends (a warp-uniform choice of loop).
    uint64_t x_end = kRansL;
    for (uint32_t chunk = 0; chunk < chunks; chunk++) {
        __syncwarp();
        const uint32_t left = my_n - min(my_n, chunk * (uint32_t)kDecChunk);  // symbols of mine from this chunk on
        if (__any_sync(0xffffffffu, left >= 1u && left <= (uint32_t)kDecChunk)) {
            for (uint32_t k0 = 0; k0 < (uint32_t)kDecChunk; k0 += kTopUp) {
                rd.top_up();
#pragma unroll
                for (uint32_t k = k0; k < k0 + kTopUp; k++) {
                    my_row[k] = (uint16_t)rans_get_s<LutT>(x, rd, TS, lut_s, lut_shift, bits, mask);
                    x_end = left == k + 1u ? x : x_end;
                }
            }
        } else {
            for (uint32_t k0 = 0; k0 < (uint32_t)kDecChunk; k0 += kTopUp) {
                rd.top_up();
#pragma unroll
                for (uint32_t k = k0; k < k0 + kTopUp; k++)
                    my_row[k] = (uint16_t)rans_get_s<LutT>(x, rd, TS, lut_s, lut_shift, bits, mask);
            }
        }
        __syncwarp();
        stage_store_chunk(stage, symbols, s_off, s_n, chunk);
    }
    if (live && my_n == m.n && x_end != kRansL && results[s].status == HOH_S_OK) results[s].status = HOH_S_BAD_STATE;
}

// -------------------------------------------------------------------------------------------------
// Static-table sweep (config 4): rans64.hpp loops with one table shared by every stream.
// Streams are implicit: stream i = symbols [i*stream_len, ...).  4 warps per CTA share the table.
// -------------------------------------------------------------------------------------------------
constexpr int kStaticWarps = 4;

template <int DIV>  // how x / freq is taken (rans_put), chosen by the host from prob_bits
__global__ void __launch_bounds__(kStaticWarps * 32) k_rans_encode_static(
    const uint16_t* __restrict__ symbols, uint64_t n_total, uint32_t stream_len,
    const uint32_t* __restrict__ cum_g, uint32_t range, uint32_t bits, uint8_t* __restrict__ out,
    uint32_t slab_bytes, uint32_t* __restrict__ payload_bytes) {
    __shared__ uint32_t s_cum[HOH_MAX_RANGE + 8];
    __shared__ __align__(16) uint16_t s_stage[kStaticWarps][32 * kSymStride];
    __shared__ uint64_t s_off[kStaticWarps][32];
    __shared__ uint32_t s_n[kStaticWarps][32];
    for (uint32_t i = threadIdx.x; i <= range; i += blockDim.x) s_cum[i] = cum_g[i];
    const uint32_t w = threadIdx.x >> 5, lane = lane_id();
    const uint64_t n_streams = (n_total + stream_len - 1) / stream_len;
    const uint64_t s = ((uint64_t)blockIdx.x * kStaticWarps + w) * 32u + lane;
    const bool live = s < n_streams;
    const uint64_t first = s * stream_len;
    const uint32_t my_n = live ? (uint32_t)min((uint64_t)stream_len, n_total - first) : 0u;
    s_off[w][lane] = live ? first : 0ull;
    s_n[w][lane] = my_n;
    __syncthreads();
    if (__ballot_sync(0xffffffffu, live) == 0u) return;
    const SharedTable<uint32_t> T{s_cum};
    uint16_t* stage = s_stage[w];
    const bool fits = (uint64_t)slab_bytes >= rans_words_bound(my_n, bits) * 4u;
    uint32_t* words = reinterpret_cast<uint32_t*>(out + (live ? s : 0) * slab_bytes);
    const uint32_t cap_words = slab_bytes / 4u;
    uint32_t widx = cap_words;
    uint64_t x = kRansL;
    const uint32_t run_n = (live && fits) ? my_n : 0u;
    uint32_t n_max = run_n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, d));
    const uint16_t* my_row = stage + lane * kSymStride;
    const uint32_t full = 1u << bits;
    const uint32_t zero = slab_bytes & 1u;  // slabs are whole words: 0 at run time, unknown to the compiler
    for (int chunk = (int)((n_max + kChunk - 1) / kChunk) - 1; chunk >= 0; chunk--) {
        __syncwarp();
        stage_load_chunk(stage, symbols, s_off[w], s_n[w], (uint32_t)chunk);
        stage_wait();
        const uint32_t base = (uint32_t)chunk * kChunk;
        // groups of the chunk from the last to the first; the preparation of the next group (table rows, reciprocals:
        // independent of the state) is woven into the serial steps of the current one, as in k_rans_encode
        auto prepare_one = [&](int k, uint32_t dep, uint32_t& o_start, uint32_t& o_freq, double& o_inv) {
            const bool on = base + (uint32_t)k < run_n;
            const uint32_t sym = on ? min((uint32_t)my_row[k] | dep, range - 1u) : 0u;
            const uint32_t c0 = T.cum(sym), c1 = T.cum(sym + 1u);
            o_start = on ? c0 : 0u;
            o_freq = on ? c1 - c0 : full;
            o_inv = recip_low(o_freq);
        };
        auto run_prepare = [&](const uint32_t(&r_start)[kGroup], const uint32_t(&r_freq)[kGroup], const double(&r_inv)[kGroup],
                               int k0_next, uint32_t(&p_start)[kGroup], uint32_t(&p_freq)[kGroup], double(&p_inv)[kGroup]) {
            // ptxas undoes the weaving (it sinks all eight preparations below the eight steps) unless the two streams
            // are tied together by false dependencies (0 at run time): the preparation of symbol j takes a bit of the
            // state before step j, and step j - 2 one of its reciprocal.  Worth 7 % here, where a warp has a scheduler
            // almost to itself (8.68 -> 8.10 ms at 2^30 symbols); nothing in k_rans_encode, whose 2.4 warps per
            // scheduler already fill each other's stalls.
            uint32_t tie1 = 0, tie2 = 0;
#pragma unroll
            for (int j = kGroup - 1; j >= 0; j--) {
                const uint32_t before = (uint32_t)x & zero;
                x = rans_put<DIV>(x, r_start[j], r_freq[j] | tie2, r_inv[j], bits, words, widx);
                prepare_one(k0_next + j, before, p_start[j], p_freq[j], p_inv[j]);
                tie2 = tie1;
                tie1 = (uint32_t)__double_as_longlong(p_inv[j]) & zero;
            }
        };
        uint32_t a_start[kGroup], a_freq[kGroup], b_start[kGroup], b_freq[kGroup];
        double a_inv[kGroup], b_inv[kGroup];
#pragma unroll
        for (int j = 0; j < kGroup; j++) prepare_one(kChunk - kGroup + j, 0u, a_start[j], a_freq[j], a_inv[j]);
        static_assert((kChunk / kGroup) % 2 == 0 && kChunk >= 2 * kGroup, "groups of a chunk are coded in pairs");
#pragma unroll 1
        for (int k0 = kChunk - kGroup; k0 >= 3 * kGroup; k0 -= 2 * kGroup) {
            run_prepare(a_start, a_freq, a_inv, k0 - kGroup, b_start, b_freq, b_inv);
            run_prepare(b_start, b_freq, b_inv, k0 - 2 * kGroup, a_start, a_freq, a_inv);
        }
        run_prepare(a_start, a_freq, a_inv, 0, b_start, b_freq, b_inv);  // a = group at kGroup, b = the chunk's first
#pragma unroll
        for (int j = kGroup - 1; j >= 0; j--)
            x = rans_put<DIV>(x, b_start[j], b_freq[j], b_inv[j], bits, words, widx);
    }
    if (live) {
        if (fits) {
            widx -= 2;
            words[widx] = (uint32_t)x;
            words[widx + 1] = (uint32_t)(x >> 32);
            payload_bytes[s] = (cap_words - widx) * 4u;
        } else {
            payload_bytes[s] = 0xffffffffu;
        }
    }
}

constexpr int kStaticDecWarps = 2;

__global__ void __launch_bounds__(kStaticDecWarps * 32) k_rans_decode_static(
    const uint8_t* __restrict__ in, uint32_t slab_bytes, const uint32_t* __restrict__ payload_bytes,
    uint64_t n_total, uint32_t stream_len, const uint32_t* __restrict__ cum_g, uint32_t range,
    uint32_t bits, uint16_t* __restrict__ symbols) {
    __shared__ uint32_t s_dense[HOH_MAX_RANGE + 8];
    __shared__ uint32_t s_used;
    __shared__ __align__(16) uint16_t s_stage[kStaticDecWarps][32 * kDecStride];
    __shared__ __align__(16) uint32_t s_rings[kStaticDecWarps][32 * kRingWords];
    __shared__ uint64_t s_off[kStaticDecWarps][32];
    __shared__ uint32_t s_n[kStaticDecWarps][32];
    __shared__ uint32_t s_cum[HOH_MAX_RANGE + 8];
    __shared__ uint16_t s_lut[kLutSize];
    for (uint32_t i = threadIdx.x; i <= range; i += blockDim.x) s_cum[i] = cum_g[i];
    __syncthreads();
    const uint32_t lut_shift = bits > 7u ? bits - 7u : 0u;
    const SharedDense T{s_dense};
    if (threadIdx.x == 0) {  // dense table, physical layout as in k_parse_streams
        uint32_t d = 0;
        s_dense[0] = 0u;
        for (uint32_t i = 0; i < range; i++)
            if (s_cum[i + 1] != s_cum[i]) s_dense[1u + d++] = (s_cum[i] << kSymBits) | i;
        s_dense[d + 1] = s_cum[range] << kSymBits;
        s_dense[d + 2] = 0xffffffffu;
        s_used = d;
        if (d) lut_build(T, s_lut, 1u, lut_shift, d);
    }
    const uint32_t w = threadIdx.x >> 5, lane = lane_id();
    const uint64_t n_streams = (n_total + stream_len - 1) / stream_len;
    const uint64_t s = ((uint64_t)blockIdx.x * kStaticDecWarps + w) * 32u + lane;
    const bool exists = s < n_streams;
    const uint64_t first = s * stream_len;
    const uint32_t pb = exists ? payload_bytes[s] : 0u;
    const bool live = exists && pb >= 8u && pb <= slab_bytes;
    const uint32_t my_n = live ? (uint32_t)min((uint64_t)stream_len, n_total - first) : 0u;
    s_off[w][lane] = live ? first : 0ull;
    s_n[w][lane] = my_n;
    __syncthreads();
    const uint32_t used = s_used;
    if (used == 0u || __ballot_sync(0xffffffffu, live) == 0u) return;
    const uint32_t mask = (1u << bits) - 1u;
    uint32_t n_max = my_n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, d));
    WordRing rd;
    const uint64_t total_bytes = n_streams * (uint64_t)slab_bytes;
    rd.open(in, total_bytes, live ? (s + 1) * (uint64_t)slab_bytes - pb : 0ull, s_rings[w] + lane * kRingWords);
    uint64_t x;
    {
        const uint32_t lo = rd.next;
        rd.take_if(true);
        const uint32_t hi = rd.next;
        rd.take_if(true);
        x = live ? ((uint64_t)lo | ((uint64_t)hi << 32)) : kRansL;
    }
    uint16_t* stage = s_stage[w];
    uint16_t* my_row = stage + lane * kDecStride;
    const uint32_t chunks = (n_max + kDecChunk - 1) / kDecChunk;
    for (uint32_t chunk = 0; chunk < chunks; chunk++) {
        __syncwarp();
        for (uint32_t k0 = 0; k0 < (uint32_t)kDecChunk; k0 += kTopUp) {
            rd.top_up();
#pragma unroll
            for (uint32_t k = k0; k < k0 + kTopUp; k++)
                my_row[k] = (uint16_t)rans_get(x, rd, T, s_lut, 1u, lut_shift, bits, mask);
        }
        __syncwarp();
        stage_store_chunk(stage, symbols, s_off[w], s_n[w], chunk);
    }
}

// Static decode with the reference's own lookup structure.  With ONE table for all streams the 2^prob_bits-entry
// slot -> symbol table of entropy_decoding.hpp:262-267 fits shared memory (prob_bits <= 15: at most 32 KB of
// bytes for an 8-bit alphabet) when a whole CTA of 8 warps shares it, and a symbol costs two dependent
// shared-memory reads (symbol, then its packed start | freq << 16) with no search at all — the midpoint table
// of the per-stream decoder degenerates here, because at 12 bits many symbols share a bucket.
constexpr int kStaticDirectWarps = 8;

template <typename SymT>
__global__ void __launch_bounds__(kStaticDirectWarps * 32) k_rans_decode_static_direct(
    const uint8_t* __restrict__ in, uint32_t slab_bytes, const uint32_t* __restrict__ payload_bytes,
    uint64_t n_total, uint32_t stream_len, const uint32_t* __restrict__ cum_g, uint32_t range,
    uint32_t bits, uint16_t* __restrict__ symbols) {
    extern __shared__ __align__(16) uint8_t sd_smem[];
    uint32_t* s_rings = reinterpret_cast<uint32_t*>(sd_smem);                              // [warp][32 * kRingWords]
    uint16_t* s_stage = reinterpret_cast<uint16_t*>(s_rings + kStaticDirectWarps * 32 * kRingWords);  // [warp][32 * kDecStride]
    uint32_t* s_info = reinterpret_cast<uint32_t*>(s_stage + kStaticDirectWarps * 32 * kDecStride);   // [range]
    SymT* s_c2s = reinterpret_cast<SymT*>(s_info + HOH_MAX_RANGE);                           // [1 << bits]
    __shared__ uint64_t s_off[kStaticDirectWarps][32];
    __shared__ uint32_t s_n[kStaticDirectWarps][32];
    const uint32_t total = 1u << bits;
    for (uint32_t i = threadIdx.x; i < range; i += blockDim.x) s_info[i] = cum_g[i] | ((cum_g[i + 1] - cum_g[i]) << 16);
    for (uint32_t slot = threadIdx.x; slot < total; slot += blockDim.x) {  // largest symbol with cum <= slot
        uint32_t lo = 0, hi = range;  // cum_g[lo] <= slot < cum_g[hi] (cum_g[range] = total for a valid table)
        while (hi - lo > 1u) {
            const uint32_t mid = (lo + hi) >> 1;
            if (cum_g[mid] <= slot) lo = mid;
            else hi = mid;
        }
        s_c2s[slot] = (SymT)lo;
    }
    const uint32_t w = threadIdx.x >> 5, lane = lane_id();
    const uint64_t n_streams = (n_total + stream_len - 1) / stream_len;
    const uint64_t s = ((uint64_t)blockIdx.x * kStaticDirectWarps + w) * 32u + lane;
    const bool exists = s < n_streams;
    const uint64_t first = s * stream_len;
    const uint32_t pb = exists ? payload_bytes[s] : 0u;
    const bool live = exists && pb >= 8u && pb <= slab_bytes;
    const uint32_t my_n = live ? (uint32_t)min((uint64_t)stream_len, n_total - first) : 0u;
    s_off[w][lane] = live ? first : 0ull;
    s_n[w][lane] = my_n;
    __syncthreads();
    if (__ballot_sync(0xffffffffu, live) == 0u) return;
    const uint32_t mask = total - 1u;
    uint32_t n_max = my_n;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, d));
    WordRing rd;
    const uint64_t total_bytes = n_streams * (uint64_t)slab_bytes;
    rd.open(in, total_bytes, live ? (s + 1) * (uint64_t)slab_bytes - pb : 0ull, s_rings + (w * 32u + lane) * kRingWords);
    uint64_t x;
    {
        const uint32_t lo = rd.next;
        rd.take_if(true);
        const uint32_t hi = rd.next;
        rd.take_if(true);
        x = live ? ((uint64_t)lo | ((uint64_t)hi << 32)) : kRansL;
    }
    uint16_t* stage = s_stage + w * 32u * kDecStride;
    uint16_t* my_row = stage + lane * kDecStride;
    const uint32_t chunks = (n_max + kDecChunk - 1) / kDecChunk;
    for (uint32_t chunk = 0; chunk < chunks; chunk++) {
        __syncwarp();
        for (uint32_t k0 = 0; k0 < (uint32_t)kDecChunk; k0 += kTopUp) {
            rd.top_up();
#pragma unroll
            for (uint32_t k = k0; k < k0 + kTopUp; k++) {
                const uint32_t slot = (uint32_t)x & mask;  // rans64.hpp:118-121
                const uint32_t sym = s_c2s[slot];
                const uint32_t info = s_info[sym];
                x = (uint64_t)(info >> 16) * (x >> bits) + (slot - (info & 0xffffu));  // rans64.hpp:126-134
                const bool refill = ((uint32_t)(x >> 32) | ((uint32_t)x >> 31)) == 0u;       // :137-141, x < 2^31
                x = refill ? ((x << 32) | rd.next) : x;
                rd.take_if(refill);
                my_row[k] = (uint16_t)sym;
            }
        }
        __syncwarp();
        stage_store_chunk(stage, symbols, s_off[w], s_n[w], chunk);
    }
}

// =================================================================================================
// Offsets and gather — "stream-offset prefix sums with warp shuffles" + the final gather.
// =================================================================================================
// Exclusive scan of results[i].size into off[0..n]; one CTA of 1024 threads, serial over tiles of 1024.
__global__ void __launch_bounds__(1024) k_scan_sizes(const hoh_stream_result* __restrict__ results,
                                                     uint32_t n, uint64_t* __restrict__ off) {
    __shared__ uint64_t warp_tot[32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const uint32_t lane = lane_id(), w = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint64_t v = (i < n && results[i].status == HOH_S_OK) ? results[i].size : 0ull;
        uint64_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t o = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += o;
        }
        if (lane == 31) warp_tot[w] = incl;
        __syncthreads();
        if (w == 0) {
            uint64_t t = warp_tot[lane];
            uint64_t ti = t;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint64_t o = __shfl_up_sync(0xffffffffu, ti, d);
                if ((int)lane >= d) ti += o;
            }
            warp_tot[lane] = ti - t;  // exclusive over warps
        }
        __syncthreads();
        const uint64_t c = carry;
        if (i < n) off[i] = c + warp_tot[w] + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + warp_tot[w] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) off[n] = carry;
}

// Copies every stream's bytes to its packed position.  One CTA per stream; destination-aligned
// 32-bit stores fed by two aligned source loads and a funnel shift.
__global__ void __launch_bounds__(256) k_gather_streams(const hoh_stream_result* __restrict__ results,
                                                        const uint8_t* __restrict__ src,
                                                        const uint64_t* __restrict__ off, uint8_t* __restrict__ dst,
                                                        uint64_t dst_cap) {
    const hoh_stream_result r = results[blockIdx.x];
    if (r.status != HOH_S_OK || r.size == 0) return;
    const uint64_t d0 = off[blockIdx.x];
    if (d0 + r.size > dst_cap) return;
    const uint8_t* s = src + r.start;
    uint8_t* d = dst + d0;
    // head: bytes until d is 4-aligned
    const uint32_t lead = min((uint32_t)((4u - (uint32_t)(reinterpret_cast<uint64_t>(d) & 3u)) & 3u), r.size);
    if (threadIdx.x < lead) d[threadIdx.x] = s[threadIdx.x];
    const uint32_t words = (r.size - lead) / 4u;
    const uint8_t* sb = s + lead;
    const uint64_t sa = reinterpret_cast<uint64_t>(sb);
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~3ull);
    const uint32_t sh = (uint32_t)(sa & 3ull) * 8u;
    uint32_t* dw = reinterpret_cast<uint32_t*>(d + lead);
    // four independent words per thread and trip: the copy is bound by bytes in flight, not by instructions
    uint32_t i = threadIdx.x;
    if (sh == 0) {
        for (; i + 3u * blockDim.x < words; i += 4u * blockDim.x) {
            const uint32_t a = sw[i], b = sw[i + blockDim.x], c = sw[i + 2u * blockDim.x], e = sw[i + 3u * blockDim.x];
            dw[i] = a;
            dw[i + blockDim.x] = b;
            dw[i + 2u * blockDim.x] = c;
            dw[i + 3u * blockDim.x] = e;
        }
        for (; i < words; i += blockDim.x) dw[i] = sw[i];
    } else {
        for (; i + 3u * blockDim.x < words; i += 4u * blockDim.x) {
            const uint32_t a0 = sw[i], a1 = sw[i + 1u], b0 = sw[i + blockDim.x], b1 = sw[i + blockDim.x + 1u];
            const uint32_t c0 = sw[i + 2u * blockDim.x], c1 = sw[i + 2u * blockDim.x + 1u];
            const uint32_t e0 = sw[i + 3u * blockDim.x], e1 = sw[i + 3u * blockDim.x + 1u];
            dw[i] = __funnelshift_r(a0, a1, sh);
            dw[i + blockDim.x] = __funnelshift_r(b0, b1, sh);
            dw[i + 2u * blockDim.x] = __funnelshift_r(c0, c1, sh);
            dw[i + 3u * blockDim.x] = __funnelshift_r(e0, e1, sh);
        }
        for (; i < words; i += blockDim.x) dw[i] = __funnelshift_r(sw[i], sw[i + 1], sh);
    }
    const uint32_t done = lead + words * 4u;
    if (threadIdx.x < r.size - done) d[done + threadIdx.x] = s[done + threadIdx.x];
}

// =================================================================================================
// Predictor primitives — predictor_operations.hpp (u16 forms, C int promotion semantics)
// =================================================================================================
__device__ __forceinline__ int p_mid(int a, int b) { return a + (b - a) / 2; }  // :8-10, truncating
// x % c for c a power of two, with C's truncation for negative x (what the reference's `% centre` does with an
// out-of-range pixel).  c is a run-time value in these kernels, so `%` itself compiles to a software division
// (~14 instructions; it was a quarter of k_section_costs).
__device__ __forceinline__ int mod_pow2(int x, int c) {
    const int r = abs(x) & (c - 1);
    return x < 0 ? -r : r;
}
__device__ __forceinline__ int p_med(int a, int b, int c) {                     // :37-60
    const int lo = min(a, b), hi = max(a, b);
    return c < lo ? lo : (c > hi ? hi : c);
}
__device__ __forceinline__ int p_avg3(int a, int b, int c) { return (a + b + c) / 3; }  // :66-68
__device__ __forceinline__ int p_paeth(int A, int B, int C) {                            // :89-106
    const int p = A + B - C;
    const int da = abs(A - p), db = abs(B - p), dc = abs(C - p);
    if (da < db) return da < dc ? A : C;
    return db < dc ? B : C;
}
// median(T, L, (u16)(T + L - TL)): the gradient wraps to u16 before the median (SURVEY H6)
__device__ __forceinline__ int p_med_grad(int T, int L, int TL) { return p_med(T, L, (T + L - TL) & 0xffff); }
// The same on two u16 lanes of one register (sm_100a has native 16x2 integer add / min / max:
// VIADD.16x2, VIMNMX.U16x2, VIADDMNMX.U16x2).  The lanes wrap modulo 2^16 exactly like the reference's
// uint16_t gradient, and the comparisons are unsigned, so this IS predictor_operations.hpp:37-60 on
// (T, L, (u16)(T + L - TL)) for two channels at once.
__device__ __forceinline__ uint32_t p_med_grad2(uint32_t T, uint32_t L, uint32_t TL) {
    const uint32_t lo = __vminu2(T, L), hi = __vmaxu2(T, L);
    const uint32_t grad = __vsub2(__vadd2(T, L), TL);
    return __vmaxu2(lo, __vminu2(hi, grad));
}
constexpr uint32_t kHalfRB = 256u | (256u << 16);   // c/2 of the two 9-bit planes (R-G, B-G), one per lane
constexpr uint32_t kMaskRB = 511u | (511u << 16);
// pixel 0x00BBGGRR -> g and (R-G+256 | B-G+256 << 16)   (channel.hpp:75-77)
__device__ __forceinline__ void planes2_of(uint32_t p, uint32_t& g, uint32_t& rb) {
    g = (p >> 8) & 255u;
    rb = __vadd2(__vsub2(p & 0x00ff00ffu, g * 0x00010001u), kHalfRB);
}

// =================================================================================================
// Colour transform — channel.hpp:73-79 and its algebraic inverse (SURVEY D4)
// =================================================================================================
__global__ void k_subtract_green(const uint8_t* __restrict__ rgb, uint64_t pixels, uint16_t* __restrict__ g,
                                 uint16_t* __restrict__ rg, uint16_t* __restrict__ bg) {
    for (uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; p < pixels; p += (uint64_t)gridDim.x * blockDim.x) {
        const int r = rgb[3 * p], gg = rgb[3 * p + 1], b = rgb[3 * p + 2];
        g[p] = (uint16_t)gg;
        rg[p] = (uint16_t)(r - gg + 256);
        bg[p] = (uint16_t)(b - gg + 256);
    }
}

__global__ void k_add_green(const uint16_t* __restrict__ g, const uint16_t* __restrict__ rg,
                            const uint16_t* __restrict__ bg, uint64_t pixels, uint8_t* __restrict__ rgb) {
    for (uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; p < pixels; p += (uint64_t)gridDim.x * blockDim.x) {
        const int gg = g[p];
        rgb[3 * p] = (uint8_t)((rg[p] + gg - 256) & 255);
        rgb[3 * p + 1] = (uint8_t)gg;
        rgb[3 * p + 2] = (uint8_t)((bg[p] + gg - 256) & 255);
    }
}

// =================================================================================================
// channelpredict_fastpath — prediction.hpp:6-44.  Per-pixel data parallel on planes.
// =================================================================================================
// out_stride: u16 elements between consecutive residual planes (>= w*h)
constexpr int kFastpathBand = 16;  // rows per CTA trip: the row above travels down in registers

__global__ void k_predict_fastpath(const uint16_t* __restrict__ planes, uint64_t n_planes, int w, int h,
                                   int depth, uint16_t* __restrict__ resid, uint64_t out_stride) {
    const int c = 1 << depth, half = c >> 1;
    // grid-stride over (plane, band of rows); a thread owns a column of the band: one new pixel and its left
    // neighbour per row, T and TL come from the previous row's registers
    const uint32_t bands = ((uint32_t)h + kFastpathBand - 1u) / kFastpathBand;
    const uint64_t jobs = n_planes * bands;
    for (uint64_t job = blockIdx.x; job < jobs; job += gridDim.x) {
        const uint64_t pl = job / bands;
        const int y0 = (int)(job % bands) * kFastpathBand, y1 = min(y0 + kFastpathBand, h);
        const uint16_t* base = planes + pl * (uint64_t)w * h;
        uint16_t* obase = resid + pl * out_stride;
        for (int x = threadIdx.x; x < w; x += blockDim.x) {
            int T = y0 ? base[(size_t)(y0 - 1) * w + x] : half;
            int TL = (x && y0) ? base[(size_t)(y0 - 1) * w + x - 1] : half;
            for (int y = y0; y < y1; y++) {
                const uint16_t* p = base + (size_t)y * w + x;
                const int v = p[0];
                const int L = x ? p[-1] : half;
                obase[(size_t)y * w + x] = (uint16_t)((v - p_med_grad(T, L, TL) + half + c) & (c - 1));  // numerator > 0
                T = v;
                TL = x ? L : half;
            }
        }
    }
}

// Raster-serial inverse of the above for one plane per thread (used when back-references are
// present: unprediction.hpp:63-65 makes a pixel depend on an arbitrary earlier one).
__global__ void k_unpredict_fastpath_serial(const uint16_t* __restrict__ resid, uint64_t n_planes, int w, int h,
                                            int depth, const uint16_t* __restrict__ backref,
                                            uint16_t* __restrict__ planes) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    const int c = 1 << depth, half = c >> 1;
    const uint64_t per = (uint64_t)w * h;
    const uint16_t* r = resid + p * per;
    const uint16_t* br = backref ? backref + p * per : nullptr;
    uint16_t* o = planes + p * per;
    uint64_t k = 0;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const uint64_t at = (uint64_t)y * w + x;
            if (br && br[at]) {
                o[at] = o[at - br[at]];
                continue;
            }
            const int L = x ? o[at - 1] : half;
            const int T = y ? o[at - w] : half;
            const int TL = (x && y) ? o[at - w - 1] : half;
            o[at] = (uint16_t)(((int)r[k++] + p_med_grad(T, L, TL) - half) & (c - 1));
        }
}

// Wavefront inverse of channelpredict_fastpath on planes: one warp per plane, lane = row inside a
// 32-row band, lane r works on column t - r at step t, T comes from lane r-1 by shuffle.
__global__ void __launch_bounds__(128) k_unpredict_fastpath_wave(const uint16_t* __restrict__ resid,
                                                                 uint64_t n_planes, int w, int h, int depth,
                                                                 uint16_t* __restrict__ planes) {
    extern __shared__ uint16_t s_rows[];  // 4 warps * w: last row of the previous band
    const uint32_t wid = threadIdx.x >> 5, lane = lane_id();
    const uint64_t p = (uint64_t)blockIdx.x * 4u + wid;
    if (p >= n_planes) return;
    const int c = 1 << depth, half = c >> 1;
    const uint64_t per = (uint64_t)w * h;
    const uint16_t* r = resid + p * per;
    uint16_t* o = planes + p * per;
    uint16_t* carry = s_rows + (size_t)wid * w;
    for (int band = 0; band * 32 < h; band++) {
        const int y = band * 32 + (int)lane;
        const bool row_ok = y < h;
        int left = half, top_left = half, mine = half;
        for (int t = 0; t < w + 31; t++) {
            const int x = t - (int)lane;
            int top = __shfl_up_sync(0xffffffffu, mine, 1);
            if (lane == 0) top = (band && x >= 0 && x < w) ? carry[x] : half;
            if (y == 0) top = half;
            if (row_ok && x >= 0 && x < w) {
                if (x == 0) {
                    left = half;
                    top_left = half;
                }
                if (y == 0) top_left = half;
                const int v = ((int)r[(uint64_t)y * w + x] + p_med_grad(top, left, top_left) - half) & (c - 1);
                o[(uint64_t)y * w + x] = (uint16_t)v;
                mine = v;
                left = v;
                top_left = top;
                if (lane == 31) carry[x] = (uint16_t)v;
            }
        }
        __syncwarp();
    }
}

// =================================================================================================
// channelpredict_all / unpredict_all — prediction.hpp:153-229, unprediction.hpp:6-91.
// One plane per thread, raster order (the chain is serial: SURVEY H4); row state in global scratch.
// =================================================================================================
struct Cand {
    int v[16];
};
// The 16 candidate predictions (prediction.hpp:190-207).  section_order selects
// channelpredict_section's paeth(L, T, TL) argument order (prediction.hpp:126).
__device__ __forceinline__ void candidates(int L, int T, int TL, int TR, bool section_order, Cand& k) {
    k.v[0] = L;
    k.v[1] = T;
    k.v[2] = TL;
    k.v[3] = TR;
    k.v[4] = p_med_grad(T, L, TL);
    k.v[5] = p_mid(L, T);
    k.v[6] = p_mid(L, TL);
    k.v[7] = p_mid(TL, T);
    k.v[8] = p_mid(T, TR);
    k.v[9] = section_order ? p_paeth(L, T, TL) : p_paeth(L, TL, T);
    k.v[10] = p_avg3(L, L, TL);
    k.v[11] = p_avg3(L, TL, TL);
    k.v[12] = p_avg3(TL, TL, T);
    k.v[13] = p_avg3(TL, T, T);
    k.v[14] = p_avg3(T, T, TR);
    k.v[15] = p_avg3(T, TR, TR);
}
__device__ __forceinline__ int cand_at(const Cand& k, int j) {
    int r = k.v[0];
#pragma unroll
    for (int i = 1; i < 16; i++) r = (j == i) ? k.v[i] : r;
    return r;
}
// prediction.hpp:138-146: lowest index wins ties, stays 0 when nothing beats 2*c
__device__ __forceinline__ int pick_best(int v, const Cand& k, uint32_t mask, int c) {
    // as a minimum over keys error << 4 | index (a forbidden candidate's key is INT_MAX): the smallest error wins and
    // among equal errors the lowest index, which is what the reference's ascending walk with a strict `<` keeps
    int key = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < 16; j++) key = min(key, ((mask >> j) & 1u) ? abs(v - k.v[j]) * 16 + j : 0x7fffffff);
    return (key >> 4) < 2 * c ? (key & 15) : 0;
}

// pick_best for a walk that keeps the same mask for a whole grid cell: the mask is folded once per cell into 16
// additive biases (j for an allowed candidate, j + 2^30 for a forbidden one), after which a candidate costs a
// subtract, an absolute value, a multiply-add and a minimum.  Same answer as pick_best: smallest error, lowest
// index among equals, 0 when no allowed candidate has an error below 2c.
struct MaskBias {
    int jb[16];
};
__device__ __forceinline__ void mask_bias(uint32_t mask, MaskBias& m) {
#pragma unroll
    for (int j = 0; j < 16; j++) m.jb[j] = ((mask >> j) & 1u) ? j : (0x40000000 | j);
}
__device__ __forceinline__ int pick_best_biased(int v, const Cand& k, const MaskBias& m, int c) {
    int key = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < 16; j++) key = min(key, abs(v - k.v[j]) * 16 + m.jb[j]);
    return (key >> 4) < 2 * c ? (key & 15) : 0;
}

// cand_at / pick_best_biased with the selects and minima arranged as trees (depth 4 instead of 15): the walks are
// bound by the dependent chain of a pixel, and both sit on it (the index comes from the previous pixel's argmin).
__device__ __forceinline__ int cand_at_tree(const Cand& k, int j) {
    const bool b0 = j & 1, b1 = j & 2, b2 = j & 4, b3 = j & 8;
    int a[8], b[4];
#pragma unroll
    for (int i = 0; i < 8; i++) a[i] = b0 ? k.v[2 * i + 1] : k.v[2 * i];
#pragma unroll
    for (int i = 0; i < 4; i++) b[i] = b1 ? a[2 * i + 1] : a[2 * i];
    const int c0 = b2 ? b[1] : b[0], c1 = b2 ? b[3] : b[2];
    return b3 ? c1 : c0;
}
__device__ __forceinline__ int pick_best_biased_tree(int v, const Cand& k, const MaskBias& m, int c) {
    int key[16];
#pragma unroll
    for (int j = 0; j < 16; j++) key[j] = abs(v - k.v[j]) * 16 + m.jb[j];
#pragma unroll
    for (int d = 8; d > 0; d >>= 1)
#pragma unroll
        for (int j = 0; j < d; j++) key[j] = min(key[j], key[j + d]);
    return (key[0] >> 4) < 2 * c ? (key[0] & 15) : 0;
}

// state per plane in global scratch: top[w] u16 followed by bp[w] u8
template <bool INVERSE>
__global__ void __launch_bounds__(64) k_raster_walk(const uint16_t* __restrict__ in, uint64_t n_planes, int w,
                                                    int h, int depth, int x_tiles, int y_tiles,
                                                    const uint16_t* __restrict__ tile_maps,
                                                    const uint16_t* __restrict__ backref,
                                                    uint16_t* __restrict__ out, uint16_t* __restrict__ top_s,
                                                    uint8_t* __restrict__ bp_s, uint64_t out_stride) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    const int c = 1 << depth, half = c >> 1;
    const int tw = (w + x_tiles - 1) / x_tiles, th = (h + y_tiles - 1) / y_tiles;
    const uint64_t per = (uint64_t)w * h;
    const uint16_t* src = in + p * per;
    const uint16_t* br = (INVERSE && backref) ? backref + p * per : nullptr;
    uint16_t* dst = out + p * out_stride;
    const uint16_t* tmap = tile_maps + p * (uint64_t)x_tiles * y_tiles;
    uint16_t* top = top_s + p * (uint64_t)w;
    uint8_t* bp = bp_s + p * (uint64_t)w;
    for (int i = 0; i < w; i++) {
        top[i] = (uint16_t)half;
        bp[i] = 4;
    }
    uint64_t next_resid = 0;
    for (int y = 0; y < h; y++) {
        int left = half, left_top = half;
        int bp_left = bp[w - 1];  // bp[(x-1) mod w] for x == 0: last column, still the previous row's
        const bool last_row = y + 1 >= h;
        const uint16_t* mrow = tmap + (size_t)((y + 1) / th) * x_tiles;
        int first_of_row = 0;
        MaskBias mb;
        int in_cell = tw;
        for (int x = 0; x < w; x++) {
            if (in_cell == tw) {  // a new grid cell of the row below: fold its mask once
                in_cell = 0;
                mask_bias(last_row ? 0u : *mrow++, mb);
            }
            in_cell++;
            const uint64_t at = (uint64_t)y * w + x;
            // TR of the last column = top[0], which already holds this row's first pixel
            const int tr = (x + 1 < w) ? top[x + 1] : (w > 1 ? first_of_row : top[0]);
            const int t = top[x];
            Cand k;
            candidates(left, t, left_top, tr, false, k);
            const int bpx = bp[x];
            const int pred = p_mid(cand_at(k, bpx), cand_at(k, bp_left));
            int v;
            if (!INVERSE) {
                v = src[at];
                dst[at] = (uint16_t)mod_pow2(v - pred + half + c, c);  // prediction.hpp:208
            } else if (br && br[at]) {
                v = dst[at - br[at]];  // unprediction.hpp:63-65
                dst[at] = (uint16_t)v;
            } else {
                const uint32_t tval = (uint32_t)((int)src[next_resid++] - c - half + pred) & 0xffffu;  // :67
                v = (int)(tval & (uint32_t)(c - 1));  // % c, c a power of two
                dst[at] = (uint16_t)v;
            }
            if (x == 0) first_of_row = v;
            left_top = t;
            top[x] = (uint16_t)v;
            left = v;
            const int nb = last_row ? 0 : pick_best_biased(v, k, mb, c);  // prediction.hpp:213-225
            bp[x] = (uint8_t)nb;
            bp_left = nb;
        }
    }
}

// -------------------------------------------------------------------------------------------------
// channelpredict_all on the ENCODE side, every pixel in parallel.  The walk above is serial only through its
// state arrays; when all pixel values are known (encoding) that state is a function of the pixels:
//   bp[x] while (x, y) is predicted = the best predictor of the pixel ABOVE, (x, y-1)  [4 on the first row]
//   bp_left                         = the best predictor of the pixel to the LEFT, (x-1, y); for x == 0 it is
//                                     bp[w-1], which still holds row y-1's last pixel             [4 at (0, 0)]
//   best predictor of pixel q       = 0 on the last row, else the argmin over the mask of the cell that holds
//                                     the pixel BELOW q (prediction.hpp:213-225)
// Phase 1 computes the best predictor of every pixel, phase 2 the residuals (k_predict_all_fused).
// -------------------------------------------------------------------------------------------------
// Division of a 31-bit number by a run-time constant without the software divide (~20 instructions; the per-pixel
// kernels below spent half of theirs splitting a linear index into plane / row / column / grid cell): the host
// prepares (multiplier, shift) once per launch, the device needs a multiply-high, an add and a shift.
struct FastDiv {
    uint32_t d, mul, shift;
};
__host__ __device__ inline FastDiv fastdiv_make(uint32_t d) {  // d >= 1; exact for every n < 2^31
    FastDiv f;
    f.d = d;
    uint32_t s = 0;
    while ((1ull << s) < d) s++;
    f.shift = s;
    f.mul = (uint32_t)((((1ull << s) - d) << 32) / d + 1ull);
    return f;
}
__device__ __forceinline__ uint32_t fd_div(uint32_t n, const FastDiv& f) { return (__umulhi(n, f.mul) + n) >> f.shift; }

__device__ __forceinline__ void pa_candidates(const uint16_t* __restrict__ src, int w, int x, int y, int half, Cand& k) {
    const uint16_t* row = src + (size_t)y * w;
    const uint16_t* up = row - w;
    const int L = x > 0 ? row[x - 1] : half;
    const int T = y > 0 ? up[x] : half;
    const int TL = (x > 0 && y > 0) ? up[x - 1] : half;
    int TR;
    if (x + 1 < w) TR = y > 0 ? up[x + 1] : half;
    else TR = w > 1 ? row[0] : (y > 0 ? up[0] : half);  // last column: top[0] already holds this row's first pixel
    candidates(L, T, TL, TR, false, k);
}

// Both phases in ONE kernel for a 32 x 16 pixel tile of a plane: the best predictors of the tile (and of the row above
// it and the column to its left, which are recomputed: +9 % of phase 1) go through shared memory, and the 16 candidates
// of a pixel, its neighbour loads and its position arithmetic are made once.  (Round 2 started with two kernels and a u8
// plane of best predictors in global memory: 275 + 216 executed instructions per pixel, ncu on a config-3 slice;
// fused: config 3 encode 427 -> 411 ms, config 5 280 -> 262 ms.)  A thread owns the pixels (tx, ty) and (tx, ty + 8) of
// the tile and keeps their candidates in registers between the phases.
constexpr int kPaTx = 32, kPaTy = 16;
__global__ void __launch_bounds__(256) k_predict_all_fused(const uint16_t* __restrict__ planes, uint64_t n_planes, int w,
                                                           int h, int depth, int x_tiles, int y_tiles,
                                                           const uint16_t* __restrict__ tile_maps,
                                                           uint16_t* __restrict__ out, uint64_t out_stride, FastDiv d_tpp,
                                                           FastDiv d_tpr, FastDiv d_tw, FastDiv d_th) {
    // best predictor of pixel (x0 - 1 + i, y0 - 1 + j) at s_best[j][i]; row 0 / column 0 are the halo
    __shared__ uint8_t s_best[kPaTy + 1][kPaTx + 4];
    const uint32_t pl = fd_div(blockIdx.x, d_tpp);  // d_tpp = tiles per plane, d_tpr = tiles per tile row
    if (pl >= n_planes) return;
    const uint32_t t_in = blockIdx.x - pl * d_tpp.d;
    const uint32_t t_y = fd_div(t_in, d_tpr), t_x = t_in - t_y * d_tpr.d;
    const int x0 = (int)t_x * kPaTx, y0 = (int)t_y * kPaTy;
    const int c = 1 << depth, half = c >> 1;
    const uint32_t per = (uint32_t)w * (uint32_t)h;
    const uint16_t* src = planes + (uint64_t)pl * per;
    const uint16_t* maps = tile_maps + (uint64_t)pl * (uint64_t)x_tiles * y_tiles;
    // prediction.hpp:213-225: 0 on the last row, else the argmin under the mask of the cell holding the pixel below
    auto best_of = [&](int x, int y, const Cand& k) -> int {
        if (y + 1 >= h) return 0;
        const uint32_t mask = maps[(size_t)fd_div((uint32_t)(y + 1), d_th) * x_tiles + fd_div((uint32_t)x, d_tw)];
        return pick_best(src[(size_t)y * w + x], k, mask, c);
    };
    const int tx = (int)(threadIdx.x & 31u), ty = (int)(threadIdx.x >> 5);
    const int x = x0 + tx, ya = y0 + ty, yb = y0 + ty + 8;
    const bool in_a = x < w && ya < h, in_b = x < w && yb < h;
    Cand ka, kb;
    if (in_a) {
        pa_candidates(src, w, x, ya, half, ka);
        s_best[ty + 1][tx + 1] = (uint8_t)best_of(x, ya, ka);
    }
    if (in_b) {
        pa_candidates(src, w, x, yb, half, kb);
        s_best[ty + 9][tx + 1] = (uint8_t)best_of(x, yb, kb);
    }
    // halo: threads 0..31 the row above the tile, threads 32..47 the column to its left.  For column 0 "the pixel to the
    // left" is the previous row's last pixel (bp[w - 1] still holds it when the walk starts a row: SURVEY H4); positions
    // that do not exist (row -1) read 4, the initial value of the reference's arrays (prediction.hpp:170-174)
    if (threadIdx.x < 32u + (uint32_t)kPaTy) {
        int hx, hy, sx, sy;
        if (threadIdx.x < 32u) {
            hx = x0 + tx, hy = y0 - 1, sx = tx + 1, sy = 0;
        } else {
            const int r = (int)threadIdx.x - 32;
            sx = 0, sy = r + 1;
            if (x0 > 0) hx = x0 - 1, hy = y0 + r;
            else hx = w - 1, hy = y0 + r - 1;
        }
        int b = 4;
        if (hx < w && hy >= 0 && hy < h) {
            Cand kh;
            pa_candidates(src, w, hx, hy, half, kh);
            b = best_of(hx, hy, kh);
        }
        s_best[sy][sx] = (uint8_t)b;
    }
    __syncthreads();
    if (in_a) {
        const int pred = p_mid(cand_at(ka, s_best[ty][tx + 1]), cand_at(ka, s_best[ty + 1][tx]));
        const size_t at = (size_t)ya * w + x;
        out[(uint64_t)pl * out_stride + at] = (uint16_t)mod_pow2((int)src[at] - pred + half + c, c);  // prediction.hpp:208
    }
    if (in_b) {
        const int pred = p_mid(cand_at(kb, s_best[ty + 8][tx + 1]), cand_at(kb, s_best[ty + 9][tx]));
        const size_t at = (size_t)yb * w + x;
        out[(uint64_t)pl * out_stride + at] = (uint16_t)mod_pow2((int)src[at] - pred + half + c, c);
    }
}

// =================================================================================================
// channelpredict_section — prediction.hpp:46-151.  One thread per (plane, cell, mask).
// Writes the cell's residuals in cell-raster order.  COST mode instead accumulates
// sum(cost[resid]) in double precision in raster order (layer_encode.hpp:192-195).
// =================================================================================================
constexpr int kMaxCellW = 64;  // the predictor grid is 40 px (layer_encode.hpp:124): cells are <= 40 wide

template <bool COST>
__global__ void __launch_bounds__(64) k_section(const uint16_t* __restrict__ planes, uint64_t n_planes, int w,
                                                int h, int depth, int x_tiles, int y_tiles,
                                                const uint16_t* __restrict__ masks, int n_masks,
                                                uint16_t* __restrict__ resid, uint32_t cell_cap,
                                                uint32_t* __restrict__ counts, const double* __restrict__ cost,
                                                double* __restrict__ sums, uint16_t* __restrict__ wide_top,
                                                uint8_t* __restrict__ wide_bp) {
    const int cells = x_tiles * y_tiles;
    const uint64_t job = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t jobs = n_planes * (uint64_t)cells * n_masks;
    if (job >= jobs) return;
    const int mi = (int)(job % n_masks);
    const int cell = (int)((job / n_masks) % cells);
    const uint64_t p = job / ((uint64_t)n_masks * cells);
    const uint32_t mask = masks[mi];
    const int c = 1 << depth, half = c >> 1;
    const int tw = (w + x_tiles - 1) / x_tiles, th = (h + y_tiles - 1) / y_tiles;
    const int cx = cell % x_tiles, cy = cell / x_tiles;
    const int x0 = cx * tw, y0 = cy * th;
    const uint64_t per = (uint64_t)w * h;
    const uint16_t* data = planes + p * per;
    const double* ctab = COST ? cost + p * (uint64_t)c : nullptr;
    uint16_t* dst = COST ? nullptr : resid + job * cell_cap;

    uint16_t top_local[kMaxCellW];
    uint8_t bp_local[kMaxCellW];
    // cells of the 40-px predictor grid fit the local arrays; arbitrary callers (tw > 64) use scratch
    uint16_t* top = tw <= kMaxCellW ? top_local : wide_top + job * (uint64_t)tw;
    uint8_t* bp = tw <= kMaxCellW ? bp_local : wide_bp + job * (uint64_t)tw;
    // prediction.hpp:76-94 — tw entries of the row above are read even when the cell is clipped at
    // the right edge (the read then runs into the next image row); reads are clamped to the plane.
    for (int i = 0; i < tw; i++) {
        bp[i] = 4;
        if (cy) {
            const int64_t idx = (int64_t)y0 * w + x0 + i - w;
            top[i] = (idx >= 0 && (uint64_t)idx < per) ? data[idx] : (uint16_t)0;
        } else {
            top[i] = (uint16_t)half;
        }
    }
    uint32_t k = 0;
    double sum = 0.0;
    for (int ym = 0; ym < th && y0 + ym < h; ym++) {
        int left, left_top;
        if (cx) {  // prediction.hpp:97-105
            left = data[(uint64_t)(y0 + ym) * w + x0 - 1];
            left_top = (ym || cy) ? data[(uint64_t)(y0 + ym - 1) * w + x0 - 1] : half;
        } else {
            left = left_top = half;
        }
        for (int xm = 0; xm < tw && x0 + xm < w; xm++) {
            const int v = data[(uint64_t)(y0 + ym) * w + x0 + xm];
            Cand kk;
            // (xm + 1) % tw and (xm + tw - 1) % tw as selects: tw is a run-time value, `%` a software division
            candidates(left, top[xm], left_top, top[xm + 1 == tw ? 0 : xm + 1], true, kk);  // :115 TR wraps inside the cell
            const int pred = p_mid(cand_at(kk, bp[xm]), cand_at(kk, bp[xm ? xm - 1 : tw - 1]));  // :134
            const int r = mod_pow2(v - pred + half + c, c);
            if (COST) sum += ctab[r]; else if (k < cell_cap) dst[k] = (uint16_t)r;
            k++;
            left_top = top[xm];
            top[xm] = (uint16_t)v;
            left = v;
            bp[xm] = (uint8_t)pick_best(v, kk, mask, c);
        }
    }
    if (COST) sums[job] = sum; else counts[job] = k;
}

// The search's cost sums (layer_encode.hpp:176-203, 233-272) for ALL masks of a cell in one walk.  k_section<true>
// spends its time recomputing what does not depend on the mask: the 16 candidates of a pixel and its 16
// prediction errors.  Here a thread owns one (plane, cell), computes those once per pixel, parks the
// candidates in shared memory ([candidate][thread], one 32-bit word each: bank = lane) and then runs the
// NM masks over them: the per-mask best predictors of a column live in one 64-bit word (4 bits per mask), the
// argmin is a min over keys (error << 4 | index: lowest index wins ties, prediction.hpp:138-146), and each
// mask's cost is accumulated in raster order in its own double exactly as the one-mask walk does.
// STOCK: the masks are the first NM of the reference's own list (layer_encode.hpp:159-175, the only list the
// encoder uses): they are compile-time constants then, so after unrolling every mask's kind and indices fold
// away — a singleton's key is a register, no branches, no per-mask descriptors in registers.
__device__ __forceinline__ void mask_kind(uint32_t mk, uint32_t& kind, uint32_t& a, uint32_t& b) {
    mk &= 0xffffu;
    const int pc = __popc(mk);
    kind = 3u;
    a = b = 0u;
    if (pc >= 15) {
        kind = 0u;
        a = pc == 16 ? 16u : (uint32_t)__ffs((int)(~mk & 0xffffu)) - 1u;
    } else if (pc == 1 || pc == 2) {
        kind = (uint32_t)pc;
        a = (uint32_t)__ffs((int)mk) - 1u;
        b = 31u - (uint32_t)__clz((int)mk);
    }
}
template <int NM, bool STOCK>
__global__ void __launch_bounds__(64) k_section_costs(const uint16_t* __restrict__ planes, uint64_t n_planes, int w,
                                                      int h, int depth, int x_tiles, int y_tiles,
                                                      const uint16_t* __restrict__ masks,
                                                      const double* __restrict__ cost, double* __restrict__ sums) {
    __shared__ uint32_t s_cand[16][64];
    const int cells = x_tiles * y_tiles;
    const uint64_t job = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (job >= n_planes * (uint64_t)cells) return;
    const int cell = (int)(job % cells);
    const uint64_t p = job / (uint64_t)cells;
    const int c = 1 << depth, half = c >> 1;
    const int tw = (w + x_tiles - 1) / x_tiles, th = (h + y_tiles - 1) / y_tiles;
    const int cx = cell % x_tiles, cy = cell / x_tiles;
    const int x0 = cx * tw, y0 = cy * th;
    const uint64_t per = (uint64_t)w * h;
    const uint16_t* data = planes + p * per;
    const uint32_t ctab0 = (uint32_t)p * (uint32_t)c;  // this plane's cost table inside `cost` (32-bit index arithmetic)
    // The reference's masks are single predictors, pairs, "all" and "all but one" (layer_encode.hpp:160-174), and for
    // those the masked argmin needs no walk over the 16 keys: a singleton or pair is one or two keys, and the minimum
    // over all-but-j is the second smallest key when the smallest is j's, else the smallest (keys are distinct: the
    // index is part of the key).  The two smallest keys are found once per pixel.  info = kind | a << 2 | b << 7;
    // kind 0: all / all but a (a = 16: none missing), 1: {a}, 2: {a, b}, 3: anything else (the generic walk).
    constexpr uint32_t kStock[14] = {0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd,
                                     0xfffb, 0xfff7, 0xffef, 0xffdf, 0xff7f, 0xfdff, 0xffff};
    uint32_t info[STOCK ? 1 : NM];
    if (!STOCK) {
#pragma unroll
        for (int m = 0; m < NM; m++) {
            uint32_t kind, a, b;
            mask_kind(masks[m], kind, a, b);
            info[m] = kind | (a << 2) | (b << 7);
        }
    }
    uint16_t top[kMaxCellW];
    uint64_t bpcol[kMaxCellW];
    for (int i = 0; i < tw; i++) {  // prediction.hpp:76-94, as in k_section
        bpcol[i] = 0x4444444444444444ull;
        if (cy) {
            const int64_t idx = (int64_t)y0 * w + x0 + i - w;
            top[i] = (idx >= 0 && (uint64_t)idx < per) ? data[idx] : (uint16_t)0;
        } else {
            top[i] = (uint16_t)half;
        }
    }
    double sum[NM];
#pragma unroll
    for (int m = 0; m < NM; m++) sum[m] = 0.0;
    const uint32_t tid = threadIdx.x;
    for (int ym = 0; ym < th && y0 + ym < h; ym++) {
        int left, left_top;
        if (cx) {  // prediction.hpp:97-105
            left = data[(uint64_t)(y0 + ym) * w + x0 - 1];
            left_top = (ym || cy) ? data[(uint64_t)(y0 + ym - 1) * w + x0 - 1] : half;
        } else {
            left = left_top = half;
        }
        for (int xm = 0; xm < tw && x0 + xm < w; xm++) {
            const int v = data[(uint64_t)(y0 + ym) * w + x0 + xm];
            Cand kk;
            candidates(left, top[xm], left_top, top[xm + 1 == tw ? 0 : xm + 1], true, kk);  // :115 TR wraps inside the cell
            int key[16];
#pragma unroll
            for (int j = 0; j < 16; j++) {
                s_cand[j][tid] = (uint32_t)kk.v[j];
                key[j] = abs(v - kk.v[j]) * 16 + j;  // "error below 2c" (prediction.hpp:138) is tested on the winner only
            }
            int b1 = 0x7fffffff, b2 = 0x7fffffff;  // the two smallest keys
#pragma unroll
            for (int j = 0; j < 16; j++) {
                b2 = min(b2, max(b1, key[j]));
                b1 = min(b1, key[j]);
            }
            auto key_of = [&](uint32_t j) { return abs(v - (int)s_cand[j][tid]) * 16 + (int)j; };
            const uint64_t above = bpcol[xm];
            const uint64_t before = bpcol[xm ? xm - 1 : tw - 1];  // :134 (xm + tw - 1) % tw: this row's left pixel once xm > 0
            uint64_t now = 0;
#pragma unroll
            for (int m = 0; m < NM; m++) {
                const uint32_t bt = (uint32_t)(above >> (4 * m)) & 15u, bl = (uint32_t)(before >> (4 * m)) & 15u;
                const int pred = p_mid((int)s_cand[bt][tid], (int)s_cand[bl][tid]);
                // (v - pred + half + c) % c: the operand is positive for pixels below c, and the table has c entries
                const uint32_t r = (uint32_t)(v - pred + half + c) & (uint32_t)(c - 1);
                sum[m] += __ldg(cost + (ctab0 + r));
                uint32_t kind, ia, ib;
                if (STOCK) {
                    mask_kind(kStock[m], kind, ia, ib);  // constants after unrolling
                } else {
                    kind = info[m] & 3u, ia = (info[m] >> 2) & 31u, ib = info[m] >> 7;
                }
                int best;
                if (kind == 0u) {
                    best = (uint32_t)(b1 & 15) == ia ? b2 : b1;
                } else if (kind == 3u) {
                    const uint32_t mk = STOCK ? kStock[m] : (uint32_t)masks[m];
                    best = 0x7fffffff;
#pragma unroll
                    for (int j = 0; j < 16; j++) best = min(best, ((mk >> j) & 1u) ? key[j] : 0x7fffffff);
                } else if (STOCK) {
                    // the indices are constants here: the selects fold to one register (written as selects, not as
                    // key[ia], so that the array never looks dynamically indexed and stays in registers)
                    int ka = key[0], kb = key[0];
#pragma unroll
                    for (int j = 1; j < 16; j++) {
                        ka = ia == (uint32_t)j ? key[j] : ka;
                        kb = ib == (uint32_t)j ? key[j] : kb;
                    }
                    best = kind == 2u ? min(ka, kb) : ka;
                } else {
                    best = key_of(ia);
                    if (kind == 2u) best = min(best, key_of(ib));
                }
                // "stays 0 when nothing beats 2c" (prediction.hpp:138): every candidate is a median / average / copy of
                // in-range neighbours, so an allowed candidate's error is below c; only an EMPTY mask (0x7fffffff, not in
                // the stock list) can fail the test
                const int won = STOCK ? (best & 15) : ((best >> 4) < 2 * c ? (best & 15) : 0);
                now |= (uint64_t)won << (4 * m);
            }
            bpcol[xm] = now;
            left_top = top[xm];
            top[xm] = (uint16_t)v;
            left = v;
        }
    }
#pragma unroll
    for (int m = 0; m < NM; m++) sums[job * NM + m] = sum[m];
}

// layer_encode.hpp:133-144 / :217-225: +1-smoothed histogram of a residual plane.  One CTA per plane.
__global__ void __launch_bounds__(256) k_plane_histogram(const uint16_t* __restrict__ resid, uint32_t per,
                                                         int depth, uint32_t* __restrict__ hist, uint64_t stride) {
    __shared__ uint32_t s_h[kFreqRow];
    const int c = 1 << depth;
    for (int i = threadIdx.x; i < c; i += blockDim.x) s_h[i] = 1;  // the +1 smoothing
    __syncthreads();
    const uint16_t* r = resid + (uint64_t)blockIdx.x * stride;
    for (uint32_t i = threadIdx.x; i < per; i += blockDim.x) atomicAdd(&s_h[r[i] & (c - 1)], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < c; i += blockDim.x) hist[(uint64_t)blockIdx.x * c + i] = s_h[i];
}

// cost[v] = -log2(f / size) looked up in a host-built table E[f] (SURVEY H5: glibc log2 is the
// reference; the table is indexed by the exact integer count so no device log2 is involved).
__global__ void k_cost_from_hist(const uint32_t* __restrict__ hist, uint64_t entries, const double* __restrict__ e_tab,
                                 uint32_t e_len, double* __restrict__ cost) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= entries) return;
    const uint32_t f = hist[i];
    cost[i] = e_tab[f < e_len ? f : e_len - 1];
}

// layer_encode.hpp:196-200: strict-< argmin over masks in order; 99999999999 is the starting best.
__global__ void k_pick_masks(const double* __restrict__ sums, uint64_t n_cells_total, int n_masks,
                             const uint16_t* __restrict__ masks, uint16_t* __restrict__ tile_maps,
                             uint8_t* __restrict__ index_lists) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n_cells_total) return;
    double best = 99999999999.0;
    int arg = 0;
    uint16_t m = tile_maps[i];
    bool any = false;
    for (int k = 0; k < n_masks; k++) {
        const double s = sums[i * n_masks + k];
        if (s < best) {
            best = s;
            arg = k;
            m = masks[k];
            any = true;
        }
    }
    if (any) {
        tile_maps[i] = m;
        index_lists[i] = (uint8_t)arg;
    }
}

// =================================================================================================
// Tile front end, cruncher mode 0 — choh.cpp:464-484 (tile gather) + channel.hpp:73 (subtract green)
// + prediction.hpp:6-44 (fastpath residuals) + entropy_encoding.hpp:32-39 (histograms), fused: one
// pass over the RGB bytes.  One CTA per tile.
// =================================================================================================
struct TileGeom {
    uint32_t width, height, x_tiles, y_tiles, tile_w, tile_h, tiles_per_image;
    uint32_t plane_stride;  // u16 elements reserved per channel plane (tile_w*tile_h rounded up to 8)
};

__device__ __forceinline__ void tile_rect(const TileGeom& g, uint32_t tile, uint32_t& x0, uint32_t& y0,
                                          uint32_t& tw, uint32_t& th) {
    x0 = (tile % g.x_tiles) * g.tile_w;
    y0 = (tile / g.x_tiles) * g.tile_h;
    tw = min(g.tile_w, g.width - x0);   // choh.cpp:466-474
    th = min(g.tile_h, g.height - y0);
}

// A rectangular sub-grid of an image's tile grid: the tiles of one SHAPE.  choh.cpp:459-474 gives every tile the
// nominal size except those of the last column / last row, which take what is left, so an image has up to four
// shapes (interior, right edge, bottom edge, corner); kernels that need equal tiles run once per shape.
// Local tile lt of a selection over a batch: image lt / per_image, then row-major inside the sub-grid.
struct TileSel {
    TileGeom g;
    uint32_t x_first, x_count, y_first, y_count, per_image;
};

__device__ __forceinline__ void sel_tile(const TileSel& s, uint64_t lt, uint64_t& image, uint32_t& tile_in_image,
                                         uint32_t& x0, uint32_t& y0, uint32_t& tw, uint32_t& th) {
    image = lt / s.per_image;
    const uint32_t k = (uint32_t)(lt % s.per_image);
    const uint32_t tx = s.x_first + k % s.x_count, ty = s.y_first + k / s.x_count;
    tile_in_image = ty * s.g.x_tiles + tx;
    tile_rect(s.g, tile_in_image, x0, y0, tw, th);
}

__global__ void __launch_bounds__(256) k_tile_residuals_s0_generic(const uint8_t* __restrict__ rgb, TileGeom g,
                                                           uint16_t* __restrict__ resid,
                                                           uint32_t* __restrict__ freqs) {
    __shared__ uint32_t s_h[3][kFreqRow];
    for (int i = threadIdx.x; i < 3 * kFreqRow; i += blockDim.x) (&s_h[0][0])[i] = 0;
    __syncthreads();
    const uint64_t t = blockIdx.x;  // global tile index = image * tiles_per_image + tile
    const uint64_t image = t / g.tiles_per_image;
    const uint32_t tile = (uint32_t)(t % g.tiles_per_image);
    uint32_t x0, y0, tw, th;
    tile_rect(g, tile, x0, y0, tw, th);
    const uint8_t* img = rgb + image * (uint64_t)g.width * g.height * 3u;
    uint16_t* out_g = resid + (t * 3u + 0u) * g.plane_stride;
    uint16_t* out_rg = resid + (t * 3u + 1u) * g.plane_stride;
    uint16_t* out_bg = resid + (t * 3u + 2u) * g.plane_stride;
    const uint32_t px = tw * th;
    for (uint32_t i = threadIdx.x; i < px; i += blockDim.x) {
        const uint32_t x = i % tw, y = i / tw;
        const uint8_t* p = img + ((uint64_t)(y0 + y) * g.width + x0 + x) * 3u;
        const int64_t up = -(int64_t)g.width * 3;
        const int r = p[0], gg = p[1], b = p[2];
        int Lg = 128, Lr = 256, Lb = 256, Tg = 128, Tr = 256, Tb = 256, TLg = 128, TLr = 256, TLb = 256;
        if (x) {
            const int lr = p[-3], lg = p[-2], lb = p[-1];
            Lg = lg;
            Lr = lr - lg + 256;
            Lb = lb - lg + 256;
        }
        if (y) {
            const int tr = p[up], tg = p[up + 1], tb = p[up + 2];
            Tg = tg;
            Tr = tr - tg + 256;
            Tb = tb - tg + 256;
            if (x) {
                const int ar = p[up - 3], ag = p[up - 2], ab = p[up - 1];
                TLg = ag;
                TLr = ar - ag + 256;
                TLb = ab - ag + 256;
            }
        }
        const int vg = gg, vr = r - gg + 256, vb = b - gg + 256;
        const int rg_ = (vg - p_med_grad(Tg, Lg, TLg) + 128 + 256) & 255;   // % 256
        const int rr_ = (vr - p_med_grad(Tr, Lr, TLr) + 256 + 512) & 511;   // % 512
        const int rb_ = (vb - p_med_grad(Tb, Lb, TLb) + 256 + 512) & 511;
        out_g[i] = (uint16_t)rg_;
        out_rg[i] = (uint16_t)rr_;
        out_bg[i] = (uint16_t)rb_;
        atomicAdd(&s_h[0][rg_], 1u);
        atomicAdd(&s_h[1][rr_], 1u);
        atomicAdd(&s_h[2][rb_], 1u);
    }
    __syncthreads();
    for (int ch = 0; ch < 3; ch++) {
        uint32_t* dst = freqs + (t * 3u + ch) * kFreqRow;
        for (int i = threadIdx.x; i < kFreqRow; i += blockDim.x) dst[i] = s_h[ch][i];
    }
}

// Same stage for the common geometry (image width and tile width multiples of 4): every thread takes
// four horizontally adjacent pixels = 12 bytes = three aligned words per row (plus the word holding the
// left neighbour), so global traffic is 32-bit loads and 8-byte stores and the row/column bookkeeping
// is incremental (no per-pixel division).  The two 9-bit planes (R-G, B-G) travel as two 16-bit lanes
// of one register through the packed median.
// A thread owns a column of four pixels over a band of rows and walks DOWN it: the row above is what it converted
// one iteration earlier (registers), so every RGB word is loaded and split into planes once instead of twice, and the
// next row's words are requested before the current row is worked on.
__global__ void __launch_bounds__(256) k_tile_residuals_s0(const uint8_t* __restrict__ rgb, TileGeom g,
                                                           uint16_t* __restrict__ resid,
                                                           uint32_t* __restrict__ freqs) {
    __shared__ uint32_t s_h[3][kFreqRow];
    for (int i = threadIdx.x; i < 3 * kFreqRow; i += blockDim.x) (&s_h[0][0])[i] = 0;
    __syncthreads();
    const uint64_t t = blockIdx.x;  // global tile index = image * tiles_per_image + tile
    const uint64_t image = t / g.tiles_per_image;
    const uint32_t tile = (uint32_t)(t % g.tiles_per_image);
    uint32_t x0, y0, tw, th;
    tile_rect(g, tile, x0, y0, tw, th);
    const uint8_t* img = rgb + image * (uint64_t)g.width * g.height * 3u;
    uint16_t* out_g = resid + (t * 3u + 0u) * g.plane_stride;
    uint16_t* out_rg = resid + (t * 3u + 1u) * g.plane_stride;
    uint16_t* out_bg = resid + (t * 3u + 2u) * g.plane_stride;
    const uint32_t quads = tw / 4u;  // tw % 4 == 0 on this path
    const uint32_t qpt = min(quads, 256u);  // quad columns walked at the same time
    const uint32_t n_bands = 256u / qpt, band_rows = (th + n_bands - 1u) / n_bands;
    const uint32_t band = threadIdx.x / qpt;
    const uint32_t row_words = g.width * 3u / 4u;
    if (band < n_bands) {
        const uint32_t ya = band * band_rows, yb = min(th, ya + band_rows);
        for (uint32_t q = threadIdx.x % qpt; q < quads && ya < yb; q += qpt) {
            const uint32_t* row = reinterpret_cast<const uint32_t*>(img + ((uint64_t)(y0 + ya) * g.width + x0 + 4u * q) * 3u);
            uint32_t tg[5], tr[5];  // the row above: left neighbour + the quad, as g and (rg | bg << 16)
            if (ya) {
                const uint32_t* up = row - row_words;
                const uint32_t u0 = up[0], u1 = up[1], u2 = up[2];
                planes2_of(u0 & 0xffffffu, tg[1], tr[1]);
                planes2_of((u0 >> 24) | ((u1 & 0xffffu) << 8), tg[2], tr[2]);
                planes2_of((u1 >> 16) | ((u2 & 0xffu) << 16), tg[3], tr[3]);
                planes2_of(u2 >> 8, tg[4], tr[4]);
                if (q) planes2_of(up[-1] >> 8, tg[0], tr[0]);
            } else {
#pragma unroll
                for (int i = 1; i < 5; i++) {  // row 0: T = TL = c/2
                    tg[i] = 128u;
                    tr[i] = kHalfRB;
                }
            }
            if (!q || !ya) {  // column 0 / row 0: TL = c/2
                tg[0] = 128u;
                tr[0] = kHalfRB;
            }
            uint32_t n0 = row[0], n1 = row[1], n2 = row[2], nl = q ? row[-1] : 0u;
            uint32_t at = ya * tw + 4u * q;
            for (uint32_t y = ya; y < yb; y++, at += tw) {
                const uint32_t w0 = n0, w1 = n1, w2 = n2, wl = nl;
                if (y + 1u < yb) {  // the next row's words, in flight while this row is worked on
                    row += row_words;
                    n0 = row[0];
                    n1 = row[1];
                    n2 = row[2];
                    if (q) nl = row[-1];
                }
                uint32_t cg[5], cr[5];
                planes2_of(w0 & 0xffffffu, cg[1], cr[1]);
                planes2_of((w0 >> 24) | ((w1 & 0xffffu) << 8), cg[2], cr[2]);
                planes2_of((w1 >> 16) | ((w2 & 0xffu) << 16), cg[3], cr[3]);
                planes2_of(w2 >> 8, cg[4], cr[4]);
                if (q) {
                    planes2_of(wl >> 8, cg[0], cr[0]);
                } else {  // column 0: L = c/2
                    cg[0] = 128u;
                    cr[0] = kHalfRB;
                }
                uint32_t rg_[4], rr_[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {  // prediction.hpp:35-41: (v - median + c/2 + c) % c
                    rg_[i] = (cg[i + 1] - p_med_grad2(tg[i + 1], cg[i], tg[i]) + 128u + 256u) & 255u;
                    rr_[i] = __vadd2(__vsub2(cr[i + 1], p_med_grad2(tr[i + 1], cr[i], tr[i])), kHalfRB) & kMaskRB;
                    atomicAdd(&s_h[0][rg_[i]], 1u);
                    atomicAdd(&s_h[1][rr_[i] & 0xffffu], 1u);
                    atomicAdd(&s_h[2][rr_[i] >> 16], 1u);
                }
                *reinterpret_cast<uint2*>(out_g + at) = make_uint2(rg_[0] | (rg_[1] << 16), rg_[2] | (rg_[3] << 16));
                *reinterpret_cast<uint2*>(out_rg + at) =
                    make_uint2(__byte_perm(rr_[0], rr_[1], 0x5410), __byte_perm(rr_[2], rr_[3], 0x5410));
                *reinterpret_cast<uint2*>(out_bg + at) =
                    make_uint2(__byte_perm(rr_[0], rr_[1], 0x7632), __byte_perm(rr_[2], rr_[3], 0x7632));
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    tg[i] = cg[i];
                    tr[i] = cr[i];
                }
            }
        }
    }
    __syncthreads();
    for (int ch = 0; ch < 3; ch++) {
        uint32_t* dst = freqs + (t * 3u + ch) * kFreqRow;
        for (int i = threadIdx.x; i < kFreqRow; i += blockDim.x) dst[i] = s_h[ch][i];
    }
}

// Descriptors for the 3 streams of every tile (layer_encode.hpp:57, 59, 321-324: channel header
// 10 | 00 00 | 00 10, prob_bits 15, range 1 << depth).
__global__ void k_make_tile_streams(TileGeom g, uint64_t n_tiles, uint32_t slab_bytes,
                                    hoh_enc_stream* __restrict__ streams) {
    const uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (s >= n_tiles * 3u) return;
    const uint64_t t = s / 3u;
    const uint32_t ch = (uint32_t)(s % 3u);
    uint32_t x0, y0, tw, th;
    tile_rect(g, (uint32_t)(t % g.tiles_per_image), x0, y0, tw, th);
    hoh_enc_stream st;
    st.sym_off = s * g.plane_stride;
    st.n = tw * th;
    st.range = ch == 0 ? 256u : 512u;
    st.prob_bits = 15;
    st.prefix_len = 5;
    st.prefix[0] = 0x10;
    st.prefix[1] = 0;
    st.prefix[2] = 0;
    st.prefix[3] = 0x00;
    st.prefix[4] = 0x10;
    st.prefix[5] = st.prefix[6] = st.prefix[7] = 0;
    st.out_off = s * (uint64_t)slab_bytes;
    st.out_cap = slab_bytes;
    st.reserved = 0;
    streams[s] = st;
}

// Decode side descriptors: stream s starts at packed_off[s]; checks the 5-byte mode-0 channel header.
__global__ void k_make_tile_dec_streams(TileGeom g, uint64_t n_tiles, const uint8_t* __restrict__ packed,
                                        uint64_t packed_bytes, const uint64_t* __restrict__ packed_off,
                                        hoh_dec_stream* __restrict__ streams, int32_t* __restrict__ status) {
    const uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (s >= n_tiles * 3u) return;
    const uint64_t off = packed_off[s];
    const ByteView b{packed, packed_bytes};
    const bool ok = b[off] == 0x10 && b[off + 1] == 0 && b[off + 2] == 0 && b[off + 3] == 0 && b[off + 4] == 0x10;
    uint32_t x0, y0, tw, th;
    tile_rect(g, (uint32_t)((s / 3u) % g.tiles_per_image), x0, y0, tw, th);
    hoh_dec_stream st;
    st.in_off = off + 5u;
    st.sym_off = s * g.plane_stride;
    st.sym_cap = ok ? tw * th : 0u;
    st.flags = HOH_FIX_ALL;
    streams[s] = st;
    status[s] = ok ? HOH_S_OK : HOH_S_BAD_LAYER;
}

// Tile back end, mode 0: wavefront inverse of the MED predictor on the three planes of a tile, the
// inverse colour transform and the scatter into the interleaved image (dhoh.cpp:72-84, 268-276).
// One warp per tile; lane = row inside a 32-row band; lane r works on column t - r at step t and gets
// its top neighbour from lane r-1 by shuffle (anti-diagonal wavefront).  Residuals and pixels move
// through two shared-memory rings (32 rows x 64 columns, row stride 66 words so that both the
// row-wise transfers and the diagonal accesses are bank-conflict free): every 32 steps the warp loads
// the next 32-column block of all 32 rows with coalesced reads and writes back the block that was
// completed two boundaries ago with coalesced stores.
constexpr int kRingStride = 66;                      // words per ring row (64 columns + 2 pad)
constexpr int kUnpWarps = 4;
constexpr int kUnpBlock = 16;                        // columns per transfer block; the rings hold 4 blocks
constexpr uint32_t kMidPacked = 128u | (256u << 8) | (256u << 17);  // border value c/2 of G, R-G, B-G

// Residual block (32 rows x 16 columns, three planes) -> registers: four rows per instruction, four
// columns (8 bytes per plane) per lane; the loads are issued one block ahead of their use.
struct UnpPrefetch {
    uint2 g[4], a[4], b[4];
};
template <bool ALIGNED>
__device__ __forceinline__ void unp_fetch_block(UnpPrefetch& pf, const uint16_t* __restrict__ in_g,
                                                const uint16_t* __restrict__ in_rg,
                                                const uint16_t* __restrict__ in_bg, uint32_t y_base, uint32_t th,
                                                uint32_t tw, uint32_t block) {
    const uint32_t lane = lane_id();
    const uint32_t c = kUnpBlock * block + 4u * (lane & 3u);
#pragma unroll
    for (uint32_t i = 0; i < 4; i++) {
        const uint32_t y = y_base + 8u * i + (lane >> 2);
        pf.g[i] = pf.a[i] = pf.b[i] = make_uint2(0u, 0u);
        if (y < th && c < tw) {
            const uint32_t at = y * tw + c;
            if (ALIGNED) {  // tw % 4 == 0
                pf.g[i] = *reinterpret_cast<const uint2*>(in_g + at);
                pf.a[i] = *reinterpret_cast<const uint2*>(in_rg + at);
                pf.b[i] = *reinterpret_cast<const uint2*>(in_bg + at);
            } else {
                uint32_t v[3][4];
#pragma unroll
                for (uint32_t k = 0; k < 4; k++) {
                    const bool ok = c + k < tw;
                    v[0][k] = ok ? in_g[at + k] : 0u;
                    v[1][k] = ok ? in_rg[at + k] : 0u;
                    v[2][k] = ok ? in_bg[at + k] : 0u;
                }
                pf.g[i] = make_uint2(v[0][0] | (v[0][1] << 16), v[0][2] | (v[0][3] << 16));
                pf.a[i] = make_uint2(v[1][0] | (v[1][1] << 16), v[1][2] | (v[1][3] << 16));
                pf.b[i] = make_uint2(v[2][0] | (v[2][1] << 16), v[2][2] | (v[2][3] << 16));
            }
        }
    }
}
// registers -> ring slot of `block`, packed g | rg << 8 | bg << 17
__device__ __forceinline__ void unp_commit_block(const UnpPrefetch& pf, uint32_t* ring, uint32_t block) {
    const uint32_t lane = lane_id();
    const uint32_t col = (block & 3u) * kUnpBlock + 4u * (lane & 3u);
#pragma unroll
    for (uint32_t i = 0; i < 4; i++) {
        uint32_t* dst = ring + (8u * i + (lane >> 2)) * kRingStride + col;
        const uint2 g = pf.g[i], a = pf.a[i], b = pf.b[i];
        dst[0] = (g.x & 0xffffu) | ((a.x & 0xffffu) << 8) | ((b.x & 0xffffu) << 17);
        dst[1] = (g.x >> 16) | ((a.x >> 16) << 8) | ((b.x >> 16) << 17);
        dst[2] = (g.y & 0xffffu) | ((a.y & 0xffffu) << 8) | ((b.y & 0xffffu) << 17);
        dst[3] = (g.y >> 16) | ((a.y >> 16) << 8) | ((b.y >> 16) << 17);
    }
}

// ring values are 0x00BBGGRR; block = 32 rows x 16 columns = 48 bytes per row
template <bool ALIGNED>
__device__ __forceinline__ void unp_store_block(const uint32_t* ring, uint8_t* __restrict__ img, uint32_t width,
                                                uint32_t x0, uint32_t y0, uint32_t y_base, uint32_t th, uint32_t tw,
                                                uint32_t block) {
    const uint32_t lane = lane_id();
    const uint32_t col = (block & 3u) * kUnpBlock + 4u * (lane & 3u);
    const uint32_t c = kUnpBlock * block + 4u * (lane & 3u);
#pragma unroll
    for (uint32_t i = 0; i < 4; i++) {
        const uint32_t r = 8u * i + (lane >> 2);
        const uint32_t y = y_base + r;
        if (y < th && c < tw) {
            const uint32_t* src = ring + r * kRingStride + col;
            const uint32_t A = src[0], B = src[1], C = src[2], D = src[3];
            uint8_t* dst8 = img + ((uint64_t)(y0 + y) * width + x0 + c) * 3u;
            if (ALIGNED) {  // width % 4 == 0 and tile_w % 4 == 0: 4 pixels = 3 aligned words
                uint32_t* dst = reinterpret_cast<uint32_t*>(dst8);
                dst[0] = A | (B << 24);
                dst[1] = (B >> 8) | (C << 16);
                dst[2] = (C >> 16) | (D << 8);
            } else {
                const uint32_t px[4] = {A, B, C, D};
#pragma unroll
                for (uint32_t k = 0; k < 4; k++)
                    if (c + k < tw) {
                        dst8[3 * k] = (uint8_t)px[k];
                        dst8[3 * k + 1] = (uint8_t)(px[k] >> 8);
                        dst8[3 * k + 2] = (uint8_t)(px[k] >> 16);
                    }
            }
        }
    }
}

// Tile back end, mode 0: wavefront inverse of the MED predictor on the three planes of a tile, the
// inverse colour transform and the scatter into the interleaved image (dhoh.cpp:72-84, 268-276).
// One warp per tile; lane = row inside a 32-row band; lane r works on column t - r at step t and gets
// its top neighbour from lane r-1 by shuffle (anti-diagonal wavefront).  Residuals and pixels move
// through a shared-memory ring (32 rows x 64 columns = 4 blocks of 16, row stride 66 words so that
// both the row-wise transfers and the diagonal accesses are bank-conflict free).  Every 16 steps: the
// block completed three boundaries ago is written back with coalesced stores, the residual block
// fetched (into registers) one boundary ago is committed to the ring, and the fetch of the next one is
// issued, so global-memory latency overlaps a whole block of computation.
template <bool ALIGNED>
__global__ void __launch_bounds__(kUnpWarps * 32, 5) k_tile_unpredict_s0(const uint16_t* __restrict__ resid, TileGeom g,
                                                                      uint64_t n_tiles, uint8_t* __restrict__ rgb) {
    extern __shared__ __align__(16) uint32_t s_unp[];  // per warp: the ring, carry row (tile_w words)
    const uint32_t wid = threadIdx.x >> 5, lane = lane_id();
    const uint64_t t = (uint64_t)blockIdx.x * kUnpWarps + wid;
    if (t >= n_tiles) return;
    const uint32_t carry_words = g.tile_w + (g.tile_w + 1u) / 2u;  // (rg | bg << 16) as u32 + g as u16
    const uint32_t per_warp = (32u * kRingStride + carry_words + 3u) & ~3u;  // 16-byte multiples: vector carry accesses
    // ONE ring: a slot holds the pixel's residuals until its step and the pixel from then on.  At boundary b the
    // block written back is b-3 (its last column was finished by lane 31 at step 16b-1) and the residual block
    // committed is b, which takes the slot of b-4, written back one boundary earlier.
    uint32_t* ring_in = s_unp + (size_t)wid * per_warp;
    uint32_t* ring_out = ring_in;
    uint32_t* carry_rb = ring_in + 32 * kRingStride;  // last row of the previous band
    uint16_t* carry_g = reinterpret_cast<uint16_t*>(carry_rb + g.tile_w);
    const uint64_t image = t / g.tiles_per_image;
    uint32_t x0, y0, tw, th;
    tile_rect(g, (uint32_t)(t % g.tiles_per_image), x0, y0, tw, th);
    uint8_t* img = rgb + image * (uint64_t)g.width * g.height * 3u;
    const uint16_t* in_g = resid + (t * 3u + 0u) * g.plane_stride;
    const uint16_t* in_rg = resid + (t * 3u + 1u) * g.plane_stride;
    const uint16_t* in_bg = resid + (t * 3u + 2u) * g.plane_stride;
    const uint32_t n_blocks = (tw + kUnpBlock - 1u) / kUnpBlock;
    const uint32_t* my_in = ring_in + lane * kRingStride;
    uint32_t* my_out = ring_out + lane * kRingStride;

    // row 0 of the tile has T = TL = c/2: the carry row starts as the border value
    for (uint32_t i = lane; i < tw; i += 32) {
        carry_g[i] = 128;
        carry_rb[i] = kHalfRB;
    }
    __syncwarp();
    for (uint32_t band = 0; band * 32u < th; band++) {
        const uint32_t y_base = band * 32u;
        const bool row_ok = y_base + lane < th;
        // column 0: L = TL = c/2; they are first used at x == 0 and only change from then on
        uint32_t Lg = 128u, TLg = 128u, Lrb = kHalfRB, TLrb = kHalfRB;
        uint32_t mine_g = 128u, mine_rb = kHalfRB;
        // One wavefront step.  FULL = every lane is inside its row (the steady state: 14 of 19 blocks of a
        // 256-wide tile), so there is nothing to predicate; rows past the bottom of the tile compute
        // harmless garbage there (their ring rows are never written back).
        auto step_fn = [&](uint32_t step, auto full_tag) {
            constexpr bool FULL = decltype(full_tag)::value;
            const int x = (int)step - (int)lane;
            const uint32_t tg_up = __shfl_up_sync(0xffffffffu, mine_g, 1);
            const uint32_t trb_up = __shfl_up_sync(0xffffffffu, mine_rb, 1);
            const bool in_row = FULL || (x >= 0 && x < (int)tw);
            const uint32_t xc = in_row ? (uint32_t)x : 0u;
            // lane 0's top row is the previous band's last row (carry), the others get it from the lane above
            const uint32_t Tg = lane == 0 ? (uint32_t)carry_g[xc] : tg_up;
            const uint32_t Trb = lane == 0 ? carry_rb[xc] : trb_up;
            if (FULL || (row_ok && in_row)) {
                const uint32_t v = my_in[xc & 63];  // residuals g | rg << 8 | bg << 17
                const uint32_t rg2 = ((v >> 8) & 511u) | ((v >> 17) << 16);
                // unprediction of the pure-MED fastpath: (resid + median - c/2) mod c, planes G and (R-G, B-G)
                const uint32_t vg = ((v & 255u) + p_med_grad2(Tg, Lg, TLg) - 128u) & 255u;
                const uint32_t vrb = __vsub2(__vadd2(rg2, p_med_grad2(Trb, Lrb, TLrb)), kHalfRB) & kMaskRB;
                // inverse colour transform (SURVEY D4): R = rg + g - 256, B = bg + g - 256 (mod 256)
                const uint32_t rb8 = __vsub2(__vadd2(vrb, vg * 0x00010001u), kHalfRB) & 0x00ff00ffu;
                my_out[xc & 63] = rb8 | (vg << 8);  // 0x00BBGGRR
                mine_g = vg;
                mine_rb = vrb;
                Lg = vg;
                Lrb = vrb;
                TLg = Tg;
                TLrb = Trb;
                if (lane == 31u) {
                    carry_g[xc] = (uint16_t)vg;
                    carry_rb[xc] = vrb;
                }
            }
        };
        // Four steady-state steps (ALIGNED tiles).  The carry row is what lane 0 reads (the row above the band) and
        // lane 31 writes (the band's last row): as scalar accesses those were a third of the kernel's shared-memory
        // wavefronts, which is what bounds it.  Lane 0 is at column s..s+3 — an aligned group, fetched as one 8-byte
        // and one 16-byte load — and lane 31 at s-31..s-28, so with the value it produced one step earlier (prev)
        // it completes the aligned group s-32..s-29 and stores it the same way.
        uint32_t prev_g = 128u, prev_rb = kHalfRB;
        auto group_fn = [&](uint32_t s) {
            uint2 cg = make_uint2(0u, 0u);
            uint4 crb = make_uint4(0u, 0u, 0u, 0u);
            if (lane == 0u) {
                cg = *reinterpret_cast<const uint2*>(carry_g + s);
                crb = *reinterpret_cast<const uint4*>(carry_rb + s);
            }
            const uint32_t cgv[4] = {cg.x & 0xffffu, cg.x >> 16, cg.y & 0xffffu, cg.y >> 16};
            const uint32_t crbv[4] = {crb.x, crb.y, crb.z, crb.w};
            uint32_t og[4], orb[4];
#pragma unroll
            for (uint32_t i = 0; i < 4u; i++) {
                const uint32_t xc = s + i - lane;
                const uint32_t tg_up = __shfl_up_sync(0xffffffffu, mine_g, 1);
                const uint32_t trb_up = __shfl_up_sync(0xffffffffu, mine_rb, 1);
                const uint32_t Tg = lane == 0u ? cgv[i] : tg_up;
                const uint32_t Trb = lane == 0u ? crbv[i] : trb_up;
                const uint32_t v = my_in[xc & 63];
                const uint32_t rg2 = ((v >> 8) & 511u) | ((v >> 17) << 16);
                const uint32_t vg = ((v & 255u) + p_med_grad2(Tg, Lg, TLg) - 128u) & 255u;
                const uint32_t vrb = __vsub2(__vadd2(rg2, p_med_grad2(Trb, Lrb, TLrb)), kHalfRB) & kMaskRB;
                const uint32_t rb8 = __vsub2(__vadd2(vrb, vg * 0x00010001u), kHalfRB) & 0x00ff00ffu;
                my_out[xc & 63] = rb8 | (vg << 8);
                mine_g = vg;
                mine_rb = vrb;
                Lg = vg;
                Lrb = vrb;
                TLg = Tg;
                TLrb = Trb;
                og[i] = vg;
                orb[i] = vrb;
            }
            if (lane == 31u) {
                *reinterpret_cast<uint2*>(carry_g + (s - 32u)) = make_uint2(prev_g | (og[0] << 16), og[1] | (og[2] << 16));
                *reinterpret_cast<uint4*>(carry_rb + (s - 32u)) = make_uint4(prev_rb, orb[0], orb[1], orb[2]);
            }
            prev_g = og[3];
            prev_rb = orb[3];
        };
        UnpPrefetch pf;
        unp_fetch_block<ALIGNED>(pf, in_g, in_rg, in_bg, y_base, th, tw, 0u);
        for (uint32_t blk = 0; blk < n_blocks + 3u; blk++) {
            __syncwarp();
            if (blk >= 3u) unp_store_block<ALIGNED>(ring_out, img, g.width, x0, y0, y_base, th, tw, blk - 3u);
            if (blk < n_blocks) unp_commit_block(pf, ring_in, blk);
            if (blk + 1u < n_blocks) unp_fetch_block<ALIGNED>(pf, in_g, in_rg, in_bg, y_base, th, tw, blk + 1u);
            __syncwarp();
            const uint32_t s0 = blk * kUnpBlock;
            if (s0 >= 31u && s0 + kUnpBlock <= tw) {
                if (ALIGNED) {
                    for (uint32_t k = 0; k < (uint32_t)kUnpBlock; k += 4u) group_fn(s0 + k);
                    if (lane == 31u) {  // the value of the block's last step waits for its group: a later block that
                        carry_g[s0 - 16u] = (uint16_t)prev_g;  // is not steady-state would never store it
                        carry_rb[s0 - 16u] = prev_rb;
                    }
                } else {
#pragma unroll 4
                    for (uint32_t k = 0; k < (uint32_t)kUnpBlock; k++) step_fn(s0 + k, std::true_type{});
                }
            } else {
#pragma unroll 4
                for (uint32_t k = 0; k < (uint32_t)kUnpBlock; k++) step_fn(s0 + k, std::false_type{});
                prev_g = mine_g;
                prev_rb = mine_rb;
            }
        }
        __syncwarp();
    }
}

// =================================================================================================
// layer_encode.hpp:11-412 for many planes — the decision sequence of the channel codec replayed on
// the device around the batched kernels above.  These small kernels are the glue: descriptors for each
// round of entropy coding, the predictor-map header, the "which buffer wins" logic (including the
// stale-buffer behaviour D7) and the final assembly of every channel payload.
// =================================================================================================
constexpr int kLayerSlots = 10;  // per plane: A (fastpath, 15 bits), B (predictor-index map), C (16), D (15),
                                 // E, F, G going up (17, 18, 19 bits) and going down (14, 13, 12 bits)
constexpr int kLayerHdrCap = 48;  // 0x10 + x_tiles-1 + y_tiles-1 + count + 14 masks * 2

struct LayerGeom {
    uint32_t per;         // w * h
    uint32_t per_pad;     // rounded up to 8 symbols
    uint32_t cells;       // predictor grid cells (0 when the plane is a single cell or mode == 0)
    uint32_t cells_pad;
    uint32_t xt, yt;
    uint32_t depth, mode;
    uint32_t slot_off[kLayerSlots]; // byte offset of each candidate's slab inside a plane's block
    uint32_t slot_cap[kLayerSlots]; // ... and its capacity (sized for the candidate's prob_bits; 0 = not used at this mode)
    uint32_t plane_bytes; // candidate bytes per plane
    uint32_t enc_flags;   // HOH_FIX_LONE or 0, handed to every entropy stream
    uint32_t out_cap;     // bytes of one assembled channel payload
};

// Stream descriptors.  The reference codes its candidates one after the other and only tries 17-19 bits if 16
// beat 15, else 14-12 (layer_encode.hpp:357-392).  A kernel launch here lasts as long as its longest stream
// whatever the number of streams, so BOTH directions are coded speculatively together with A, C and D in ONE
// round (round 0: 9 streams per plane at mode >= 1, just A at mode 0) and k_layer_decide looks only at the
// direction the reference would have taken.  Round 1: B = the predictor-index map at 8 bits (range = number of
// masks used), one stream per plane.
__device__ __forceinline__ uint32_t layer_slot_bits(uint32_t slot) {
    return slot == 0u ? 15u : slot == 2u ? 16u : slot == 3u ? 15u : slot <= 6u ? 13u + slot : 21u - slot;
}

// round 0: every candidate at once (speculative, small batches: a launch lasts as long as its longest stream);
// round 1: B; rounds 2 and 3 (large batches, bound by throughput: no wasted work): A, C, D, then the three
// candidates of the direction C and D decide, exactly the reference's order.
__device__ __forceinline__ uint32_t layer_round_streams(const LayerGeom& lg, int round) {
    return round == 0 ? (lg.mode ? 9u : 1u) : (round == 1 ? 1u : 3u);
}
__device__ __forceinline__ uint32_t layer_round_slot(int round, uint32_t k, bool up) {
    if (round == 0) return k == 0u ? 0u : k + 1u;  // A, then C, D, E..G up, E..G down
    if (round == 1) return 1u;
    if (round == 2) return k == 0u ? 0u : k + 1u;  // A, C, D
    return (up ? 4u : 7u) + k;
}

__global__ void k_layer_streams(LayerGeom lg, uint64_t n_planes, int round, const uint32_t* __restrict__ n_used,
                                const uint32_t* __restrict__ kept_px, const hoh_stream_result* __restrict__ results,
                                hoh_enc_stream* __restrict__ streams) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint32_t per_round = layer_round_streams(lg, round);
    if (i >= n_planes * per_round) return;
    const uint64_t p = i / per_round;
    const uint32_t k = (uint32_t)(i % per_round);
    const uint64_t resid0 = p * lg.per_pad, resid1 = (n_planes + p) * (uint64_t)lg.per_pad;
    hoh_enc_stream st;
    st.prefix_len = 0;
    for (int b = 0; b < 8; b++) st.prefix[b] = 0;
    st.reserved = lg.enc_flags;
    const bool up = round == 3 && results[p * kLayerSlots + 2].size < results[p * kLayerSlots + 3].size;  // :357
    const uint32_t slot = layer_round_slot(round, k, up);
    if (round != 1) {
        st.range = 1u << lg.depth;
        st.n = kept_px ? kept_px[p] : lg.per;  // residuals left after NUKE compaction (layer_encode.hpp:93-99, 328-333)
        st.sym_off = (slot != 0u && lg.cells != 0u) ? resid1 : resid0;
        st.prob_bits = layer_slot_bits(slot);
    } else {
        st.sym_off = 2u * n_planes * (uint64_t)lg.per_pad + p * lg.cells_pad;
        st.n = lg.cells;
        st.range = n_used[p];
        st.prob_bits = 8;
    }
    st.out_off = p * (uint64_t)lg.plane_bytes + lg.slot_off[slot];
    st.out_cap = lg.slot_cap[slot];
    streams[i] = st;
}

// After the predictor search: channel header bytes + the predictor-index symbols (layer_encode.hpp:276-306).
__global__ void k_layer_headers(LayerGeom lg, uint64_t n_planes, const uint8_t* __restrict__ index_lists,
                                uint16_t* __restrict__ symbols, uint32_t* __restrict__ n_used,
                                uint8_t* __restrict__ hdr, uint32_t* __restrict__ hdr_len) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    uint8_t* h = hdr + p * kLayerHdrCap;
    uint32_t at = 0;
    h[at++] = 0x10;  // layer_encode.hpp:57: prediction on, no compaction
    if (lg.cells == 0u) {  // :320-325 single predictor 0x0010
        h[at++] = 0;
        h[at++] = 0;
        h[at++] = 0x00;
        h[at++] = 0x10;
        n_used[p] = 1;
        hdr_len[p] = at;
        return;
    }
    const uint16_t masks[14] = {0x0001, 0x0002, 0x0020, 0x0010, 0xffbf, 0x0003, 0xfffd,
                                0xfffb, 0xfff7, 0xffef, 0xffdf, 0xff7f, 0xfdff, 0xffff};
    const uint8_t* idx = index_lists + p * lg.cells;
    uint32_t used = 0;
    for (uint32_t c = 0; c < lg.cells; c++) used |= 1u << idx[c];
    uint8_t remap[14];
    uint32_t count = 0;
    h[at++] = (uint8_t)(lg.xt - 1);
    h[at++] = (uint8_t)(lg.yt - 1);
    const uint32_t count_at = at++;
    for (uint32_t m = 0; m < 14; m++)
        if (used & (1u << m)) {  // :292-304 masks actually used, in stock order
            h[at++] = (uint8_t)(masks[m] >> 8);
            h[at++] = (uint8_t)(masks[m] & 0xff);
            remap[m] = (uint8_t)count++;
        }
    h[count_at] = (uint8_t)count;
    uint16_t* sym = symbols + 2u * n_planes * (uint64_t)lg.per_pad + p * lg.cells_pad;
    for (uint32_t c = 0; c < lg.cells; c++) sym[c] = remap[idx[c]];
    n_used[p] = count;
    hdr_len[p] = at;
}

// Histograms for round 0 of hoh_layer_encode_batch.  The nine candidates of a plane code the same residuals
// (A the fastpath ones, the other eight the searched ones) and differ only in prob_bits, so a plane needs two
// histograms, not nine: CTA (plane, which) counts once — one sub-histogram per warp, the residuals of a
// smooth image pile up on a few values and would serialise on one shared copy — and writes the result to the
// frequency row of every stream that uses it.
__global__ void __launch_bounds__(256) k_layer_histograms(uint64_t n_planes, uint32_t per_plane, uint32_t a_copies,
                                                          uint32_t b_first, uint32_t b_copies,
                                                          const hoh_enc_stream* __restrict__ streams,
                                                          const uint16_t* __restrict__ symbols,
                                                          uint32_t* __restrict__ freqs) {
    // streams of plane p: [p * per_plane, ...); the first a_copies of them code one residual array (A), the
    // b_copies from b_first on another (or the same): one count per array, written to each stream's row
    __shared__ uint32_t s_h[8][kFreqRow];
    const uint64_t p = blockIdx.x >> 1;
    const uint32_t which = blockIdx.x & 1u;
    const uint32_t copies = which ? b_copies : a_copies;
    if (copies == 0u) return;
    const uint64_t first = p * per_plane + (which ? b_first : 0u);
    const hoh_enc_stream st = streams[first];
    for (uint32_t i = threadIdx.x; i < 8u * kFreqRow; i += blockDim.x) (&s_h[0][0])[i] = 0;
    __syncthreads();
    const uint16_t* src = symbols + st.sym_off;
    uint32_t* mine = s_h[threadIdx.x >> 5];
    for (uint32_t i = threadIdx.x; i < st.n; i += blockDim.x) {
        const uint32_t v = src[i];
        if (v < st.range) atomicAdd(&mine[v], 1u);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < (uint32_t)kFreqRow; i += blockDim.x) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) t += s_h[w][i];
        for (uint32_t k = 0; k < copies; k++) freqs[(first + k) * kFreqRow + i] = t;
    }
}

// layer_encode.hpp:108-120, 326-398: which candidate's bytes are emitted and how many of them.
// fix == 0 reproduces the reference, including D7: when the 16- or 15-bit candidate wins the second stage only
// the SIZE is updated, so the emitted bytes are a stale buffer cut to that size.  fix != 0 (HOH_FIX_STALE) is
// the decodable variant: the smallest candidate's own bytes are kept, and when the plain fastpath stream (A)
// beats every searched candidate including their predictor-map overhead the channel is written with the
// single-predictor header A belongs to.
__global__ void k_layer_decide(LayerGeom lg, uint64_t n_planes, const hoh_stream_result* __restrict__ results,
                               uint32_t fix, uint8_t* __restrict__ hdr, uint32_t* __restrict__ hdr_len,
                               uint32_t* __restrict__ kept_slot, uint32_t* __restrict__ best_size,
                               uint32_t* __restrict__ with_idx, int32_t* __restrict__ status) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    const hoh_stream_result* r = results + p * kLayerSlots;
    const uint64_t bits = (uint64_t)lg.depth * lg.per;
    uint32_t best = (uint32_t)((bits + bits % 8 + 1024) / 8);  // :22
    uint32_t kept = 0xffffffffu;  // nothing kept: the reference would emit an uninitialised buffer
    uint32_t idx = lg.cells ? 1u : 0u;
    int32_t st = r[0].status;
    const bool up = lg.mode && r[2].size < r[3].size;  // layer_encode.hpp:357: 16 bits beat 15 -> try 17, 18, 19
    const uint32_t third = up ? 4u : 7u;               // first slot of the direction the reference takes
    if (lg.mode) {
        if (lg.cells) st = st ? st : r[1].status;
        st = st ? st : (r[2].status ? r[2].status : r[3].status);
        for (uint32_t k = 0; k < 3u; k++) st = st ? st : r[third + k].status;
    }
    if (fix) {
        best = r[0].size;
        kept = 0;
        if (lg.mode) {
            uint32_t sb = r[2].size, sk = 2;
            if (r[3].size < sb) {
                sb = r[3].size;
                sk = 3;
            }
            for (uint32_t k = third; k < third + 3u; k++)
                if (r[k].size < sb) {
                    sb = r[k].size;
                    sk = k;
                }
            const uint64_t searched = (uint64_t)sb + (lg.cells ? hdr_len[p] + r[1].size : 5u);
            if (searched < (uint64_t)r[0].size + 5u) {
                best = sb;
                kept = sk;
            } else if (lg.cells) {  // A under the header it was coded for: 10 | 00 00 | 00 10
                uint8_t* h = hdr + p * kLayerHdrCap;
                h[0] = 0x10;
                h[1] = 0;
                h[2] = 0;
                h[3] = 0x00;
                h[4] = 0x10;
                hdr_len[p] = 5;
                idx = 0;
            }
        }
    } else {
        if (r[0].size < best) {  // :115-120
            best = r[0].size;
            kept = 0;
        }
        if (lg.mode) {
            const uint32_t first = up ? r[2].size : r[3].size;
            if (first < best) best = first;  // size updated, buffers NOT swapped (D7): kept stays
            for (uint32_t k = 0; k < 3u; k++)
                if (r[third + k].size < best) {
                    best = r[third + k].size;
                    kept = third + k;
                }
        }
    }
    kept_slot[p] = kept;
    best_size[p] = best;
    with_idx[p] = idx;
    status[p] = st;
}

// Channel payload = header bytes | predictor-index stream | best_size bytes of the kept candidate.
// One CTA per plane.
__global__ void __launch_bounds__(256) k_layer_assemble(LayerGeom lg, const uint8_t* __restrict__ hdr,
                                                        const uint32_t* __restrict__ hdr_len,
                                                        const hoh_stream_result* __restrict__ results,
                                                        const uint32_t* __restrict__ kept_slot,
                                                        const uint32_t* __restrict__ best_size,
                                                        const uint32_t* __restrict__ with_idx,
                                                        const int32_t* __restrict__ status,
                                                        const uint8_t* __restrict__ cand, uint8_t* __restrict__ out,
                                                        uint64_t out_base, hoh_stream_result* __restrict__ final_results) {
    const uint64_t p = blockIdx.x;
    uint8_t* dst = out + out_base + p * (uint64_t)lg.out_cap;
    const hoh_stream_result* r = results + p * kLayerSlots;
    uint32_t at = hdr_len[p];
    for (uint32_t i = threadIdx.x; i < at; i += blockDim.x) dst[i] = hdr[p * kLayerHdrCap + i];
    if (with_idx[p]) {  // :308-317 the predictor-index stream follows the masks
        const uint8_t* src = cand + r[1].start;
        for (uint32_t i = threadIdx.x; i < r[1].size; i += blockDim.x) dst[at + i] = src[i];
        at += r[1].size;
    }
    const uint32_t kept = kept_slot[p], best = best_size[p];
    const uint32_t have = kept == 0xffffffffu ? 0u : r[kept].size;
    const uint8_t* src = kept == 0xffffffffu ? cand : cand + r[kept].start;
    for (uint32_t i = threadIdx.x; i < best; i += blockDim.x) dst[at + i] = i < have ? src[i] : (uint8_t)0;
    if (threadIdx.x == 0) {
        hoh_stream_result fr;
        fr.start = out_base + p * (uint64_t)lg.out_cap;
        fr.size = at + best;
        fr.status = status[p];
        fr.payload_bytes = best;
        fr.stored = kept;
        final_results[p] = fr;
    }
}

// round-local result order -> results[plane * kLayerSlots + slot]
__global__ void k_layer_scatter(LayerGeom lg, uint64_t n_planes, int round, const hoh_stream_result* __restrict__ rr,
                                hoh_stream_result* __restrict__ results) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint32_t per_round = layer_round_streams(lg, round);
    if (i >= n_planes * per_round) return;
    const uint64_t p = i / per_round;
    const uint32_t k = (uint32_t)(i % per_round);
    const bool up = round == 3 && results[p * kLayerSlots + 2].size < results[p * kLayerSlots + 3].size;
    results[p * kLayerSlots + layer_round_slot(round, k, up)] = rr[i];
}

// -------------------------------------------------------------------------------------------------
// Which candidates of a plane have to be CODED.  The reference codes all six on its path (A; C, D; three more in the
// direction C and D decide) and keeps one; a candidate's size, though, follows from its histogram and table up to one
// word (warp_estimate_words), so the decision sequence of k_layer_decide is replayed here over size INTERVALS.
// While every comparison comes out the same at both ends of the intervals involved, only two things are needed
// from the coder: the bytes of the candidate that ends up kept, and the exact size that ends up emitted when its
// interval is not a single number.  A plane with a comparison the intervals cannot settle has its whole path coded,
// as before.  need[9 * plane + k] = 1: round-0 stream k of the plane goes to the coder.
// -------------------------------------------------------------------------------------------------
struct SizeIv {
    uint32_t lo, hi;
};
__device__ __forceinline__ int iv_less(const SizeIv& a, const SizeIv& b) {  // a < b: 1 yes, 0 no, -1 depends
    return a.hi < b.lo ? 1 : (a.lo >= b.hi ? 0 : -1);
}
__global__ void k_layer_plan(LayerGeom lg, uint64_t n_planes, const hoh_enc_stream* __restrict__ streams,
                             const EncMeta* __restrict__ meta, const hoh_stream_result* __restrict__ results,
                             const uint32_t* __restrict__ hdr_len, uint32_t fix, uint32_t code_all,
                             uint8_t* __restrict__ need, uint32_t* __restrict__ counters) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    const uint32_t per = lg.mode ? 9u : 1u;
    SizeIv iv[kLayerSlots];
    bool exact[kLayerSlots];
    for (uint32_t k = 0; k < per; k++) {
        const uint32_t slot = layer_round_slot(0, k, false);
        const hoh_enc_stream st = streams[p * per + k];
        const EncMeta m = meta[p * per + k];
        const uint32_t lo = m.est & 0xffffffu, span = m.est >> 24;
        if (m.status != HOH_S_OK || st.n == 0u) {
            iv[slot].lo = iv[slot].hi = stream_size_for(st, m, 0u);
        } else if (span == 255u) {
            iv[slot].lo = 0u;
            iv[slot].hi = 0xffffffffu;
        } else {
            iv[slot].lo = stream_size_for(st, m, lo);
            iv[slot].hi = stream_size_for(st, m, lo + span);
        }
        exact[slot] = iv[slot].lo == iv[slot].hi;
    }
    uint32_t want = 0;  // bit per slot
    bool settled = !code_all;
    const uint64_t bits = (uint64_t)lg.depth * lg.per;
    const uint32_t bound = (uint32_t)((bits + bits % 8 + 1024) / 8);  // layer_encode.hpp:22
    int up = 0;
    if (settled && lg.mode) {
        up = iv_less(iv[2], iv[3]);  // layer_encode.hpp:357
        if (up < 0) settled = false;
    }
    const uint32_t third = up > 0 ? 4u : 7u;
    if (settled && !fix) {  // k_layer_decide, fix == 0
        SizeIv best{bound, bound};
        uint32_t best_slot = 0xffffffffu, kept = 0xffffffffu;
        int c = iv_less(iv[0], best);
        if (c < 0) settled = false;
        if (c > 0) {
            best = iv[0];
            best_slot = kept = 0u;
        }
        if (settled && lg.mode) {
            const uint32_t first = up > 0 ? 2u : 3u;
            c = iv_less(iv[first], best);
            if (c < 0) settled = false;
            if (c > 0) {
                best = iv[first];
                best_slot = first;
            }
            for (uint32_t k = 0; settled && k < 3u; k++) {
                c = iv_less(iv[third + k], best);
                if (c < 0) settled = false;
                if (c > 0) {
                    best = iv[third + k];
                    best_slot = kept = third + k;
                }
            }
        }
        if (settled) {
            if (kept != 0xffffffffu) want |= 1u << kept;
            if (best_slot != 0xffffffffu && !exact[best_slot]) want |= 1u << best_slot;
        }
    } else if (settled) {  // k_layer_decide, fix != 0: the smallest searched candidate against A
        uint32_t kept = 0u;
        if (lg.mode) {
            uint32_t sk = 2u;
            int c = iv_less(iv[3], iv[2]);
            if (c < 0) settled = false;
            if (c > 0) sk = 3u;
            for (uint32_t k = third; settled && k < third + 3u; k++) {
                c = iv_less(iv[k], iv[sk]);
                if (c < 0) settled = false;
                if (c > 0) sk = k;
            }
            if (settled) {
                const uint32_t extra = lg.cells ? hdr_len[p] + results[p * kLayerSlots + 1].size : 5u;
                const SizeIv searched{iv[sk].lo + extra, iv[sk].hi + extra}, plain{iv[0].lo + 5u, iv[0].hi + 5u};
                c = iv_less(searched, plain);
                if (c < 0) settled = false;
                if (c > 0) kept = sk;
            }
        }
        if (settled) want |= 1u << kept;
    }
    if (!settled) {  // the reference's whole path (both directions when even that comparison is open)
        want = 1u;
        if (lg.mode) want |= (1u << 2) | (1u << 3) | (code_all || up < 0 ? 0x3f0u : (7u << third));
    }
    uint32_t n_want = 0;
    for (uint32_t k = 0; k < per; k++) {
        const uint32_t on = (want >> layer_round_slot(0, k, false)) & 1u;
        need[p * per + k] = (uint8_t)on;
        n_want += on;
    }
    if (counters) {
        atomicAdd(&counters[0], n_want);
        if (!settled) atomicAdd(&counters[1], 1u);
        atomicAdd(&counters[2], 1u);
    }
}

// need[] -> the dense list of stream indices the coder walks, and their number.  The streams with 16-bit table lanes
// (prob_bits <= 15) come first, then those with 32-bit lanes, each group ascending: a warp of the coder serves one
// table width per launch, and a warp with both would run twice with half of its lanes idle.  One CTA.
__global__ void __launch_bounds__(1024) k_layer_order(const uint8_t* __restrict__ need,
                                                      const hoh_enc_stream* __restrict__ streams, uint32_t count,
                                                      uint32_t* __restrict__ order, uint32_t* __restrict__ n_active) {
    __shared__ uint32_t s_a[1024], s_b[1024];
    const uint32_t per = (count + 1023u) / 1024u;
    const uint32_t lo = min(count, threadIdx.x * per), hi = min(count, lo + per);
    uint32_t mine_a = 0, mine_b = 0;
    for (uint32_t i = lo; i < hi; i++)
        if (need[i]) {
            if (streams[i].prob_bits <= 15u) mine_a++;
            else mine_b++;
        }
    s_a[threadIdx.x] = mine_a;
    s_b[threadIdx.x] = mine_b;
    __syncthreads();
    for (uint32_t d = 1; d < 1024u; d <<= 1) {
        const uint32_t va = threadIdx.x >= d ? s_a[threadIdx.x - d] : 0u, vb = threadIdx.x >= d ? s_b[threadIdx.x - d] : 0u;
        __syncthreads();
        s_a[threadIdx.x] += va;
        s_b[threadIdx.x] += vb;
        __syncthreads();
    }
    uint32_t at_a = s_a[threadIdx.x] - mine_a, at_b = s_a[1023] + s_b[threadIdx.x] - mine_b;
    for (uint32_t i = lo; i < hi; i++)
        if (need[i]) {
            if (streams[i].prob_bits <= 15u) order[at_a++] = i;
            else order[at_b++] = i;
        }
    if (threadIdx.x == 1023u) *n_active = s_a[1023] + s_b[1023];
}

// The round's result records for candidates that are NOT coded: status and the lower end of the size interval (the
// plan made sure that no decision depends on where in the interval the size lies); k_finish_streams then overwrites
// the records of the coded ones.
__global__ void k_layer_est_results(uint64_t count, const hoh_enc_stream* __restrict__ streams,
                                    const EncMeta* __restrict__ meta, hoh_stream_result* __restrict__ rr) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const hoh_enc_stream st = streams[i];
    const EncMeta m = meta[i];
    hoh_stream_result r;
    r.status = m.status;
    r.start = st.out_off;
    r.size = stream_size_for(st, m, m.est & 0xffffffu);
    r.payload_bytes = 0;
    r.stored = 0;
    rr[i] = r;
}

// =================================================================================================
// lz.hpp:6-145 — the LZ match finder (SURVEY §8(f) row 1), for many tiles.
//
// The reference walks the pixels greedily and, at every pixel it lands on, tries every distance and extends
// each candidate pixel by pixel.  Here the two halves are separated:
//   k_lz_match  computes (longest run, first distance reaching it) for EVERY pixel, all pixels in parallel —
//               exactly what the reference would compute if it landed there;
//   k_lz_walk   replays the greedy walk over those answers (a warp per tile, 32 pixels per step) and emits
//               the four side streams and the NUKE map.
// Run lengths are not found by extension: for a fixed distance b the equality bits e_b[i] = (px[i] ==
// px[i-b]) of 32 consecutive pixels are one warp ballot, and the run starting at pixel i is the number of
// consecutive ones from bit i on, continued into the following ballot words.  Walking a segment backwards
// the continuation is ONE warp-uniform number (the run length at the start of the next word), so a
// (distance, 32 pixels) pair costs one load, one compare, one ballot and — only if some pixel matched — a
// shift / count-trailing-ones per lane, whatever the image content is (flat images do not blow up).
// =================================================================================================
constexpr int kLzSeg = 1024;      // pixels per warp: 32 words of 32 pixels, one (run, distance) register each
constexpr int kLzMaxRun = 259;    // lz.hpp:42
constexpr int kLzAhead = 9;       // 32-pixel words of look-ahead that a capped run can reach into
constexpr uint32_t kLzBackBits = 17;  // distances go up to 65536 (lz.hpp:54)

// Where the tiles are.  tiled == 0: n contiguous tiles of npx pixels (row length `width`), `stride` elements
// apart in every per-pixel array.  tiled == 1: the tiles of whole images cut as choh.cpp:454-484 cuts them
// (edge tiles may be smaller), per-pixel arrays still `stride` elements per tile.
struct LzShape {
    uint32_t tiled, npx, width, stride;
    uint32_t pad;        // never-matching words in front of every tile's packed pixels (>= 2^distance)
    uint32_t px_stride;  // words per tile in the packed-pixel array: pad + segments * kLzSeg + 32 * kLzAhead
    TileSel sel;         // tiled == 1: which tiles (the whole grid, or the tiles of one shape)
};

__device__ __forceinline__ void lz_dims(const LzShape& sh, uint64_t tile, uint32_t& npx, uint32_t& width) {
    if (!sh.tiled) {
        npx = sh.npx;
        width = sh.width;
        return;
    }
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sh.sel, tile, image, in_image, x0, y0, tw, th);
    npx = tw * th;
    width = tw;
}

// px[tile * px_stride + pad + i] = R | G << 8 | B << 16 of the tile's i-th pixel, framed by words that equal
// no pixel and no other framing word at any distance (top byte set, low bits = position), so the match kernel
// needs no bounds tests for distances up to `pad`.  One CTA per tile.
__global__ void __launch_bounds__(256) k_lz_pack(const uint8_t* __restrict__ rgb, LzShape sh,
                                                 uint32_t* __restrict__ px) {
    const uint64_t tile = blockIdx.x;
    uint32_t* base = px + tile * sh.px_stride;
    uint32_t* dst = base + sh.pad;
    uint32_t npx, width;
    lz_dims(sh, tile, npx, width);
    for (uint32_t i = threadIdx.x; i < sh.pad; i += blockDim.x) base[i] = 0xfe000000u | i;
    for (uint32_t i = npx + threadIdx.x; i < sh.px_stride - sh.pad; i += blockDim.x) dst[i] = 0xff000000u | (i & 0xffffffu);
    if (!sh.tiled) {
        const uint8_t* src = rgb + tile * (uint64_t)sh.npx * 3u;
        for (uint32_t i = threadIdx.x; i < sh.npx; i += blockDim.x) {
            const uint8_t* p = src + i * 3u;
            dst[i] = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16);
        }
        return;
    }
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sh.sel, tile, image, in_image, x0, y0, tw, th);
    const uint8_t* img = rgb + image * (uint64_t)sh.sel.g.width * sh.sel.g.height * 3u;
    for (uint32_t i = threadIdx.x; i < tw * th; i += blockDim.x) {
        const uint32_t x = i % tw, y = i / tw;
        const uint8_t* p = img + ((uint64_t)(y0 + y) * sh.sel.g.width + x0 + x) * 3u;
        dst[i] = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16);
    }
}

// trailing ones of w (32 when w is all ones)
__device__ __forceinline__ uint32_t lz_ones(uint32_t w) { return w == 0xffffffffu ? 32u : (uint32_t)(__ffs((int)~w) - 1); }

// A candidate is ranked by key = run << 17 | (0x1ffff - distance): the largest key is the longest run and,
// among equally long runs, the smallest distance — which is what the reference's two ascending loops with a
// strict '>' keep (lz.hpp:47, :65; the row distances of the second loop that are <= 2^distance repeat
// distances of the first, the others are larger than all of them).  A max is order-independent, so the
// distances can be visited in whatever order is cheapest.
__device__ __forceinline__ uint32_t lz_key(uint32_t run, uint32_t b) { return (run << kLzBackBits) | (0x1ffffu - b); }

// One distance for one 1024-pixel segment, exact run lengths.  CHECK = the segment touches the tile's ends
// (or the distance reaches before the tile's first pixel), so every access is bounds-tested.
template <bool CHECK>
__device__ __forceinline__ void lz_one_distance(const uint32_t* __restrict__ P, uint32_t npx, uint32_t s0,
                                             uint32_t lane, uint32_t b, const uint32_t (&mine)[32],
                                             uint32_t (&best)[32]) {
    // run length at the first pixel after the segment: forward over the look-ahead words until one breaks
    uint32_t carry = 0;
    for (uint32_t k = 32; k < 32u + kLzAhead; k++) {
        const uint32_t i = s0 + 32u * k + lane;
        bool e;
        if (CHECK) e = i < npx && i >= b && P[i] == P[i - b];
        else e = P[i] == P[i - b];
        const uint32_t w = __ballot_sync(0xffffffffu, e);
        carry += lz_ones(w);
        if (w != 0xffffffffu) break;
    }
    const uint32_t* q = P + s0 + lane - b;  // only dereferenced where s0 + 32k + lane >= b
#pragma unroll
    for (int k = 31; k >= 0; k--) {
        bool e;
        if (CHECK) {
            const uint32_t i = s0 + 32u * k + lane;
            e = i < npx && i >= b && mine[k] == q[32 * k];
        } else {
            e = mine[k] == q[32 * k];
        }
        const uint32_t w = __ballot_sync(0xffffffffu, e);
        if (w) {  // warp-uniform
            const uint32_t t = w >> lane;
            const uint32_t ones = lz_ones(t);  // bits above 31 - lane are zero: ones <= 32 - lane
            uint32_t len = ones == 32u - lane ? ones + carry : ones;
            len = min(len, (uint32_t)kLzMaxRun);
            if (len) best[k] = max(best[k], lz_key(len, b));
            carry = w == 0xffffffffu ? carry + 32u : lz_ones(w);
        } else {
            carry = 0;
        }
    }
}

// M distances r + 32 * (c0 + j), j = 0 .. M-1, for a segment all of whose partner pixels exist.  The word a
// lane compares block k with at distance b + 32 is the word it compares block k - 1 with at distance b, so
// 32 + M - 1 loads serve 32 * M comparisons; a distance none of whose 1024 comparisons hits (the normal case
// on photographic content) costs one compare per 32 pixels and nothing else.
template <int M, int R>
__device__ __forceinline__ void lz_distance_group(const uint32_t* __restrict__ P, uint32_t npx, uint32_t s0,
                                                  uint32_t lane, uint32_t r, uint32_t c0, bool exact_inside,
                                                  const uint32_t (&mine)[32], uint32_t (&best)[32]) {
    // R consecutive residues r .. r + R - 1 share one round of loads (more loads in flight per warp)
    uint32_t v[R][32 + M - 1];
#pragma unroll
    for (int u = 0; u < R; u++) {
        const uint32_t* q = P + s0 + lane - (r + u) - 32u * c0;
#pragma unroll
        for (int t = 0; t < 32 + M - 1; t++) v[u][t] = q[32 * (t - (M - 1))];
    }
    uint32_t hit_mask = 0;
#pragma unroll
    for (int u = 0; u < R; u++)
#pragma unroll
        for (int j = 0; j < M; j++) {
            bool any = false;
#pragma unroll
            for (int k = 0; k < 32; k++) any |= mine[k] == v[u][k + (M - 1) - j];
            hit_mask |= __any_sync(0xffffffffu, any) ? (1u << (u * M + j)) : 0u;
        }
    while (hit_mask) {  // warp-uniform, rare
        const uint32_t bit = (uint32_t)__ffs((int)hit_mask) - 1u;
        hit_mask &= hit_mask - 1u;
        const uint32_t b = r + bit / M + 32u * (c0 + bit % M);
        if (exact_inside) lz_one_distance<false>(P, npx, s0, lane, b, mine, best);
        else lz_one_distance<true>(P, npx, s0, lane, b, mine, best);
    }
}

// state[tile * stride + i] = longest << 17 | distance  (longest 0 when nothing matches)
__global__ void __launch_bounds__(128) k_lz_match(const uint32_t* __restrict__ px, LzShape sh, uint64_t n_tiles,
                                                  uint32_t near_limit, uint32_t wide,
                                                  uint32_t* __restrict__ state,
                                                  const uint32_t* __restrict__ only_flagged) {
    // wide: 0 = near window only (lz.hpp:53: distance <= 8), else the largest whole-row distance tried.  The reference
    // goes up to 65536 inclusive (lz.hpp:54) and then stores the distance in two bytes, so 65536 is written as 0
    // (lz.hpp:88-89): byte-exact, but no decoder can tell it from "no distance".  With HOH_FIX_LONE the encoder stops
    // at 65535, which costs one candidate distance and keeps every tile decodable.
    const uint32_t lane = lane_id();
    const uint32_t segs = (sh.stride + kLzSeg - 1) / kLzSeg;
    const uint64_t wid = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (wid >= n_tiles * segs) return;
    const uint64_t tile = wid / segs;
    const uint32_t s0 = (uint32_t)(wid % segs) * kLzSeg;
    uint32_t npx, width;
    lz_dims(sh, tile, npx, width);
    if (s0 >= npx) return;
    if (only_flagged && only_flagged[tile] == 0u) return;  // the sparse pass has answered this tile
    const uint32_t* P = px + tile * sh.px_stride + sh.pad;
    uint32_t mine[32], best[32];
#pragma unroll
    for (int k = 0; k < 32; k++) {
        const uint32_t i = s0 + 32u * k + lane;
        mine[k] = i < npx ? P[i] : 0xfd000000u;  // equals nothing in memory
        best[k] = 0;
    }
    // The framing words make every access for a distance b <= s0 + pad an in-bounds access that cannot
    // match, in front of the tile and behind it: no bounds tests on the near window (pad >= near_limit).
    // lz.hpp:34-52: every distance 1 .. 2^distance
    uint32_t done = 0;  // distances 1 .. done are finished
    {
        constexpr int M = 8;
        const uint32_t full = near_limit / (32u * M);
        for (uint32_t c = 0; c < full; c++)
            for (uint32_t r = 1; r <= 32u; r++) lz_distance_group<M, 1>(P, npx, s0, lane, r, c * M, true, mine, best);
        done = full * 32u * M;
        while (near_limit - done >= 64u) {  // the 2^6 window, or the tail of another one
            for (uint32_t r = 1; r <= 32u; r += 2) lz_distance_group<2, 2>(P, npx, s0, lane, r, done / 32u, true, mine, best);
            done += 64u;
        }
    }
    for (uint32_t b = done + 1u; b <= near_limit; b++) lz_one_distance<false>(P, npx, s0, lane, b, mine, best);
    // lz.hpp:53-74: whole rows up, multiples of the width up to 65536
    if (wide) {
        const uint32_t last = min(s0 + kLzSeg, npx) - 1u;  // highest pixel of the segment: larger distances reach nothing
        for (uint32_t b = width; b <= wide && b <= last; b += width) {  // wide = the largest row distance: 65536, see below
            const bool framed = b <= s0 + sh.pad;
            if (framed) {  // quick test first: one load and one compare per 32 pixels
                const uint32_t* q = P + s0 + lane - b;
                bool any = false;
#pragma unroll
                for (int k = 0; k < 32; k++) any |= mine[k] == q[32 * k];
                if (!__any_sync(0xffffffffu, any)) continue;
                lz_one_distance<false>(P, npx, s0, lane, b, mine, best);
            } else {
                lz_one_distance<true>(P, npx, s0, lane, b, mine, best);
            }
        }
    }
    uint32_t* S = state + tile * sh.stride;
#pragma unroll
    for (int k = 0; k < 32; k++) {
        const uint32_t i = s0 + 32u * k + lane;
        if (i < npx) S[i] = (best[k] & ~0x1ffffu) | (0x1ffffu - (best[k] & 0x1ffffu));
    }
}

// -------------------------------------------------------------------------------------------------
// Sparse candidates for wide seek windows.  Only runs of at least 4 pixels can become matches (lz.hpp:75:
// longest >= 4 + bonus), and such a run starts with four equal pixels on both sides.  So instead of testing every
// distance, the positions of a tile are chained by a 16-bit hash of their next four pixels (one atomic exchange
// per position into a table of chain heads) and a pixel only looks at the earlier positions of its own chain: on
// photographic content a chain has a couple of entries.  The order of a chain does not matter — the best
// candidate is a maximum (lz_key).  A tile with a chain longer than kLzChainLimit (flat or periodic content)
// raises a flag and is redone by the dense kernel; the others are skipped there.  The answers for pixels whose
// longest run is shorter than 4 differ from the dense kernel's (0 instead of 1..3) — the walk never looks at those.
// -------------------------------------------------------------------------------------------------
constexpr uint32_t kLzChainLimit = 64;
constexpr uint32_t kLzHeads = 1u << 16;  // chain heads per tile

__device__ __forceinline__ uint32_t lz_hash4(const uint32_t* __restrict__ P, uint32_t i) {  // 16 bits
    uint32_t h = P[i] * 0x9E3779B1u;
    h = (h ^ (h >> 15)) + P[i + 1u] * 0x85EBCA77u;
    h = (h ^ (h >> 13)) + P[i + 2u] * 0xC2B2AE3Du;
    h = (h ^ (h >> 16)) + P[i + 3u] * 0x27D4EB2Fu;
    h ^= h >> 15;
    return (h * 0x2C1B3C6Du) >> 16;
}

// heads: kLzHeads words per tile, all ones (empty) on entry; next: `stride` words per tile.
__global__ void __launch_bounds__(256) k_lz_chains(const uint32_t* __restrict__ px, LzShape sh, uint64_t n_tiles,
                                                   uint32_t* __restrict__ heads, uint32_t* __restrict__ next) {
    const uint32_t bpt = (sh.stride + 255u) / 256u;  // CTAs per tile
    const uint64_t tile = blockIdx.x / bpt;
    const uint32_t i = (blockIdx.x % bpt) * 256u + threadIdx.x;
    if (tile >= n_tiles) return;
    uint32_t npx, width_unused;
    lz_dims(sh, tile, npx, width_unused);
    if (i >= npx) return;
    const uint32_t* P = px + tile * sh.px_stride + sh.pad;  // the framing words make P[i + 3] readable
    next[tile * sh.stride + i] = atomicExch(&heads[tile * kLzHeads + lz_hash4(P, i)], i);
}

// One thread per position: the earlier positions of its chain are its only candidates.
__global__ void __launch_bounds__(256) k_lz_match_sparse(const uint32_t* __restrict__ px, LzShape sh, uint64_t n_tiles,
                                                         uint32_t near_limit, uint32_t row_limit, const uint32_t* __restrict__ heads,
                                                         const uint32_t* __restrict__ next,
                                                         uint32_t* __restrict__ state, uint32_t* __restrict__ dense_flag) {
    const uint32_t bpt = (sh.stride + 255u) / 256u;
    const uint64_t tile = blockIdx.x / bpt;
    const uint32_t i = (blockIdx.x % bpt) * 256u + threadIdx.x;
    if (tile >= n_tiles) return;
    uint32_t npx, width;
    lz_dims(sh, tile, npx, width);
    if (i >= npx) return;
    const uint32_t* P = px + tile * sh.px_stride + sh.pad;
    const uint32_t* N = next + tile * sh.stride;
    uint32_t best = 0, seen = 0;
    for (uint32_t j = heads[tile * kLzHeads + lz_hash4(P, i)]; j != 0xffffffffu; j = N[j]) {
        if (++seen > kLzChainLimit) {
            atomicOr(&dense_flag[tile], 1u);
            break;
        }
        if (j >= i) continue;  // itself, or a later position
        const uint32_t b = i - j;
        if (!(b <= near_limit || (b <= row_limit && b % width == 0u))) continue;  // lz.hpp:34, :54
        uint32_t run = 0;
        while (run < (uint32_t)kLzMaxRun && i + run < npx && P[i + run] == P[j + run]) run++;
        if (run >= 4u) best = max(best, lz_key(run, b));
    }
    state[tile * sh.stride + i] = best ? ((best & ~0x1ffffu) | (0x1ffffu - (best & 0x1ffffu))) : 0x1ffffu;
}

// choh.cpp:17-50 + :134-154: distinct colours of a tile (more than 256 = "many") -> break-even bonus.
// One CTA per tile, open-addressing hash set in shared memory.
// info (optional): bit 31 = every pixel is grey (grey_test channel.hpp:21), low bits = colours (257 = more than 256)
__global__ void __launch_bounds__(256) k_lz_bonus(const uint32_t* __restrict__ px, LzShape sh,
                                                  int32_t* __restrict__ bonus, uint32_t* __restrict__ info) {
    uint32_t npx, width_unused;
    lz_dims(sh, blockIdx.x, npx, width_unused);
    __shared__ uint32_t s_set[1024];
    __shared__ uint32_t s_count;
    for (uint32_t i = threadIdx.x; i < 1024u; i += blockDim.x) s_set[i] = 0xffffffffu;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    const uint32_t* P = px + (uint64_t)blockIdx.x * sh.px_stride + sh.pad;
    volatile uint32_t* seen = &s_count;
    for (uint32_t base = 0; base < npx; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        if (i < npx && *seen <= 256u) {
            const uint32_t v = P[i];
            uint32_t h = (v * 2654435761u) >> 22;
            for (;;) {
                const uint32_t old = atomicCAS(&s_set[h], 0xffffffffu, v);
                if (old == 0xffffffffu) {
                    atomicAdd(&s_count, 1u);
                    break;
                }
                if (old == v) break;
                h = (h + 1u) & 1023u;
                if (*seen > 256u) break;  // the set cannot fill up: at most 257 + 256 in-flight inserts
            }
        }
        if (__syncthreads_or(*seen > 256u)) break;  // same answer in every thread
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t c = *seen;
        bonus[blockIdx.x] = c > 256u ? 0 : (c <= 4u ? 32 : (c <= 8u ? 20 : (c <= 16u ? 10 : (c <= 32u ? 2 : 0))));
    }
    if (info) {
        bool grey = true;
        for (uint32_t i = threadIdx.x; i < npx; i += blockDim.x) {
            const uint32_t v = P[i];
            grey &= (v & 0xffu) == ((v >> 8) & 0xffu) && (v & 0xffu) == (v >> 16);
        }
        const int all_grey = __syncthreads_and(grey);
        if (threadIdx.x == 0) info[blockIdx.x] = min(*seen, 257u) | (all_grey ? 0x80000000u : 0u);
    }
}

// The greedy walk (lz.hpp:33, 75-96) over the per-pixel answers.  One warp per tile.  side: u16 symbol
// buffers, 4 per tile, side_stride elements apart (since_last, length - 4, distance % 256, distance / 256);
// counts[tile * 4 + k] = symbols in each.
__global__ void __launch_bounds__(128) k_lz_walk(const uint32_t* __restrict__ state, LzShape sh, uint64_t n_tiles,
                                                 const int32_t* __restrict__ bonus, int32_t fixed_bonus, uint32_t wide,
                                                 uint8_t* __restrict__ nuke, uint32_t nuke_stride,
                                                 uint16_t* __restrict__ side, uint32_t side_stride,
                                                 uint32_t* __restrict__ counts) {
    const uint32_t lane = lane_id();
    const uint64_t tile = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (tile >= n_tiles) return;
    uint32_t npx, width_unused;
    lz_dims(sh, tile, npx, width_unused);
    const uint32_t* S = state + tile * sh.stride;
    uint8_t* N = nuke + tile * nuke_stride;
    uint16_t* side0 = side + (tile * 4u) * side_stride;
    uint16_t* side1 = side0 + side_stride;
    uint16_t* side2 = side1 + side_stride;
    uint16_t* side3 = side2 + side_stride;
    const uint32_t threshold = 4u + (uint32_t)(bonus ? bonus[tile] : fixed_bonus);  // lz.hpp:75
    uint32_t pos = 0, gap = 0, c0 = 0, c1 = 0;  // c1 counts matches: the other three streams grow together
    uint32_t v = lane < npx ? S[lane] : 0u;
    while (pos < npx) {
        const uint32_t i = pos + lane;
        // the block after this one is requested now: when nothing matches here (the usual case) the walk
        // continues with it and the chain of dependent loads is off the critical path
        const uint32_t ahead = i + 32u < npx ? S[i + 32u] : 0u;
        const uint32_t hits = __ballot_sync(0xffffffffu, i < npx && (v >> kLzBackBits) >= threshold);
        const uint32_t room = min(32u, npx - pos);
        const uint32_t skipped = hits ? (uint32_t)(__ffs((int)hits) - 1) : room;  // pixels without a match
        if (lane < skipped) N[i] = 0;
        gap += skipped;
        if (gap >= 255u) {  // lz.hpp:77-81 (at most once: skipped <= 32)
            if (lane == 0) side0[c0] = 255;
            c0++;
            gap -= 255u;
        }
        pos += skipped;
        if (!hits) {
            v = ahead;
            continue;
        }
        const uint32_t m = __shfl_sync(0xffffffffu, v, (int)skipped);
        const uint32_t len = m >> kLzBackBits, back = m & ((1u << kLzBackBits) - 1u);
        if (lane == 0) {  // lz.hpp:85-91
            side0[c0] = (uint16_t)gap;
            side1[c1] = (uint16_t)(len - 4u);
            side2[c1] = (uint16_t)(back & 255u);
            if (wide) side3[c1] = (uint16_t)((back >> 8) & 255u);
        }
        c0++;
        c1++;
        gap = 0;
        for (uint32_t k = lane; k < len; k += 32) N[pos + k] = 1;  // lz.hpp:92-94
        pos += len;                                                 // :95
        v = pos + lane < npx ? S[pos + lane] : 0u;
    }
    if (lane == 0) {
        counts[tile * 4u + 0] = c0;
        counts[tile * 4u + 1] = c1;
        counts[tile * 4u + 2] = c1;
        counts[tile * 4u + 3] = wide ? c1 : 0u;
    }
}

// descriptors of the 4 side streams of every tile (lz.hpp:102-141: range 256, 10 bits)
__global__ void k_lz_streams(uint64_t n_tiles, const uint32_t* __restrict__ counts, uint32_t side_stride,
                             uint32_t slab, uint32_t enc_flags, hoh_enc_stream* __restrict__ streams) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n_tiles * 4u) return;
    hoh_enc_stream st;
    st.sym_off = i * side_stride;
    st.n = counts[i];
    st.range = 256;
    st.prob_bits = 10;
    st.prefix_len = 0;
    for (int b = 0; b < 8; b++) st.prefix[b] = 0;
    st.out_off = i * (uint64_t)slab;
    st.out_cap = slab;
    st.reserved = enc_flags;
    streams[i] = st;
}

// LEMPEL bytes of a tile = 0x03 | stream 0 | stream 1 | stream 2 [| stream 3]  (lz.hpp:100-142).  One CTA per tile.
__global__ void __launch_bounds__(128) k_lz_assemble(const hoh_stream_result* __restrict__ results,
                                                     const uint8_t* __restrict__ slabs, uint32_t wide,
                                                     uint8_t* __restrict__ lz, uint32_t lz_stride,
                                                     uint32_t* __restrict__ lz_size, int32_t* __restrict__ status) {
    const uint64_t tile = blockIdx.x;
    uint8_t* dst = lz + tile * lz_stride;
    uint32_t at = 1;
    int32_t st = HOH_S_OK;
    if (threadIdx.x == 0) dst[0] = 0x03;
    for (uint32_t k = 0; k < (wide ? 4u : 3u); k++) {
        const hoh_stream_result r = results[tile * 4u + k];
        st = st ? st : r.status;
        const uint32_t size = at + r.size <= lz_stride ? r.size : 0u;
        if (size != r.size) st = st ? st : HOH_S_OVERFLOW;
        const uint8_t* src = slabs + r.start;
        for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) dst[at + i] = src[i];
        at += size;
    }
    if (threadIdx.x == 0) {
        lz_size[tile] = at;
        if (status) status[tile] = st;
    }
}

// layer_encode.hpp:93-99: residuals of LZ-covered pixels are dropped (stable compaction, in place).  One
// warp per stream; the stream descriptor's symbol count becomes the number of kept residuals.
__global__ void __launch_bounds__(128) k_compact_nuke(TileGeom g, uint64_t n_tiles, const uint8_t* __restrict__ nuke,
                                                      uint32_t nuke_stride, uint16_t* __restrict__ resid,
                                                      hoh_enc_stream* __restrict__ streams) {
    const uint32_t lane = lane_id();
    const uint64_t s = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (s >= n_tiles * 3u) return;
    const uint64_t t = s / 3u;
    uint32_t x0, y0, tw, th;
    tile_rect(g, (uint32_t)(t % g.tiles_per_image), x0, y0, tw, th);
    const uint32_t n = tw * th;
    const uint8_t* N = nuke + t * nuke_stride;
    uint16_t* R = resid + s * g.plane_stride;
    uint32_t kept = 0;
    for (uint32_t base = 0; base < n; base += 32) {
        const uint32_t i = base + lane;
        const bool keep = i < n && N[i] == 0;
        const uint16_t v = i < n ? R[i] : (uint16_t)0;
        const uint32_t m = __ballot_sync(0xffffffffu, keep);
        __syncwarp();  // every lane has read its element before any lane overwrites an earlier position
        if (keep) R[kept + __popc(m & ((1u << lane) - 1u))] = v;
        kept += __popc(m);
    }
    if (lane == 0) streams[s].n = kept;
}

// layer_encode.hpp:93-99 / 328-333 for plane residuals: plane p uses NUKE map p / planes_per_map.  In place,
// one warp per plane; kept_px[p] = residuals left.
__global__ void __launch_bounds__(128) k_compact_planes(uint64_t n_planes, uint32_t per, uint64_t plane_stride,
                                                        const uint8_t* __restrict__ nuke, uint64_t nuke_stride,
                                                        uint32_t planes_per_map, uint16_t* __restrict__ resid,
                                                        uint32_t* __restrict__ kept_px) {
    const uint32_t lane = lane_id();
    const uint64_t p = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (p >= n_planes) return;
    const uint8_t* N = nuke + (p / planes_per_map) * nuke_stride;
    uint16_t* R = resid + p * plane_stride;
    uint32_t kept = 0;
    for (uint32_t base = 0; base < per; base += 32) {
        const uint32_t i = base + lane;
        const bool keep = i < per && N[i] == 0;
        const uint16_t v = i < per ? R[i] : (uint16_t)0;
        const uint32_t m = __ballot_sync(0xffffffffu, keep);
        __syncwarp();
        if (keep) R[kept + __popc(m & ((1u << lane) - 1u))] = v;
        kept += __popc(m);
    }
    if (lane == 0) kept_px[p] = kept;
}

// channel.hpp:63-71: one channel of interleaved bytes -> u16 plane
__global__ void k_channel_picker(const uint8_t* __restrict__ src, uint64_t n_px, uint32_t total, uint32_t target,
                                 uint16_t* __restrict__ out) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_px; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = src[i * total + target];
}

// =================================================================================================
// encode_tile (choh.cpp:104-382) for the tiles of whole images, photographic colour modes: what is left
// around the LZ finder and the batched layer_encode — colour planes of a tile, the colour-mode comparison
// and the emission of the tile's bytes.
// =================================================================================================
// planes8[(t * per8 + k) * npx]: k = 0 green, and (per8 == 3, cruncher mode > 2: choh.cpp:263-290) 1 red, 2 blue;
// planes9[(t * 2 + k) * npx]: R - G + 256, B - G + 256 (channel.hpp:73-79).  One CTA per tile, uniform tiles.
__global__ void __launch_bounds__(256) k_tile_planes(const uint8_t* __restrict__ rgb, TileSel sel, uint32_t per8,
                                                     uint16_t* __restrict__ planes8,
                                                     uint16_t* __restrict__ planes9) {
    const uint64_t lt = blockIdx.x;
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sel, lt, image, in_image, x0, y0, tw, th);
    const TileGeom& g = sel.g;
    const uint32_t npx = tw * th;
    const uint8_t* img = rgb + image * (uint64_t)g.width * g.height * 3u;
    uint16_t* p8 = planes8 + lt * per8 * (uint64_t)npx;
    uint16_t* p9 = planes9 + lt * 2u * (uint64_t)npx;
    for (uint32_t i = threadIdx.x; i < npx; i += blockDim.x) {
        const uint32_t x = i % tw, y = i / tw;
        const uint8_t* p = img + ((uint64_t)(y0 + y) * g.width + x0 + x) * 3u;
        const uint32_t r = p[0], gr = p[1], b = p[2];
        p8[i] = (uint16_t)gr;
        if (per8 == 3u) {
            p8[npx + i] = (uint16_t)r;
            p8[2u * npx + i] = (uint16_t)b;
        }
        p9[i] = (uint16_t)(r + 256u - gr);
        p9[npx + i] = (uint16_t)(b + 256u - gr);
    }
}

constexpr uint32_t kTileGrey = 1u, kTilePalette = 2u;  // = HOH_TILE_GREY, HOH_TILE_PALETTE

// choh.cpp:295-327 (without the palette competitor) + sizes of what :328-363 emits.  One thread per tile.
__global__ void k_tile_decide(uint64_t n_tiles, TileSel sel, uint64_t first_image, uint32_t per8,
                              const hoh_stream_result* __restrict__ res8, const hoh_stream_result* __restrict__ res9,
                              const uint32_t* __restrict__ lz_size, const int32_t* __restrict__ lz_status,
                              const uint32_t* __restrict__ info, hoh_tile_result* __restrict__ tiles) {
    const uint64_t lt = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (lt >= n_tiles) return;
    const hoh_stream_result g = res8[lt * per8], rg = res9[lt * 2u], bg = res9[lt * 2u + 1u];
    hoh_tile_result tr;
    tr.status = lz_status[lt] ? lz_status[lt] : (g.status ? g.status : (rg.status ? rg.status : bg.status));
    tr.colour_mode = 128;
    tr.chan_size[0] = g.size;
    tr.chan_size[1] = rg.size;
    tr.chan_size[2] = bg.size;
    if (per8 == 3u) {
        const hoh_stream_result r = res8[lt * 3u + 1u], b = res8[lt * 3u + 2u];
        if (!tr.status) tr.status = r.status ? r.status : b.status;
        // :289, :309: plain RGB replaces sub-green when its three channels are smaller (LZ bytes on both sides)
        if ((uint64_t)r.size + g.size + b.size < (uint64_t)g.size + rg.size + bg.size) {
            tr.colour_mode = 2;
            tr.chan_size[1] = r.size;
            tr.chan_size[2] = b.size;
        }
    }
    tr.lz_size = lz_size[lt];
    const uint32_t c = info[lt] & 0x7fffffffu;
    tr.flags = ((info[lt] >> 31) ? kTileGrey : 0u) | (c <= 256u ? kTilePalette : 0u);
    tr.size = 3u + tr.lz_size + 1u + hohfmt::varint_len(tr.chan_size[0]) + hohfmt::varint_len(tr.chan_size[1]) + tr.chan_size[0] +
              tr.chan_size[1] + tr.chan_size[2];
    tr.start = 0;
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sel, lt, image, in_image, x0, y0, tw, th);
    tiles[(first_image + image) * sel.g.tiles_per_image + in_image] = tr;
}

// off[first + i + 1] = off[first] + sizes of tiles first .. first + i.  One CTA of 1024 threads.
__global__ void __launch_bounds__(1024) k_tile_scan(hoh_tile_result* __restrict__ tiles, uint64_t first, uint32_t n,
                                                    uint64_t* __restrict__ off) {
    __shared__ uint64_t warp_tot[32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = off[first];
    __syncthreads();
    const uint32_t lane = lane_id(), w = threadIdx.x >> 5;
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint64_t v = i < n ? tiles[first + i].size : 0ull;
        uint64_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t o = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += o;
        }
        if (lane == 31) warp_tot[w] = incl;
        __syncthreads();
        if (w == 0) {
            uint64_t t = warp_tot[lane];
            uint64_t ti = t;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint64_t o = __shfl_up_sync(0xffffffffu, ti, d);
                if ((int)lane >= d) ti += o;
            }
            warp_tot[lane] = ti - t;
        }
        __syncthreads();
        const uint64_t c = carry;
        if (i < n) {
            tiles[first + i].start = c + warp_tot[w] + incl - v;
            off[first + i + 1] = c + warp_tot[w] + incl;
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + warp_tot[w] + incl;
        __syncthreads();
    }
}

__device__ __forceinline__ void cta_copy(uint8_t* dst, const uint8_t* src, uint32_t n) {
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

// choh.cpp:112-116, 328-363: 00 00 | colour mode | LZ record | 0x24 | varint(size 1) varint(size 2) | channels.
__global__ void __launch_bounds__(256) k_tile_emit(TileSel sel, uint64_t first_image, uint32_t per8,
                                                   const hoh_stream_result* __restrict__ res8,
                                                   const hoh_stream_result* __restrict__ res9,
                                                   const uint8_t* __restrict__ out8, const uint8_t* __restrict__ out9,
                                                   const uint8_t* __restrict__ lz, uint32_t lz_stride,
                                                   hoh_tile_result* __restrict__ tiles, uint8_t* __restrict__ packed,
                                                   uint64_t packed_cap) {
    const uint64_t lt = blockIdx.x;
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sel, lt, image, in_image, x0, y0, tw, th);
    hoh_tile_result& tr = tiles[(first_image + image) * sel.g.tiles_per_image + in_image];
    if (tr.start + tr.size > packed_cap) {
        if (threadIdx.x == 0 && !tr.status) tr.status = HOH_S_OVERFLOW;
        return;
    }
    uint8_t* dst = packed + tr.start;
    const uint32_t v0 = hohfmt::varint_len(tr.chan_size[0]), v1 = hohfmt::varint_len(tr.chan_size[1]);
    if (threadIdx.x == 0) {
        dst[0] = 0;
        dst[1] = 0;
        dst[2] = (uint8_t)tr.colour_mode;
        uint8_t* q = dst + 3u + tr.lz_size;
        q[0] = 0x24;
        hohfmt::put_varint(q, 1u, tr.chan_size[0]);
        hohfmt::put_varint(q, 1u + v0, tr.chan_size[1]);
    }
    cta_copy(dst + 3, lz + lt * (uint64_t)lz_stride, tr.lz_size);
    uint8_t* body = dst + 3u + tr.lz_size + 1u + v0 + v1;
    const bool plain = tr.colour_mode == 2u;
    const hoh_stream_result c0 = res8[lt * per8];
    const hoh_stream_result c1 = plain ? res8[lt * 3u + 1u] : res9[lt * 2u];
    const hoh_stream_result c2 = plain ? res8[lt * 3u + 2u] : res9[lt * 2u + 1u];
    cta_copy(body, out8 + c0.start, c0.size);
    cta_copy(body + c0.size, (plain ? out8 : out9) + c1.start, c1.size);
    cta_copy(body + c0.size + c1.size, (plain ? out8 : out9) + c2.start, c2.size);
}

// =================================================================================================
// Tile decoder, any cruncher mode — the inverse of encode_tile as a WORKING decoder has to do it
// (dhoh.cpp:22-141, un_lz.hpp:66-180, layer_decode.hpp:127-277 with SURVEY defects D2, D3, D4, D8, D9, D10,
// D12 corrected; none of the corrections touches hot-path arithmetic).  A tile's bytes are parsed in
// phases, because every entropy stream's end is only known once its header has been read:
//   begin -> LZ side stream 0 .. 3 (one batched decode each) -> channels (order byte, size varints, layer
//   headers) -> predictor-index streams -> residual streams -> LZ expansion -> un-prediction -> colour.
// =================================================================================================
struct DTile {
    uint64_t cursor;      // next unread byte of the tile
    uint64_t end;         // one past the tile's last byte
    uint32_t colour_mode; // 128 or 2
    int32_t status;
    uint32_t lz_n[4];     // symbols in each LZ side stream
    uint32_t lz_streams;  // 3 or 4
    uint32_t uncovered;   // pixels no LZ match covers = residuals per channel
};

struct DPlane {
    uint64_t main_off;    // where the residual stream's header starts (set after the index stream is decoded)
    uint64_t chan_end;    // one past the channel's last byte: the residual stream must end exactly there
    uint32_t kind;        // 0: single predictor 0x0010 = pure MED (fastpath inverse); 1: predictor grid
    uint32_t depth;       // 8 or 9
    uint32_t n_masks;
    int32_t status;
    uint16_t masks[16];
};

// tile header: 00 00 | colour mode | LZ tag.  Local tile t's bytes are [off, end); status != 0 makes it a tile that
// decodes nothing (every later phase skips a tile or plane whose status is set).
__device__ __forceinline__ void dt_begin_tile(uint64_t t, uint64_t off, uint64_t end, int32_t status, ByteView b,
                                              uint32_t side_stride, DTile* __restrict__ tiles,
                                              hoh_dec_stream* __restrict__ streams) {
    const uint64_t packed_bytes = b.size;
    DTile d;
    d.end = end;
    d.status = status;
    d.colour_mode = b[off + 2];
    // 1x1 sub-tiles (choh.cpp:112-116), a colour mode this library emits, the LZ tag find_lz_rgb writes (lz.hpp:100)
    if (b[off] != 0 || b[off + 1] != 0 || (d.colour_mode != 128u && d.colour_mode != 2u) || b[off + 3] != 0x03 ||
        d.end > packed_bytes || d.end < off + 4u)
        d.status = HOH_S_BAD_LAYER;
    d.cursor = off + 4u;
    for (int k = 0; k < 4; k++) d.lz_n[k] = 0;
    d.lz_streams = 3;
    d.uncovered = 0;
    tiles[t] = d;
    hoh_dec_stream st;
    st.in_off = d.cursor;
    st.sym_off = (t * 4u) * side_stride;
    st.sym_cap = d.status ? 0u : side_stride;
    st.flags = HOH_FIX_DECODER;
    streams[t] = st;
}

__global__ void k_dt_begin(uint64_t n_tiles, TileSel sel, uint64_t first_image, const uint8_t* __restrict__ packed,
                           uint64_t packed_bytes, const uint64_t* __restrict__ tile_off, uint32_t side_stride,
                           DTile* __restrict__ tiles, hoh_dec_stream* __restrict__ streams) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sel, t, image, in_image, x0, y0, tw, th);
    const uint64_t gt = (first_image + image) * sel.g.tiles_per_image + in_image;  // the tile's index in the batch
    dt_begin_tile(t, tile_off[gt], tile_off[gt + 1], HOH_S_OK, ByteView{packed, packed_bytes}, side_stride, tiles,
                  streams);
}

// after LZ side stream k: advance, describe stream k + 1.  The fourth stream exists only for seek windows wider
// than 2^8 (lz.hpp:132) and nothing in the bytes says so (D3): it is there iff the next byte starts an entropy
// stream of range 256 (0x81 0x7f), which the channel-order byte that follows otherwise (0x24) never is.
__global__ void k_dt_lz_next(uint64_t n_tiles, uint32_t k, const uint8_t* __restrict__ packed, uint64_t packed_bytes,
                             const hoh_dec_result* __restrict__ res, uint32_t side_stride, DTile* __restrict__ tiles,
                             hoh_dec_stream* __restrict__ streams) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    DTile& d = tiles[t];
    const ByteView b{packed, packed_bytes};
    const bool ran = d.status == HOH_S_OK && (k < 3u || d.lz_streams == 4u);
    if (ran) {
        const hoh_dec_result r = res[t];
        if (r.status) d.status = r.status;
        else if (r.end_off > d.end || r.range != 256u) d.status = HOH_S_BAD_LAYER;
        else {
            d.cursor = r.end_off;
            d.lz_n[k] = r.n;
        }
    }
    if (k == 2u && d.status == HOH_S_OK && b[d.cursor] == 0x81 && b[d.cursor + 1] == 0x7f) d.lz_streams = 4;
    if (k >= 3u) return;
    const bool next = d.status == HOH_S_OK && (k + 1u < 3u || d.lz_streams == 4u);
    hoh_dec_stream st;
    st.in_off = d.cursor;
    st.sym_off = (t * 4u + k + 1u) * side_stride;
    st.sym_cap = next ? side_stride : 0u;
    st.flags = HOH_FIX_DECODER;
    streams[t] = st;
}

// channel-order byte, two size varints, and the layer header of each of the three channels
// (layer_decode.hpp:136-139, 208-235).  One thread per tile.  idx_streams: 3 per tile (inactive: capacity 0).
__global__ void k_dt_channels(uint64_t n_tiles, const uint8_t* __restrict__ packed, uint64_t packed_bytes, uint32_t xt,
                              uint32_t yt, uint32_t cells_pad, DTile* __restrict__ tiles, DPlane* __restrict__ planes,
                              hoh_dec_stream* __restrict__ idx_streams) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    DTile& d = tiles[t];
    const ByteView b{packed, packed_bytes};
    uint64_t at = d.cursor;
    uint64_t chan[4];
    if (d.status == HOH_S_OK) {
        if (b[at] != 0x24) d.status = HOH_S_BAD_LAYER;  // three channels, never reordered (choh.cpp:352)
        at++;
        uint32_t size[2];
        for (int k = 0; k < 2; k++) {  // read_varint varint.hpp:6-27
            const uint32_t b0 = b[at++];
            uint32_t v = b0;
            if (b0 & 0x80u) {
                const uint32_t b1 = b[at++];
                v = ((b0 & 0x7fu) << 7) + b1;
                if (b1 & 0x80u) v = ((b0 & 0x7fu) << 14) + ((b1 & 0x7fu) << 7) + b[at++];
            }
            size[k] = v;
        }
        chan[0] = at;
        chan[1] = chan[0] + size[0];
        chan[2] = chan[1] + size[1];
        chan[3] = d.end;
        if (chan[2] > d.end) d.status = HOH_S_BAD_LAYER;
    }
    for (uint32_t c = 0; c < 3u; c++) {
        DPlane pl;
        pl.status = d.status;
        pl.kind = 0;
        pl.depth = (c == 0u || d.colour_mode == 2u) ? 8u : 9u;  // sub-green differences are 9-bit (choh.cpp:240, 251; D4)
        pl.n_masks = 1;
        pl.main_off = 0;
        pl.chan_end = d.status == HOH_S_OK ? chan[c + 1] : 0;
        for (int m = 0; m < 16; m++) pl.masks[m] = 0x0010;
        hoh_dec_stream st;
        st.in_off = d.cursor;
        st.sym_off = (t * 3u + c) * cells_pad;
        st.sym_cap = 0;
        st.flags = HOH_FIX_DECODER;
        if (pl.status == HOH_S_OK) {
            uint64_t q = chan[c];
            if (b[q] != 0x10) pl.status = HOH_S_BAD_LAYER;  // prediction on, no compaction (layer_encode.hpp:57)
            const uint32_t gx = (uint32_t)b[q + 1] + 1u, gy = (uint32_t)b[q + 2] + 1u;
            q += 3;
            if (gx == 1u && gy == 1u) {
                const uint32_t mask = ((uint32_t)b[q] << 8) | b[q + 1];
                q += 2;
                if (mask != 0x0010u) pl.status = HOH_S_BAD_LAYER;  // the only single predictor the encoder emits
                pl.main_off = q;
            } else {
                if (gx != xt || gy != yt) pl.status = HOH_S_BAD_LAYER;  // the grid is a function of the tile size
                pl.kind = 1;
                pl.n_masks = b[q++];
                if (pl.n_masks == 0u || pl.n_masks > 14u) pl.status = HOH_S_BAD_LAYER;
                for (uint32_t m = 0; m < pl.n_masks && m < 16u; m++, q += 2)
                    pl.masks[m] = (uint16_t)(((uint32_t)b[q] << 8) | b[q + 1]);
                if (pl.status == HOH_S_OK) {
                    st.in_off = q;
                    st.sym_cap = xt * yt;
                }
            }
            if (q > chan[c + 1]) pl.status = HOH_S_BAD_LAYER;
        }
        planes[t * 3u + c] = pl;
        idx_streams[t * 3u + c] = st;
    }
}

// residual stream descriptors (after the index streams are decoded) + the planes' predictor maps
__global__ void k_dt_main(uint64_t n_planes, uint32_t cells, uint32_t cells_pad, uint32_t plane_stride, uint32_t npx,
                          const hoh_dec_result* __restrict__ idx_res, const uint16_t* __restrict__ idx_syms,
                          DPlane* __restrict__ planes, uint16_t* __restrict__ maps,
                          hoh_dec_stream* __restrict__ streams) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    DPlane& pl = planes[p];
    if (pl.status == HOH_S_OK && pl.kind == 1u) {
        const hoh_dec_result r = idx_res[p];
        if (r.status) pl.status = r.status;
        else if (r.n != cells || r.range != pl.n_masks) pl.status = HOH_S_BAD_LAYER;
        else {
            pl.main_off = r.end_off;
            for (uint32_t c = 0; c < cells; c++) {
                const uint32_t i = idx_syms[p * cells_pad + c];
                maps[p * cells + c] = pl.masks[i < pl.n_masks ? i : 0u];  // layer_decode.hpp:231-233
            }
        }
    }
    hoh_dec_stream st;
    st.in_off = pl.main_off;
    st.sym_off = p * (uint64_t)plane_stride;
    st.sym_cap = pl.status == HOH_S_OK ? npx : 0u;
    st.flags = HOH_FIX_DECODER;
    streams[p] = st;
}

// un_lz.hpp:150-170 as it has to work: runs of 255 accumulate, the entry after them completes the count of
// uncovered pixels, then one match of length + 4 at the recorded distance; what follows the last match is
// uncovered (D12).  One warp per tile: the walk is warp-uniform, the fills are cooperative.
__global__ void __launch_bounds__(128) k_dt_unlz(uint64_t n_tiles, uint32_t npx, uint32_t plane_stride,
                                                 const uint16_t* __restrict__ side, uint32_t side_stride,
                                                 DTile* __restrict__ tiles, uint16_t* __restrict__ backref) {
    const uint32_t lane = lane_id();
    const uint64_t t = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    if (t >= n_tiles) return;
    DTile& d = tiles[t];
    uint16_t* B = backref + t * plane_stride;
    for (uint32_t i = lane; i < npx; i += 32) B[i] = 0;
    __syncwarp();
    if (d.status != HOH_S_OK) return;
    const uint16_t* s0 = side + (t * 4u) * side_stride;
    const uint16_t* s1 = s0 + side_stride;
    const uint16_t* s2 = s1 + side_stride;
    const uint16_t* s3 = s2 + side_stride;
    const bool wide = d.lz_streams == 4u;
    uint32_t pos = 0, group = 0, covered = 0, i = 0;
    int32_t st = HOH_S_OK;
    const uint32_t n0 = d.lz_n[0];
    if (d.lz_n[1] != d.lz_n[2] || (wide && d.lz_n[3] != d.lz_n[1])) st = HOH_S_BAD_LAYER;
    while (st == HOH_S_OK && i < n0) {
        uint32_t count = 0;
        while (i < n0 && s0[i] == 255u) {
            count += 255u;
            i++;
        }
        if (i >= n0) break;
        count += s0[i++];
        pos += count;
        if (group >= d.lz_n[1]) {
            st = HOH_S_BAD_LAYER;
            break;
        }
        const uint32_t len = (uint32_t)s1[group] + 4u;
        const uint32_t back = (wide ? ((uint32_t)s3[group] << 8) : 0u) + s2[group];
        group++;
        if (pos + len > npx || back == 0u || back > pos) {
            st = HOH_S_BAD_LAYER;
            break;
        }
        for (uint32_t k = lane; k < len; k += 32) B[pos + k] = (uint16_t)back;
        pos += len;
        covered += len;
    }
    if (lane == 0) {
        if (st) d.status = st;
        d.uncovered = npx - covered;
    }
}

// Un-prediction of every plane (one thread per plane, raster order, LZ copies interleaved as in
// unprediction.hpp:63-65): kind 0 = exact inverse of channelpredict_fastpath (D10), kind 1 = unpredict_all.
__global__ void __launch_bounds__(64) k_dt_unpredict(uint64_t n_planes, int w, int h, int x_tiles, int y_tiles,
                                                     uint32_t plane_stride, const DPlane* __restrict__ planes,
                                                     const DTile* __restrict__ tiles,
                                                     const hoh_dec_result* __restrict__ main_res,
                                                     const uint16_t* __restrict__ resid,
                                                     const uint16_t* __restrict__ maps,
                                                     const uint16_t* __restrict__ backref, uint16_t* __restrict__ out,
                                                     uint16_t* __restrict__ top_s, uint8_t* __restrict__ bp_s,
                                                     int32_t* __restrict__ plane_status, uint32_t only_kind0) {
    const uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (p >= n_planes) return;
    const DPlane pl = planes[p];
    const DTile& dt = tiles[p / 3u];
    int32_t st = pl.status ? pl.status : dt.status;
    if (!st) st = main_res[p].status;
    if (!st && (main_res[p].n != dt.uncovered || main_res[p].range != (1u << pl.depth) ||
                main_res[p].end_off != pl.chan_end))  // channels follow one another without gaps (choh.cpp:355-363)
        st = HOH_S_BAD_LAYER;
    if (only_kind0 && pl.kind != 0u) return;  // predictor-grid planes are walked by k_dt_unpredict16
    plane_status[p] = st;
    if (st) return;
    const int c = 1 << pl.depth, half = c >> 1;
    const uint16_t* src = resid + p * (uint64_t)plane_stride;
    const uint16_t* br = backref + (p / 3u) * (uint64_t)plane_stride;
    uint16_t* dst = out + p * (uint64_t)plane_stride;
    uint64_t next_resid = 0;
    const bool grouped = (w & 7) == 0 && w >= 16 && (plane_stride & 7u) == 0u;  // the 8-pixel group walks below
    if (pl.kind == 0u && grouped) {
        // pure MED inverse, inputs fetched one 8-pixel group ahead (see the predictor-grid walk below)
        const uint32_t hh = (uint32_t)half * 0x00010001u;
        uint4 c_br, c_top, c_src, n_br, n_top, n_src;
        auto fetch0 = [&](uint4& Gbr, uint4& Gtop, uint4& Gsrc, int y, int x0, uint64_t nr) {
            const uint64_t at = (uint64_t)y * w + x0;
            Gbr = __ldg(reinterpret_cast<const uint4*>(br + at));
            Gtop = y ? *reinterpret_cast<const uint4*>(dst + at - w) : make_uint4(hh, hh, hh, hh);
            if ((nr & 7u) == 0u && nr + 8u <= plane_stride) {
                Gsrc = __ldg(reinterpret_cast<const uint4*>(src + nr));
            } else {
                uint32_t r[8];
#pragma unroll
                for (int k = 0; k < 8; k++) r[k] = nr + k < plane_stride ? (uint32_t)__ldg(src + nr + k) : 0u;
                Gsrc = make_uint4(r[0] | (r[1] << 16), r[2] | (r[3] << 16), r[4] | (r[5] << 16), r[6] | (r[7] << 16));
            }
        };
        auto uncovered0 = [](const uint4& b) {
            auto z = [](uint32_t wd) { return (uint32_t)((wd & 0xffffu) == 0u) + (uint32_t)((wd >> 16) == 0u); };
            return z(b.x) + z(b.y) + z(b.z) + z(b.w);
        };
        fetch0(c_br, c_top, c_src, 0, 0, 0);
        n_br = c_br, n_top = c_top, n_src = c_src;
        for (int y = 0; y < h; y++) {
            int L = half, TL = half;
            for (int x0 = 0; x0 < w; x0 += 8) {
                const bool row_goes_on = x0 + 8 < w;
                if (row_goes_on || y + 1 < h)
                    fetch0(n_br, n_top, n_src, row_goes_on ? y : y + 1, row_goes_on ? x0 + 8 : 0,
                           next_resid + uncovered0(c_br));
                const uint32_t brw[4] = {c_br.x, c_br.y, c_br.z, c_br.w};
                const uint32_t tpw[4] = {c_top.x, c_top.y, c_top.z, c_top.w};
                uint32_t q0 = c_src.x, q1 = c_src.y, q2 = c_src.z, q3 = c_src.w;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const uint64_t at = (uint64_t)y * w + x0 + k;
                    const uint32_t back = (k & 1) ? (brw[k >> 1] >> 16) : (brw[k >> 1] & 0xffffu);
                    const int T = (int)((k & 1) ? (tpw[k >> 1] >> 16) : (tpw[k >> 1] & 0xffffu));
                    int v;
                    if (back) {
                        v = dst[at - back];
                    } else {
                        v = ((int)(q0 & 0xffffu) + p_med_grad(T, L, TL) - half) & (c - 1);
                        q0 = __funnelshift_r(q0, q1, 16);
                        q1 = __funnelshift_r(q1, q2, 16);
                        q2 = __funnelshift_r(q2, q3, 16);
                        q3 >>= 16;
                        next_resid++;
                    }
                    dst[at] = (uint16_t)v;
                    L = v;
                    TL = T;
                }
                c_br = n_br, c_top = n_top, c_src = n_src;
            }
        }
        return;
    }
    if (pl.kind == 0u) {
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) {
                const uint64_t at = (uint64_t)y * w + x;
                if (br[at]) {
                    dst[at] = dst[at - br[at]];
                    continue;
                }
                const int L = x ? dst[at - 1] : half;
                const int T = y ? dst[at - w] : half;
                const int TL = (x && y) ? dst[at - w - 1] : half;
                dst[at] = (uint16_t)(((int)src[next_resid++] + p_med_grad(T, L, TL) - half) & (c - 1));
            }
        return;
    }
    const int tw = (w + x_tiles - 1) / x_tiles, th = (h + y_tiles - 1) / y_tiles;
    const uint16_t* tmap = maps + p * (uint64_t)x_tiles * y_tiles;
    uint16_t* top = top_s + p * (uint64_t)w;
    uint8_t* bp = bp_s + p * (uint64_t)w;
    if (grouped) {
        // The same walk with every global-memory access taken off the pixel chain (the scalar walk below spends
        // 80 % of its time waiting on loads: ncu, long scoreboard).  Pixels go in groups of 8 whose inputs — the
        // back-reference map, the row above (which is simply the previous row of `dst`: no `top` array), the best
        // predictors of the row above and the next 8 residuals — are fetched as 16-byte words ONE GROUP AHEAD into
        // registers; where the residuals of the next group start only depends on this group's back-references.
        // The residuals sit in a 128-bit shift register, the new best predictors are stored as one 8-byte word.
        struct Grp {
            uint4 br, top, src;
            uint2 bp;
        };
        const uint32_t hh = (uint32_t)half * 0x00010001u;
        auto fetch = [&](Grp& G, int y, int x0, uint64_t nr) {
            const uint64_t at = (uint64_t)y * w + x0;
            G.br = __ldg(reinterpret_cast<const uint4*>(br + at));
            if (y) {
                G.top = *reinterpret_cast<const uint4*>(dst + at - w);
                G.bp = *reinterpret_cast<const uint2*>(bp + x0);
            } else {
                G.top = make_uint4(hh, hh, hh, hh);
                G.bp = make_uint2(0x04040404u, 0x04040404u);
            }
            if ((nr & 7u) == 0u && nr + 8u <= plane_stride) {
                G.src = __ldg(reinterpret_cast<const uint4*>(src + nr));
            } else {  // planes with LZ matches: the residuals of a group start anywhere
                uint32_t r[8];
#pragma unroll
                for (int k = 0; k < 8; k++) r[k] = nr + k < plane_stride ? (uint32_t)__ldg(src + nr + k) : 0u;
                G.src = make_uint4(r[0] | (r[1] << 16), r[2] | (r[3] << 16), r[4] | (r[5] << 16), r[6] | (r[7] << 16));
            }
        };
        auto uncovered = [](const uint4& b) {  // how many of the 8 pixels take a residual
            auto z = [](uint32_t wd) { return (uint32_t)((wd & 0xffffu) == 0u) + (uint32_t)((wd >> 16) == 0u); };
            return z(b.x) + z(b.y) + z(b.z) + z(b.w);
        };
        Grp cur, nxt;
        fetch(cur, 0, 0, 0);
        nxt = cur;
        int bp_row_end = 4;  // best predictor of the previous row's last pixel (bp[w - 1])
        for (int y = 0; y < h; y++) {
            int left = half, left_top = half;
            int bp_left = bp_row_end;
            const bool last_row = y + 1 >= h;
            const uint16_t* mrow = tmap + (size_t)((y + 1) / th) * x_tiles;
            uint32_t next_mask = last_row ? 0u : mrow[0];
            int cell_i = 0;
            int first_of_row = 0;
            MaskBias mb;
            int in_cell = tw;
            for (int x0 = 0; x0 < w; x0 += 8) {
                const bool row_goes_on = x0 + 8 < w;
                if (row_goes_on || !last_row)
                    fetch(nxt, row_goes_on ? y : y + 1, row_goes_on ? x0 + 8 : 0, next_resid + uncovered(cur.br));
                const uint32_t brw[4] = {cur.br.x, cur.br.y, cur.br.z, cur.br.w};
                const uint32_t tpw[4] = {cur.top.x, cur.top.y, cur.top.z, cur.top.w};
                const uint32_t bpw[2] = {cur.bp.x, cur.bp.y};
                uint32_t q0 = cur.src.x, q1 = cur.src.y, q2 = cur.src.z, q3 = cur.src.w;  // residual queue, next one lowest
                uint32_t nbw[2] = {0u, 0u};
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int x = x0 + k;
                    if (in_cell == tw) {
                        in_cell = 0;
                        mask_bias(next_mask, mb);
                        cell_i++;
                        next_mask = (last_row || cell_i >= x_tiles) ? 0u : mrow[cell_i];
                    }
                    in_cell++;
                    const uint64_t at = (uint64_t)y * w + x;
                    const uint32_t back = (k & 1) ? (brw[k >> 1] >> 16) : (brw[k >> 1] & 0xffffu);
                    const int t = (int)((k & 1) ? (tpw[k >> 1] >> 16) : (tpw[k >> 1] & 0xffffu));
                    int tr;
                    if (k < 7)
                        tr = (int)(((k + 1) & 1) ? (tpw[(k + 1) >> 1] >> 16) : (tpw[(k + 1) >> 1] & 0xffffu));
                    else
                        tr = row_goes_on ? (int)(nxt.top.x & 0xffffu) : first_of_row;
                    const int bpx = (int)((bpw[k >> 2] >> (8 * (k & 3))) & 0xffu);
                    Cand kk;
                    candidates(left, t, left_top, tr, false, kk);
                    const int pred = p_mid(cand_at_tree(kk, bpx), cand_at_tree(kk, bp_left));
                    int v;
                    if (back) {
                        v = dst[at - back];  // unprediction.hpp:63-65
                    } else {
                        const uint32_t tval = (uint32_t)((int)(q0 & 0xffffu) - c - half + pred) & 0xffffu;  // :67
                        v = (int)(tval & (uint32_t)(c - 1));
                        q0 = __funnelshift_r(q0, q1, 16);
                        q1 = __funnelshift_r(q1, q2, 16);
                        q2 = __funnelshift_r(q2, q3, 16);
                        q3 >>= 16;
                        next_resid++;
                    }
                    dst[at] = (uint16_t)v;
                    if (x == 0) first_of_row = v;
                    left_top = t;
                    left = v;
                    const int nb = last_row ? 0 : pick_best_biased_tree(v, kk, mb, c);
                    nbw[k >> 2] |= (uint32_t)nb << (8 * (k & 3));
                    bp_left = nb;
                }
                *reinterpret_cast<uint2*>(bp + x0) = make_uint2(nbw[0], nbw[1]);
                cur = nxt;
            }
            bp_row_end = bp_left;
        }
        return;
    }
    for (int i = 0; i < w; i++) {
        top[i] = (uint16_t)half;
        bp[i] = 4;
    }
    for (int y = 0; y < h; y++) {  // same walk as k_raster_walk<true>
        int left = half, left_top = half;
        int bp_left = bp[w - 1];
        const bool last_row = y + 1 >= h;
        const uint16_t* mrow = tmap + (size_t)((y + 1) / th) * x_tiles;
        int first_of_row = 0;
        MaskBias mb;
        int in_cell = tw;
        for (int x = 0; x < w; x++) {
            if (in_cell == tw) {
                in_cell = 0;
                mask_bias(last_row ? 0u : *mrow++, mb);
            }
            in_cell++;
            const uint64_t at = (uint64_t)y * w + x;
            const int tr = (x + 1 < w) ? top[x + 1] : (w > 1 ? first_of_row : top[0]);
            const int t = top[x];
            Cand k;
            candidates(left, t, left_top, tr, false, k);
            const int pred = p_mid(cand_at(k, bp[x]), cand_at(k, bp_left));
            int v;
            if (br[at]) {
                v = dst[at - br[at]];  // unprediction.hpp:63-65
            } else {
                const uint32_t tval = (uint32_t)((int)src[next_resid++] - c - half + pred) & 0xffffu;  // :67
                v = (int)(tval & (uint32_t)(c - 1));  // % c, c a power of two
            }
            dst[at] = (uint16_t)v;
            if (x == 0) first_of_row = v;
            left_top = t;
            top[x] = (uint16_t)v;
            left = v;
            const int nb = last_row ? 0 : pick_best_biased(v, k, mb, c);
            bp[x] = (uint8_t)nb;
            bp_left = nb;
        }
    }
}

// The same un-prediction with the 16 candidate predictors of a pixel spread over 16 lanes: a half-warp per plane.
// The walk stays serial per plane (H4), but what one thread did in ~200 dependent instructions per pixel — 16
// candidates, 16 errors, a 16-way masked argmin, two 16-way selects — becomes one candidate and one error per
// lane, two shuffles for the prediction and a 4-step shuffle minimum for the best predictor.  The row above
// and its best predictors live in shared memory (w * 3 bytes per plane); lane 0 of the half-warp owns all
// stores.  Planes under the single-predictor header (kind 0) are walked by lane 0 alone.
constexpr int kUp16Planes = 8;  // planes (half-warps) per CTA

__global__ void __launch_bounds__(kUp16Planes * 16) k_dt_unpredict16(
    uint64_t n_planes, int w, int h, int x_tiles, int y_tiles, uint32_t plane_stride, const DPlane* __restrict__ planes,
    const DTile* __restrict__ tiles, const hoh_dec_result* __restrict__ main_res, const uint16_t* __restrict__ resid,
    const uint16_t* __restrict__ maps, const uint16_t* __restrict__ backref, uint16_t* __restrict__ out,
    int32_t* __restrict__ plane_status) {
    extern __shared__ __align__(16) uint8_t up_smem[];
    const uint32_t hw = threadIdx.x >> 4, j = threadIdx.x & 15u;
    const int w_pad = (w + 1) & ~1;
    uint16_t* top = reinterpret_cast<uint16_t*>(up_smem + (size_t)hw * w_pad * 3);
    uint8_t* bp = up_smem + (size_t)hw * w_pad * 3 + (size_t)w_pad * 2;
    const uint64_t p = (uint64_t)blockIdx.x * kUp16Planes + hw;
    // The two half-warps of a warp walk their planes in lockstep (same w, h: same trip counts) so that every
    // shuffle is one full-warp instruction; a half without a plane to decode runs along and stores nothing.
    bool alive = p < n_planes;
    DPlane pl;
    pl.kind = 0;
    pl.depth = 8;
    if (alive) {
        pl = planes[p];
        const DTile& dt = tiles[p / 3u];
        int32_t st = pl.status ? pl.status : dt.status;
        if (!st) st = main_res[p].status;
        if (!st && (main_res[p].n != dt.uncovered || main_res[p].range != (1u << pl.depth) ||
                    main_res[p].end_off != pl.chan_end))  // channels follow one another without gaps (choh.cpp:355-363)
            st = HOH_S_BAD_LAYER;
        if (pl.kind == 1u && j == 0) plane_status[p] = st;  // kind 0 planes belong to k_dt_unpredict
        alive = st == 0 && pl.kind == 1u;
    }
    if (__ballot_sync(0xffffffffu, alive) == 0u) return;
    const uint64_t q = alive ? p : 0;  // a plane index that is safe to read from
    const int c = 1 << pl.depth, half = c >> 1;
    const uint16_t* src = resid + q * (uint64_t)plane_stride;
    const uint16_t* br = backref + (q / 3u) * (uint64_t)plane_stride;
    uint16_t* dst = out + q * (uint64_t)plane_stride;
    // my candidate (prediction.hpp:190-207) = type(A, B, C) with the operands picked from (L, T, TL, TR) = 0..3:
    //   j        0  1  2  3 | 4            | 5       6        7        8        | 9               | 10 .. 15
    //   type     the operand | med-grad     | midpoint                            | paeth           | average of three
    //   A B C    L  T TL TR  | T L TL       | L,T     L,TL     TL,T     T,TR     | L TL T          | L L TL / L TL TL / TL TL T / TL T T / T T TR / T TR TR
    // The four neighbours are 16-bit values packed in two registers (L | T << 16, TL | TR << 16); an operand is one
    // byte-permute with a per-lane selector (0x4410 + 0x22 * code puts halfword `code` in the low half) and a mask.
    const uint32_t type = j < 4u ? 0u : (j == 4u ? 3u : (j < 9u ? 1u : (j == 9u ? 4u : 2u)));
    const uint32_t sel_a = 0x4410u + 0x22u * ((0x5a0181e4u >> (2u * j)) & 3u);
    const uint32_t sel_b = 0x4410u + 0x22u * ((0xd68b6400u >> (2u * j)) & 3u);
    const uint32_t sel_c = 0x4410u + 0x22u * ((0xf5a40200u >> (2u * j)) & 3u);
    const bool is_id = type == 0u, is_mid = type == 1u, is_med = type == 3u, is_paeth = type == 4u;
    const int tw = (w + x_tiles - 1) / x_tiles, th = (h + y_tiles - 1) / y_tiles;
    const uint16_t* tmap = maps + q * (uint64_t)x_tiles * y_tiles;
    for (int i = (int)j; i < w; i += 16) {
        top[i] = (uint16_t)half;
        bp[i] = 4;
    }
    __syncwarp();
    const bool writer = alive && j == 0u;
    const int bias = -c - half;
    const uint32_t cmask = (uint32_t)(c - 1);
    const int err_cap = 2 * c;
    const uint16_t* br_p = br;
    uint16_t* dst_p = dst;
    const uint16_t* src_p = src;
    const uint16_t* src_end = src + (size_t)w * h;
    for (int y = 0; y < h; y++) {  // the walk of k_raster_walk<true>
        int left = half, left_top = half;
        int bp_left = bp[w - 1];
        const bool last_row = y + 1 >= h;
        const uint16_t* mrow = tmap + (size_t)((y + 1) / th) * x_tiles;
        int first_of_row = 0;
        int t = top[0];
        int in_cell = tw;
        uint32_t mask = 0, my_bit = 0;
        for (int x = 0; x < w; x++) {
            if (in_cell == tw) {  // next grid cell of the row below: its mask picks this pixel's best predictor
                in_cell = 0;
                mask = (last_row || !alive) ? 0u : *mrow++;
                my_bit = (mask >> j) & 1u;
            }
            in_cell++;
            const bool last_col = x + 1 >= w;
            const int t_next = last_col ? 0 : top[x + 1];
            const int tr = last_col ? (w > 1 ? first_of_row : t) : t_next;
            const int bp_top = bp[x];
            const uint32_t brv = alive ? *br_p : 0u;
            br_p++;
            const int rv = (alive && src_p < src_end) ? (int)*src_p : 0;
            src_p += brv ? 0 : 1;
            const uint32_t lo = (uint32_t)left | ((uint32_t)t << 16), hi2 = (uint32_t)left_top | ((uint32_t)tr << 16);
            const int A = (int)(__byte_perm(lo, hi2, sel_a) & 0xffffu), B = (int)(__byte_perm(lo, hi2, sel_b) & 0xffffu),
                      C = (int)(__byte_perm(lo, hi2, sel_c) & 0xffffu);
            const int mid = p_mid(A, B), avg = p_avg3(A, B, C), med = p_med_grad(A, B, C), pae = p_paeth(A, B, C);
            int cand = is_id ? A : (is_mid ? mid : avg);
            cand = is_med ? med : cand;
            cand = is_paeth ? pae : cand;
            const int pa = __shfl_sync(0xffffffffu, cand, bp_top, 16), pb = __shfl_sync(0xffffffffu, cand, bp_left, 16);
            // unprediction.hpp:63-65: an LZ-covered pixel is a copy; lane 0 wrote every earlier pixel of this plane
            int copy = 0;
            if (writer && brv) copy = (int)*(dst_p - brv);
            copy = __shfl_sync(0xffffffffu, copy, 0, 16);
            const uint32_t tval = (uint32_t)(rv + bias + p_mid(pa, pb)) & 0xffffu;  // :67
            const int v = brv ? copy : (int)(tval & cmask);
            // best predictor for the pixels below / to the right: lowest index among the smallest errors < 2c
            const int err = abs(v - cand);
            uint32_t key = (err < err_cap && my_bit) ? ((uint32_t)err << 4) | j : 0x7fffffffu;
#pragma unroll
            for (int d = 8; d > 0; d >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, d, 16));
            const int nb = key == 0x7fffffffu ? 0 : (int)(key & 15u);  // (mask is 0 on the last row: nb = 0)
            if (writer) *dst_p = (uint16_t)v;
            dst_p++;
            if (j == 0u) {
                top[x] = (uint16_t)v;
                bp[x] = (uint8_t)nb;
            }
            first_of_row = x == 0 ? v : first_of_row;
            left_top = t;
            left = v;
            bp_left = nb;
            t = t_next;
        }
        __syncwarp();  // lane 0's row of top / bp becomes visible to its half-warp
    }
}

// planes -> interleaved RGB in the image (inverse of channel.hpp:73-79 for colour mode 128, D4), tile status
__global__ void __launch_bounds__(256) k_dt_store(TileSel sel, uint64_t first_image, uint32_t plane_stride,
                                                  const DTile* __restrict__ tiles,
                                                  const int32_t* __restrict__ plane_status,
                                                  const uint16_t* __restrict__ planes, uint8_t* __restrict__ rgb,
                                                  int32_t* __restrict__ status) {
    const uint64_t lt = blockIdx.x;
    uint64_t image;
    uint32_t in_image, x0, y0, tw, th;
    sel_tile(sel, lt, image, in_image, x0, y0, tw, th);
    const TileGeom& g = sel.g;
    int32_t st = tiles[lt].status;
    for (int c = 0; c < 3; c++) st = st ? st : plane_status[lt * 3u + c];
    if (threadIdx.x == 0) status[(first_image + image) * g.tiles_per_image + in_image] = st;
    if (st) return;
    uint8_t* img = rgb + (first_image + image) * (uint64_t)g.width * g.height * 3u;
    const uint16_t* a = planes + (lt * 3u) * (uint64_t)plane_stride;
    const uint16_t* b = a + plane_stride;
    const uint16_t* c = b + plane_stride;
    const bool sub_green = tiles[lt].colour_mode == 128u;
    for (uint32_t i = threadIdx.x; i < tw * th; i += blockDim.x) {
        const uint32_t x = i % tw, y = i / tw;
        uint8_t* o = img + ((uint64_t)(y0 + y) * g.width + x0 + x) * 3u;
        const uint32_t gr = a[i];
        o[1] = (uint8_t)gr;
        o[0] = (uint8_t)(sub_green ? (b[i] + gr - 256u) & 255u : b[i]);
        o[2] = (uint8_t)(sub_green ? (c[i] + gr - 256u) & 255u : c[i]);
    }
}

// -------------------------------------------------------------------------------------------------
// Region decode (hoh_decode_regions): the crop_w x crop_h window of every image; only the tiles a window touches go
// through the phases above.  Each image gets the same number of SLOTS per tile shape, fixed on the host from the crop
// size, so no launch size depends on the windows (no device-to-host copy).  Slot k of shape c of image i is entry
// i * per_image + first[c] + k of the slot list: the index (in its image) of the tile it decodes, or kRoiIdle (the
// window touches fewer tiles of the shape than it has slots), or kRoiBadWindow (the window does not lie inside the
// image: every slot of the image).  A pass over shape c runs cols[c] * rows[c] slots per image through
// k_dt_begin_roi, the unchanged phases and k_dt_store_window; local tile lt is slot lt % (cols * rows) of image
// lt / (cols * rows).
// -------------------------------------------------------------------------------------------------
constexpr uint32_t kRoiIdle = 0xffffffffu, kRoiBadWindow = 0xfffffffeu;

struct RoiPlan {
    TileGeom g;
    uint32_t crop_w, crop_h, n_cls;
    uint32_t per_image;                                       // slots of one image, all shapes
    uint32_t x_first[4], x_count[4], y_first[4], y_count[4];  // shape c's sub-grid of the tile grid (TileSel)
    uint32_t cols[4], rows[4], first[4];                      // shape c: cols x rows slots from slot first[c]
};

// One thread per image: checks the window and lists, per shape, the touched part of the shape's sub-grid row-major.
__global__ void k_roi_select(uint64_t n_images, uint64_t first_image, const uint32_t* __restrict__ origin, RoiPlan p,
                             uint32_t* __restrict__ slots) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n_images) return;
    const uint32_t wx = origin[2 * (first_image + i)], wy = origin[2 * (first_image + i) + 1];
    const bool inside = (uint64_t)wx + p.crop_w <= p.g.width && (uint64_t)wy + p.crop_h <= p.g.height;
    uint32_t* s = slots + i * p.per_image;
    // x lies in tile column x / tile_w (only the last column is narrower, and width <= x_tiles * tile_w)
    const uint32_t gx0 = inside ? wx / p.g.tile_w : 0u, gx1 = inside ? (wx + p.crop_w - 1u) / p.g.tile_w : 0u;
    const uint32_t gy0 = inside ? wy / p.g.tile_h : 0u, gy1 = inside ? (wy + p.crop_h - 1u) / p.g.tile_h : 0u;
    for (uint32_t c = 0; c < p.n_cls; c++) {
        const uint32_t n_slots = p.cols[c] * p.rows[c];
        const uint32_t cx0 = max(gx0, p.x_first[c]), cx1 = min(gx1, p.x_first[c] + p.x_count[c] - 1u);
        const uint32_t cy0 = max(gy0, p.y_first[c]), cy1 = min(gy1, p.y_first[c] + p.y_count[c] - 1u);
        const uint32_t nx = inside && cx1 >= cx0 ? cx1 - cx0 + 1u : 0u, ny = inside && cy1 >= cy0 ? cy1 - cy0 + 1u : 0u;
        assert(nx <= p.cols[c] && ny <= p.rows[c]);  // the bound roi_plan proves
        for (uint32_t k = 0; k < n_slots; k++)
            s[p.first[c] + k] = !inside ? kRoiBadWindow
                              : k < nx * ny ? (cy0 + k / nx) * p.g.x_tiles + cx0 + k % nx
                                            : kRoiIdle;
    }
}

// k_dt_begin for the slots of one shape (cls_slots = cols * rows of it).  An idle or bad-window slot becomes a tile
// with a status whose streams point at the zero padding at the end of the input (in range, and no tile's bytes):
// every later phase skips it as it skips a damaged tile, so the bytes of untouched tiles never decide anything.
__global__ void k_dt_begin_roi(uint64_t n_tiles, uint32_t cls_slots, uint32_t first, uint32_t per_image,
                               uint32_t tiles_per_image, uint64_t first_image, const uint8_t* __restrict__ packed,
                               uint64_t packed_bytes, const uint64_t* __restrict__ tile_off, uint32_t side_stride,
                               const uint32_t* __restrict__ slots, DTile* __restrict__ tiles,
                               hoh_dec_stream* __restrict__ streams) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const uint64_t image = t / cls_slots;
    const uint32_t e = slots[image * per_image + first + t % cls_slots];
    const ByteView b{packed, packed_bytes};
    if (e >= kRoiBadWindow) {
        dt_begin_tile(t, packed_bytes - 32u, packed_bytes - 32u, HOH_S_BAD_WINDOW, b, side_stride, tiles, streams);
        return;
    }
    const uint64_t gt = (first_image + image) * tiles_per_image + e;
    dt_begin_tile(t, tile_off[gt], tile_off[gt + 1], HOH_S_OK, b, side_stride, tiles, streams);
}

// k_dt_store for the slots of one shape: tile ∩ window goes to the image's dense crop at (x - wx, y - wy), and the
// slot's status to slot_status (idle and bad-window slots write nothing).
__global__ void __launch_bounds__(256) k_dt_store_window(uint32_t cls_slots, uint32_t first, uint64_t first_image,
                                                         RoiPlan p, uint32_t plane_stride,
                                                         const uint32_t* __restrict__ origin,
                                                         const uint32_t* __restrict__ slots,
                                                         const DTile* __restrict__ tiles,
                                                         const int32_t* __restrict__ plane_status,
                                                         const uint16_t* __restrict__ planes,
                                                         uint8_t* __restrict__ crops, int32_t* __restrict__ slot_status) {
    const uint64_t lt = blockIdx.x;
    const uint64_t image = lt / cls_slots;
    const uint64_t at = image * p.per_image + first + lt % cls_slots;
    const uint32_t e = slots[at];
    if (e >= kRoiBadWindow) return;
    int32_t st = tiles[lt].status;
    for (int c = 0; c < 3; c++) st = st ? st : plane_status[lt * 3u + c];
    if (threadIdx.x == 0) slot_status[at] = st;
    if (st) return;
    uint32_t x0, y0, tw, th;
    tile_rect(p.g, e, x0, y0, tw, th);
    const uint32_t wx = origin[2 * (first_image + image)], wy = origin[2 * (first_image + image) + 1];
    const uint32_t ix0 = max(x0, wx), ix1 = min(x0 + tw, wx + p.crop_w);
    const uint32_t iy0 = max(y0, wy), iy1 = min(y0 + th, wy + p.crop_h);
    if (ix1 <= ix0 || iy1 <= iy0) return;  // never for a touched tile
    const uint32_t nw = ix1 - ix0;
    uint8_t* crop = crops + (first_image + image) * (uint64_t)p.crop_w * p.crop_h * 3u;
    const uint16_t* a = planes + (lt * 3u) * (uint64_t)plane_stride;
    const uint16_t* b = a + plane_stride;
    const uint16_t* c = b + plane_stride;
    const bool sub_green = tiles[lt].colour_mode == 128u;
    for (uint32_t i = threadIdx.x; i < nw * (iy1 - iy0); i += blockDim.x) {
        const uint32_t x = ix0 + i % nw, y = iy0 + i / nw;
        const uint32_t q = (y - y0) * tw + (x - x0);
        uint8_t* o = crop + ((uint64_t)(y - wy) * p.crop_w + (x - wx)) * 3u;
        const uint32_t gr = a[q];
        o[1] = (uint8_t)gr;
        o[0] = (uint8_t)(sub_green ? (b[q] + gr - 256u) & 255u : b[q]);
        o[2] = (uint8_t)(sub_green ? (c[q] + gr - 256u) & 255u : c[q]);
    }
}

// One thread per image: HOH_S_BAD_WINDOW, else the status of the failing touched tile with the lowest index, else 0.
__global__ void k_roi_fold(uint64_t n_images, uint64_t first_image, RoiPlan p, const uint32_t* __restrict__ slots,
                           const int32_t* __restrict__ slot_status, int32_t* __restrict__ status) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n_images) return;
    const uint32_t* s = slots + i * p.per_image;
    const int32_t* ss = slot_status + i * p.per_image;
    int32_t st = HOH_S_OK;
    uint32_t lowest = kRoiIdle;
    if (s[0] == kRoiBadWindow) {
        st = HOH_S_BAD_WINDOW;
    } else {
        for (uint32_t k = 0; k < p.per_image; k++)
            if (s[k] != kRoiIdle && ss[k] != HOH_S_OK && s[k] < lowest) {
                lowest = s[k];
                st = ss[k];
            }
    }
    status[first_image + i] = st;
}

// -------------------------------------------------------------------------------------------------
// Fused mode-0 tile decoder: rANS decode + MED un-prediction + colour inverse + tile scatter in ONE kernel.
// -------------------------------------------------------------------------------------------------
// The rANS step of a stream is one long dependent chain that leaves half of the issue slots of an SM idle
// (k_rans_decode: 2.5 warps per scheduler, ~60 instructions per ~315-cycle step), and the un-prediction of a pixel
// is a second, independent chain: v = (r + med(T, L, T + L - TL) - c/2) mod c depends on the pixel to the left, not
// on the coder's state.  Run in the same lane they interleave, the residual planes never exist in memory (the
// unfused pair writes and re-reads 2 x 6.4 GB of u16 symbols at BASELINE config 2) and k_tile_unpredict_s0's launch
// (4.3 ms) disappears.
//
// One warp per CTA, 30 lanes = the G, R-G, B-G streams of 10 whole tiles (lanes 30, 31 idle), all tiles of the launch
// of one shape with tile_w % 8 == 0.  At step k a lane holds residual k of its plane, i.e. pixel (k / tile_w,
// k % tile_w): its left neighbour is the value it produced one step ago (a register), and the row above comes from
// the OUTPUT IMAGE itself — the RGB bytes this warp stored tile_w steps earlier, re-read through L2 (__ldcg, after
// the __syncwarp that orders the stores) 24 bytes = 8 pixels at a time, one group ahead of their use, and turned back
// into the lane's plane (G, or R - G + 256 / B - G + 256: channel.hpp:75-77).  The finished value reaches the other
// two channels of its tile by one shuffle (G), every lane puts ITS byte of the pixel into a 24-byte row of shared
// memory, and after 8 steps each lane stores 8 of its tile's 24 bytes with one aligned 8-byte store.
// Streams in stored mode (entropy_encoding.hpp:244-267) are read by the same lanes from the same word ring
// (maxbits per symbol, MSB first); a tile with a damaged stream is reported and left untouched.
constexpr int kFusedTiles = 10;                  // tiles per warp
constexpr int kFusedLanes = 3 * kFusedTiles;     // working lanes
constexpr int kFusedStage = 272;                 // bytes of output staging per warp

struct StoredYes { static constexpr bool value = true; };
struct StoredNo { static constexpr bool value = false; };

template <typename LutT>
__global__ void __launch_bounds__(32) k_rans_decode_tiles_s0(const hoh_dec_stream* __restrict__ streams,
                                                             uint32_t n_streams, const uint8_t* __restrict__ in,
                                                             uint64_t in_bytes, const uint32_t* __restrict__ cumtab,
                                                             const DecMeta* __restrict__ meta,
                                                             const hoh_dec_result* __restrict__ results, TileGeom g,
                                                             uint8_t* __restrict__ rgb, int32_t* __restrict__ status,
                                                             uint32_t rows_lo, uint32_t rows) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint32_t* tab = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* rings = tab + (size_t)rows * 32u;
    uint8_t* stage = reinterpret_cast<uint8_t*>(rings + 32 * kRingWords);  // 11 rows of 24 bytes: 10 tiles + one for the idle lanes
    LutT* lut = reinterpret_cast<LutT*>(stage + kFusedStage);

    const uint32_t lane = lane_id();
    const uint32_t ch = lane % 3u, tl = lane / 3u;  // channel (0 G, 1 R-G, 2 B-G) and tile inside the warp
    const uint32_t s = blockIdx.x * (uint32_t)kFusedLanes + lane;
    const bool exists = lane < (uint32_t)kFusedLanes && s < n_streams;
    hoh_dec_stream st;
    DecMeta m;
    st.sym_cap = 0;
    m.kind = 0;
    m.n = 0;
    m.range = 1;
    m.prob_bits = 1;
    m.maxbits = 1;
    m.payload_off = 0;
    m.status = HOH_S_OK;
    m.used = 0;
    int32_t my_status = HOH_S_OK;
    if (exists) {
        st = streams[s];
        m = meta[s];
        my_status = status[s];
        if (my_status == HOH_S_OK) my_status = results[s].status;
    }
    const uint32_t tw = g.tile_w, th = g.tile_h, npx = tw * th;
    // a stream that can fill its plane: sound header, one symbol per pixel (no LZ map here), rANS or stored
    const bool sound = exists && my_status == HOH_S_OK && (m.kind == 2u || m.kind == 1u) && m.n == npx && st.sym_cap >= npx;
    if (exists && my_status == HOH_S_OK && !sound) my_status = HOH_S_BAD_LAYER;
    const bool coded = sound && m.kind == 2u;   // takes part in the rANS chain
    const bool stored = sound && m.kind == 1u;  // reads maxbits-wide symbols
    uint32_t need = coded ? m.used + 3u : 1u;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) need = max(need, __shfl_xor_sync(0xffffffffu, need, d));
    if (need <= rows_lo || need > rows) return;  // another class's launch
    // the whole tile is decoded or none of it
    const uint32_t base_lane = lane - ch;
    // (three unconditional shuffles: with && a lane whose first answer is 0 would skip the others and fall out of step)
    const int ok0 = __shfl_sync(0xffffffffu, (int)sound, min(base_lane, 31u));
    const int ok1 = __shfl_sync(0xffffffffu, (int)sound, min(base_lane + 1u, 31u));
    const int ok2 = __shfl_sync(0xffffffffu, (int)sound, min(base_lane + 2u, 31u));
    const bool tile_ok = (ok0 & ok1 & ok2) != 0 && lane < (uint32_t)kFusedLanes;

    for (uint32_t j = 0; j < (uint32_t)kFusedLanes; j++) {
        const uint32_t sj = blockIdx.x * (uint32_t)kFusedLanes + j;
        const bool lj = __shfl_sync(0xffffffffu, (int)coded, j) != 0;
        const uint32_t uj = __shfl_sync(0xffffffffu, m.used, j);
#ifdef HOH_DEBUG_FUSED
        if (blockIdx.x == 0 && j < 3 && (lane == 0 || lane == 5)) printf("fill j %u lane %u lj %d uj %u my used %u\n", j, lane, (int)lj, uj, m.used);
#endif
        if (!lj) continue;
        const uint32_t* src = cumtab + (size_t)sj * kCumRow;
        for (uint32_t i = lane; i < uj + 3u; i += 32) tab[i * 32u + j] = src[i];
    }
    __syncwarp();
#ifdef HOH_DEBUG_FUSED
    if (blockIdx.x == 0 && lane == 0) printf("A after fill: tab[128]=%08x tab[160]=%08x rows=%u need=%u\n", tab[128], tab[160], rows, need);
#endif

    const PerLaneDense T{tab, lane};
    const PerLaneDenseS TS{(uint32_t)__cvta_generic_to_shared(tab + lane)};              // the hot loop's view of it
    const uint32_t lut_s = (uint32_t)__cvta_generic_to_shared(lut + lane);
    const uint32_t bits = coded ? m.prob_bits : 1u;
    const uint32_t mask = (1u << bits) - 1u;
    const uint32_t lut_shift = bits > 7u ? bits - 7u : 0u;
    for (uint32_t i = lane; i < (uint32_t)kFusedStage / 4u; i += 32) reinterpret_cast<uint32_t*>(stage)[i] = 0u;
    if (coded) {
        lut_build(T, lut + lane, 32u, lut_shift, m.used);
    } else {  // stored / idle / damaged lane: a one-symbol table that owns the whole range, so that its state never moves
        tab[lane] = 0u;
        tab[32u + lane] = 0u;
        tab[64u + lane] = (1u << bits) << kSymBits;
        tab[96u + lane] = 0xffffffffu;
        for (uint32_t j = 0; j < (uint32_t)kLutSize; j++) lut[j * 32u + lane] = (LutT)1;
    }
    __syncwarp();
#ifdef HOH_DEBUG_FUSED
    if (blockIdx.x == 0 && lane == 0) printf("B after lut: tab[128]=%08x tab[160]=%08x\n", tab[128], tab[160]);
#endif

    WordRing rd;
    rd.open(in, in_bytes, sound ? m.payload_off : 0ull, rings + lane * kRingWords);
#ifdef HOH_DEBUG_FUSED
    if (blockIdx.x == 0 && lane == 0) printf("C after open: tab[128]=%08x tab[160]=%08x\n", tab[128], tab[160]);
#endif
    uint64_t x = kRansL;
    if (coded) {  // rans64.hpp:107-116
        const uint32_t lo = rd.next;
        rd.take_if(true);
        const uint32_t hi = rd.next;
        rd.take_if(true);
        x = (uint64_t)lo | ((uint64_t)hi << 32);
    }
#ifdef HOH_DEBUG_FUSED
    if (blockIdx.x == 0 && lane < 3) {
        printf("lane %u cumtab: %08x %08x %08x %08x %08x %08x %08x\n", lane, cumtab[(size_t)s * kCumRow], cumtab[(size_t)s * kCumRow + 1], cumtab[(size_t)s * kCumRow + 2], cumtab[(size_t)s * kCumRow + 3], cumtab[(size_t)s * kCumRow + 4], cumtab[(size_t)s * kCumRow + 5], cumtab[(size_t)s * kCumRow + 6]);
        printf("lane %u tab:    %08x %08x %08x %08x %08x %08x %08x\n", lane, T.at(0), T.at(1), T.at(2), T.at(3), T.at(4), T.at(5), T.at(6));
        printf("lane %u s %u payload_off %llu x0 %llx rows: %08x %08x %08x %08x %08x lut0 %u lut64 %u lut127 %u pos %u shift %u\n", lane, s,
               (unsigned long long)m.payload_off, (unsigned long long)x, T.at(0), T.at(1), T.at(2), T.at(3), T.at(4), (unsigned)lut[lane],
               (unsigned)lut[64 * 32 + lane], (unsigned)lut[127 * 32 + lane], rd.pos, rd.shift);
    }
#endif
    const bool any_stored = __any_sync(0xffffffffu, stored);
    uint64_t acc = 0;  // stored lanes: bits not yet consumed, left-aligned
    uint32_t have = 0;
    const uint32_t sbits = m.maxbits;

    // geometry of the lane's tile (all tiles of the launch have the shape tw x th)
    const uint64_t t_glob = (uint64_t)blockIdx.x * kFusedTiles + min(tl, (uint32_t)kFusedTiles - 1u);
    const uint64_t image = t_glob / g.tiles_per_image;
    const uint32_t tile = (uint32_t)(t_glob % g.tiles_per_image);
    const uint32_t x0 = (tile % g.x_tiles) * g.tile_w, y0 = (tile / g.x_tiles) * g.tile_h;
    uint8_t* img = rgb + image * (uint64_t)g.width * g.height * 3u;
    const uint64_t row_bytes = (uint64_t)g.width * 3u;
    uint8_t* tile0 = img + ((uint64_t)y0 * g.width + x0) * 3u;  // pixel (0, 0) of the tile
    // per-lane constants of the colour transform: byte of the pixel this lane owns (R, G, B = 0, 1, 2)
    const uint32_t half = ch == 0u ? 128u : 256u, cmask = ch == 0u ? 255u : 511u;
    const uint32_t own_shift = ch == 0u ? 8u : (ch == 1u ? 0u : 16u);
    const uint32_t g_keep = ch == 0u ? 0u : 0xffffffffu, hi_keep = ch == 0u ? 0u : 0x01010101u;  // planes 1, 2 are differences to G
    const uint32_t my_stage_s = (uint32_t)__cvta_generic_to_shared(stage + tl * 24u + (own_shift >> 3));
    const uint2* my_out_src = reinterpret_cast<const uint2*>(stage + tl * 24u + 8u * ch);
    // Image addresses advance incrementally, one 64-bit add per group: p_cur = first byte of the current group of 8
    // pixels, p_px = where this lane stores its 8 bytes of the group the pixel in flight belongs to.  (Recomputed from
    // (x, y) per group they cost two chains of 64-bit multiply-adds and constant-bank loads, and the `if` around the
    // store a divergent region with its reconvergence barrier: ~200 cycles per group in the ncu source view.)
    const uint64_t row_skip = row_bytes - (uint64_t)(tw - 8u) * 3u;  // last group of a row -> first group of the next
    uint8_t* p_cur = tile0;
    uint8_t* p_px = tile0 + 8u * ch;

    // The two chains are woven by hand (`step` below): the far-walk vote of every step is a branch the compiler
    // schedules nothing across, so what fills the lookup's two shared-memory round trips has to stand there in the source.
    uint32_t L = half, TLv = half;
    uint2 ta = make_uint2(0x80808080u, 0x80808080u), tb = ta, tc = ta;  // the 24 bytes above the current group (row 0: c/2)
    const uint32_t groups = npx / 8u;                 // tw % 8 == 0
    uint32_t gx = 0, gy = 0;                          // position of the current group in the tile (warp-uniform)
    // A pixel is finished in two parts that sit in the two shadows of the NEXT symbol's lookup (see the step below):
    // un-prediction proper (and the shuffle that carries G to the difference planes) while the midpoint entry is on
    // its way, the staging of the byte while the four table rows are.
    uint32_t v_pend = 0, gv_pend = 0;  // the pixel between its two parts: value in its plane, G of its tile
    auto pixel_part1 = [&](uint32_t r, uint32_t t, bool row_start) {
        if (row_start) {  // prediction.hpp:25-26
            L = half;
            TLv = half;
        }
        // median(T, L, (u16)(T + L - TL)) on 10-bit values: a negative gradient wraps to a huge unsigned value in 32 bits
        // exactly as it does in the reference's 16 (predictor_operations.hpp:37-60, SURVEY H6), so no 16-bit mask is needed
        const uint32_t grad = t + L - TLv;
        const uint32_t med = max(min(t, L), min(max(t, L), grad));
        const uint32_t v = (r + med - half) & cmask;  // inverse of prediction.hpp:34
        TLv = t;
        L = v;
        v_pend = v;
        gv_pend = __shfl_sync(0xffffffffu, v, base_lane);
    };
    auto pixel_part2 = [&](uint32_t slot) {  // inverse of channel.hpp:75-77 (mod 256: the +256 drops out)
        asm volatile("st.shared.u8 [%0], %1;" ::"r"(my_stage_s + 3u * slot), "r"(v_pend + (gv_pend & g_keep)) : "memory");
    };
    // T of the 8 pixels of a group from the 24 RGB bytes above them, byte-wise: own byte minus G (mod 256) in t_lo, and for
    // the difference planes the ninth bit (R - G + 256 has bit 8 set iff R >= G) in t_hi; row 0 is fed bytes 0x80, which
    // give c/2 for every plane (prediction.hpp:20-22)
    uint32_t t01 = 0, t23 = 0, t45 = 0, t67 = 0;  // T of pixels (0,1), (2,3), (4,5), (6,7) of the group, two u16 each
    // __byte_perm selectors that pick this lane's own byte of pixels 0-3 / 4-7 out of three words (R, G or B)
    const uint32_t own_sel1 = ch == 0u ? 0x0741u : (ch == 1u ? 0x0630u : 0x0052u);
    const uint32_t own_sel2 = ch == 0u ? 0x6210u : (ch == 1u ? 0x5210u : 0x7410u);
    auto t_prepare = [&](uint2 a, uint2 b, uint2 c) {
        // bytes: a.x = R0 G0 B0 R1 | a.y = G1 B1 R2 G2 | b.x = B2 R3 G3 B3 | b.y = R4 G4 B4 R5 | c.x = G5 B5 R6 G6 | c.y = B6 R7 G7 B7
        const uint32_t g03 = __byte_perm(__byte_perm(a.x, a.y, 0x0741), b.x, 0x6210);  // G0 G1 G2 G3
        const uint32_t g47 = __byte_perm(__byte_perm(b.y, c.x, 0x0741), c.y, 0x6210);  // G4 G5 G6 G7
        const uint32_t o03 = __byte_perm(__byte_perm(a.x, a.y, own_sel1), b.x, own_sel2);
        const uint32_t o47 = __byte_perm(__byte_perm(b.y, c.x, own_sel1), c.y, own_sel2);
        const uint32_t lo03 = __vsub4(o03, g03 & g_keep), lo47 = __vsub4(o47, g47 & g_keep);
        const uint32_t hi03 = __vcmpgeu4(o03, g03) & hi_keep, hi47 = __vcmpgeu4(o47, g47) & hi_keep;
        t01 = __byte_perm(lo03, hi03, 0x5140);  // lo0 hi0 lo1 hi1
        t23 = __byte_perm(lo03, hi03, 0x7362);
        t45 = __byte_perm(lo47, hi47, 0x5140);
        t67 = __byte_perm(lo47, hi47, 0x7362);
    };
    auto t_of = [&](uint32_t i) -> uint32_t {
        const uint32_t pair = i < 2u ? t01 : (i < 4u ? t23 : (i < 6u ? t45 : t67));
        return (i & 1u) ? (pair >> 16) : (pair & 0xffffu);
    };
    // One symbol (rans_get_s, rans64.hpp:118-142) and one pixel, ordered by hand for the in-order issue of a warp: the
    // lookup of a symbol has two shared-memory round trips on the coder's chain (midpoint entry, then four table rows),
    // and ptxas leaves instructions where the source has them.  So the slot and the midpoint load of the NEXT symbol are
    // issued the moment the state is renormalised, the un-prediction of the symbol just decoded follows (it fills the
    // first round trip), and the staging of that pixel's byte comes after the row loads of the next step (it starts
    // filling the second).  Written as "finish the previous pixel, then decode" the two round trips were bare:
    // 48 + 40 cycles of a 311-cycle step waiting with nothing to issue (ncu source view).
    uint32_t slot = 0, key = 0, p_lut = 0;
    auto lookup_begin = [&]() {
        slot = (uint32_t)x & mask;  // rans64.hpp:118-121
        key = (slot + 1u) << kSymBits;
        if (sizeof(LutT) == 1) {
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(p_lut) : "r"(lut_s + (slot >> lut_shift) * 32u));
        } else {
            asm volatile("ld.shared.u16 %0, [%1];" : "=r"(p_lut) : "r"(lut_s + (slot >> lut_shift) * 64u));
        }
    };
    auto step = [&](auto has_stored, uint32_t i, bool row_start) {
        uint32_t em, e0, e1, e2;
        TS.at4(p_lut, em, e0, e1, e2);
        pixel_part2((i + 7u) & 7u);  // the pixel decoded one step ago (step 0: pixel 7 of the previous group)
        const bool down = e0 >= key;  // see rans_lookup_near
        const bool up = e1 < key;
        uint32_t e = down ? em : (up ? e1 : e0);
        uint32_t up_ones;
        asm("set.lt.u32.u32 %0, %1, %2;" : "=r"(up_ones) : "r"(e1), "r"(key));
        uint32_t hi = down ? e0 : e1 + ((e2 - e1) & up_ones);
        const bool near = e < key && hi >= key;
        const uint64_t top = x >> bits;
        uint64_t next = (uint64_t)((hi >> kSymBits) - (e >> kSymBits)) * top + (slot - (e >> kSymBits));  // rans64.hpp:126-134
        if (__builtin_expect(__any_sync(0xffffffffu, !near), 0)) {
            const ulonglong2 fixed = rans_far_step(TS, key, p_lut, e, hi, top, slot);
            next = fixed.x;
            e = (uint32_t)fixed.y;
        }
        x = next;
        const bool refill = ((uint32_t)(x >> 32) | ((uint32_t)x >> 31)) == 0u;  // rans64.hpp:137-141
        x = refill ? ((x << 32) | rd.next) : x;
        rd.take_if(refill);
        uint32_t r = e & kSymMask;
        if (decltype(has_stored)::value) {
            const bool fill = stored && have < sbits;
            if (fill) {
                acc |= (uint64_t)__byte_perm(rd.next, 0u, 0x0123) << (32u - have);
                have += 32u;
            }
            rd.take_if(fill);
            if (stored) {
                r = (uint32_t)(acc >> (64u - sbits));
                acc <<= sbits;
                have -= sbits;
            }
        }
        lookup_begin();
        pixel_part1(r, t_of(i), row_start);
    };
    auto flush_group = [&]() {  // the 24 staged bytes of every tile -> the image (a predicated store, no branch)
        __syncwarp();
        const uint2 v = *my_out_src;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.u32 p, %3, 0;\n"
            "@p st.global.v2.u32 [%0], {%1, %2};\n"
            "}\n" ::"l"(p_px),
            "r"(v.x), "r"(v.y), "r"((uint32_t)tile_ok)
            : "memory");
        __syncwarp();  // the stage may be rewritten, and the stores are ordered before the loads of later groups
    };
    // the loop exists twice: warps without a stored-mode stream (nearly all) run a copy without the bit reader
    auto run = [&](auto has_stored) {
    for (uint32_t grp = 0; grp < groups; grp++) {
        rd.top_up();
        uint32_t nx = gx + 8u, ny = gy;
        const bool wrap = nx == tw;
        if (wrap) {
            nx = 0u;
            ny++;
        }
        uint8_t* p_next = p_cur + (wrap ? row_skip : 24ull);
        t_prepare(ta, tb, tc);
        // step 0: symbol 0 of this group, and the byte of pixel 7 of the previous one, which completes that group.  (In
        // group 0 there is no such pixel: a zero byte goes to slot 7 and the flush stores the zeroed stage to the
        // tile's first 24 bytes, which group 0's own flush overwrites one group later - cheaper than a branch here.)
        step(has_stored, 0u, gx == 0u);
        flush_group();
        // the bytes above the NEXT group: stored at least one whole group ago (tile_w >= 16), and after the flush above
        uint2 na = make_uint2(0x80808080u, 0x80808080u), nb = na, nc = na;
        if (ny > 0u && ny < th && tile_ok) {
            const uint2* src = reinterpret_cast<const uint2*>(p_next - row_bytes);
            na = __ldcg(src);
            nb = __ldcg(src + 1);
            nc = __ldcg(src + 2);
        }
#pragma unroll
        for (uint32_t i = 1; i < 8u; i++) step(has_stored, i, false);
        p_px = p_cur + 8u * ch;
        p_cur = p_next;
        ta = na;
        tb = nb;
        tc = nc;
        gx = nx;
        gy = ny;
    }
    };
    lookup_begin();  // the first symbol's
    if (any_stored) {
        run(StoredYes{});
    } else {
        run(StoredNo{});
    }
    pixel_part2(7u);
    flush_group();
    // rans64.hpp:65: decoding undoes the encoder's steps, so a sound stream ends in the encoder's initial state
    if (coded && x != kRansL) my_status = HOH_S_BAD_STATE;
    if (exists) status[s] = my_status;
}

// Mode-0 tile back end WITH LZ back-references (hoh_decode_images_s0, d_backref != NULL): a copied pixel may
// depend on any earlier pixel of its tile (unprediction.hpp:63-65), so the wavefront does not apply; one thread
// walks one channel plane in raster order.  Residuals are dense (only the pixels no match covers have one,
// layer_encode.hpp:93-99); a stream that holds fewer or more residuals than the map leaves uncovered is reported.
__global__ void __launch_bounds__(64) k_tile_unpredict_s0_backref(const uint16_t* __restrict__ resid, TileGeom g,
                                                                  uint64_t n_tiles, const hoh_dec_result* __restrict__ res,
                                                                  const uint16_t* __restrict__ backref,
                                                                  uint16_t* __restrict__ planes,
                                                                  int32_t* __restrict__ status) {
    const uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (s >= n_tiles * 3u) return;
    if (status[s] != HOH_S_OK) return;
    const uint64_t t = s / 3u;
    const uint32_t ch = (uint32_t)(s % 3u);
    uint32_t x0, y0, tw, th;
    tile_rect(g, (uint32_t)(t % g.tiles_per_image), x0, y0, tw, th);
    const int c = ch == 0 ? 256 : 512, half = c >> 1;
    const uint16_t* r = resid + s * (uint64_t)g.plane_stride;
    const uint16_t* br = backref + t * (uint64_t)g.plane_stride;
    uint16_t* o = planes + s * (uint64_t)g.plane_stride;
    const uint32_t have = res[s].n;
    uint32_t k = 0;
    bool bad = false;
    for (uint32_t y = 0; y < th; y++)
        for (uint32_t x = 0; x < tw; x++) {
            const uint32_t at = y * tw + x;
            const uint32_t b = br[at];
            if (b) {
                if (b > at) {
                    bad = true;
                    o[at] = (uint16_t)half;
                } else {
                    o[at] = o[at - b];
                }
                continue;
            }
            const int L = x ? o[at - 1] : half;
            const int T = y ? o[at - tw] : half;
            const int TL = (x && y) ? o[at - tw - 1] : half;
            const int rv = k < have ? r[k] : half;
            k++;
            o[at] = (uint16_t)((rv + p_med_grad(T, L, TL) - half) & (c - 1));
        }
    if (bad || k != have) status[s] = HOH_S_BAD_LAYER;
}

// planes (G, R-G, B-G at s*plane_stride) -> RGB8 in the image: algebraic inverse of channel.hpp:73-79 + tile scatter
__global__ void __launch_bounds__(256) k_tile_store_s0(const uint16_t* __restrict__ planes, TileGeom g,
                                                       uint8_t* __restrict__ rgb) {
    const uint64_t t = blockIdx.x;
    const uint64_t image = t / g.tiles_per_image;
    uint32_t x0, y0, tw, th;
    tile_rect(g, (uint32_t)(t % g.tiles_per_image), x0, y0, tw, th);
    uint8_t* img = rgb + image * (uint64_t)g.width * g.height * 3u;
    const uint16_t* a = planes + (t * 3u) * (uint64_t)g.plane_stride;
    const uint16_t* b = a + g.plane_stride;
    const uint16_t* c = b + g.plane_stride;
    for (uint32_t i = threadIdx.x; i < tw * th; i += blockDim.x) {
        const uint32_t x = i % tw, y = i / tw;
        uint8_t* o = img + ((uint64_t)(y0 + y) * g.width + x0 + x) * 3u;
        const uint32_t gr = a[i];
        o[1] = (uint8_t)gr;
        o[0] = (uint8_t)((b[i] + gr - 256u) & 255u);
        o[2] = (uint8_t)((c[i] + gr - 256u) & 255u);
    }
}

}  // namespace hohk
