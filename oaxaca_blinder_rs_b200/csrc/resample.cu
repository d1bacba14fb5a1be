// csrc/resample.cu -- replicate generation: the multiplicity matrix C (rows x replicate slots).
//
// Replaces DataFrame::sample_n_literal(n_g, with_replacement=true) + the gather of every column
// (builder.rs:822-829): a replicate is fully described by how often each row was drawn, so the
// resample is a count vector c[:,b] ~ Multinomial(n_g; 1/n_g, ..) and no row is ever moved.
//
// Layout per group: C[panel][row][BM] (count_t = uint8/uint16), panel = 128 replicate slots, so a
// (32 rows x 128 slots) tile is one contiguous TMA bulk copy for gram.cu.  Slot 0 of panel 0 is the
// point estimate (count 1 on every valid row); slot s >= 1 is global replicate rep_first + s - 1.
//
// Two sources:
//  (a) counts_from_indices: explicit index stream (parity tests) -> exact histogram, bit-exact
//      against the oracle's gather for any stream.
//  (b) counts_philox: native counter-based stream.  Exact multinomial without n*B global atomics:
//        body   c_i ~ iid Poisson(lambda), lambda = 1 - delta/n, delta = ceil(8 sqrt(n)), by 64-bit
//               inverse-CDF of a Philox4x32-10 word keyed by (seed; row, group, replicate)
//               -> conditional on the column sum S the body is Multinomial(S; uniform);
//        fix-up n - S (about 8 sqrt(n), >= 0 except with probability < 1e-15) further uniform draws
//               added with atomics -> Multinomial(n; uniform) exactly, sum of counts = n_g as the
//               reference's unweighted means require (estimation.rs:66, ols.rs:83).
//      Every draw is keyed by global ids, so counts do not depend on grid shape, batch split or on
//      how replicates/rows are sharded over GPUs.
//  (c) bayes_weights: the Bayesian bootstrap's fp32 weights E_i ~ Exp(1) in the same layout (see BayesArgs).
#include "common.cuh"
#include "internal.h"

#include <cstdlib>

#include <cmath>

namespace ob {

constexpr int KMAX = 24;  // P(Poisson(<=1) > 23) < 2^-64

struct PoissonTable {
    unsigned long long T[KMAX];  // T[k] = floor(P(X <= k) * 2^64); count = #{k : U >= T[k]}
    unsigned short T16[KMAX];    // top 16 bits of T[k]
    int lambda_zero;
};

// counter layout: (c0, c1, c2, c3) = (row_lo | draw_lo, row_hi | group<<8, replicate key, stream tag)
enum : uint32_t { STREAM_BODY = 0x0B0D1u, STREAM_REFINE = 0x0F19Eu, STREAM_FIXUP = 0x0F1Cu };

// A count is the inverse CDF of a 64-bit uniform U = (u16 : 48 refinement bits), resolved lazily:
//   1. the top 14 bits of u16 index a 16 KB byte table (built once per call, copied to shared memory): the count if
//      every U of that bucket gives the same one, else AMBIG -- a threshold falls inside ~7 of the 16384 buckets;
//   2. AMBIG: compare all 16 bits with the thresholds' top 16 bits; still undecided only if u16 EQUALS one of them;
//   3. only then (p ~ 1e-4) are the low 48 bits drawn, from the refinement stream keyed by the single
//      (row, replicate), and the full 64-bit comparison made.
// The result is exactly the 64-bit inverse CDF, at 16 random bits and one LDS per count.
constexpr int LUT_BITS = 14;
constexpr int LUT_SIZE = 1 << LUT_BITS;
constexpr unsigned AMBIG = 255u;

__device__ __forceinline__ int cdf_count(unsigned long long U, const PoissonTable& t) {
    int c = 0;
#pragma unroll 1
    for (int k = 0; k < KMAX; ++k) c += (U >= t.T[k]) ? 1 : 0;
    return c;
}

// device copy of the thresholds behind the byte table (read by the rare resolve path through a pointer, so that the
// body kernel needs no stack frame for it)
struct PoissonDev { unsigned long long T[KMAX]; unsigned int T16[KMAX]; };

__global__ void __launch_bounds__(256) counts_lut_kernel(const PoissonTable tab, unsigned char* __restrict__ lut) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= LUT_SIZE) return;
    if (b < KMAX) {
        PoissonDev* d = reinterpret_cast<PoissonDev*>(lut + LUT_SIZE);
        d->T[b] = tab.T[b]; d->T16[b] = tab.T16[b];
    }
    const unsigned long long lo = (unsigned long long)b << (64 - LUT_BITS);
    const unsigned long long hi = lo | ((1ull << (64 - LUT_BITS)) - 1ull);
    const int cl = cdf_count(lo, tab), ch = cdf_count(hi, tab);
    lut[b] = (unsigned char)(cl == ch ? cl : AMBIG);
}

__device__ __noinline__ unsigned poisson_resolve(uint32_t u16, const PoissonDev* __restrict__ t, uint64_t row, uint32_t c1,
                                                 uint64_t rep, uint32_t k0, uint32_t k1) {
    unsigned c = 0; bool tie = false;
#pragma unroll 1
    for (int k = 0; k < KMAX; ++k) { c += (u16 > t->T16[k]) ? 1u : 0u; tie |= (u16 == t->T16[k]); }
    if (!tie) return c;
    const Philox4 r = philox4x32_10((uint32_t)row, c1, (uint32_t)rep, STREAM_REFINE ^ (uint32_t)(rep >> 32), k0, k1);
    const unsigned long long U = ((unsigned long long)u16 << 48) | ((unsigned long long)r.x << 16) | (r.y >> 16);
    c = 0;
#pragma unroll 1
    for (int k = 0; k < KMAX; ++k) c += (U >= t->T[k]) ? 1u : 0u;
    return c;
}

// Replicate r draws from stream id r + 1 (so that, unsharded, stream ids coincide with slots: the point estimate
// occupies slot 0); one Philox4x32-10 call yields the 16-bit uniforms of the 8 stream ids of an aligned octet.
// SH = (stream id of local slot 0) mod 8, uniform over the launch -> compile-time: a thread's 16 consecutive slots
// span 2 (SH == 0) or 3 octets.
// 3 resident blocks per SM (80 registers, no spills): measured 4.5 % faster than 2 (113 registers) and than 4 (64, spills)
template <typename CountT, int SH>
__global__ void __launch_bounds__(256, 3) counts_philox_body(CountT* __restrict__ C, long long n, long long n_pad,
                                                          long long slots, long long rep0, int first_slot, int group,
                                                          uint32_t k0, uint32_t k1, int lambda_zero,
                                                          const unsigned char* __restrict__ lut_g,
                                                          long long* __restrict__ colsum, int rows_per_block,
                                                          long long row_begin_global) {
    __shared__ __align__(16) unsigned char lut[LUT_SIZE];
    __shared__ int ssum[BM];
    for (int b = threadIdx.x; b < LUT_SIZE / 16; b += blockDim.x)
        reinterpret_cast<uint4*>(lut)[b] = reinterpret_cast<const uint4*>(lut_g)[b];
    if (threadIdx.x < BM) ssum[threadIdx.x] = 0;
    __syncthreads();

    const int panel = blockIdx.y;
    const int q = threadIdx.x & 7;           // 16-slot group within the panel
    const int rl = threadIdx.x >> 3;         // row lane 0..31
    const long long slot0 = (long long)panel * BM + q * 16;
    const long long row_begin = (long long)blockIdx.x * rows_per_block;
    const uint32_t c1base = ((uint32_t)group << 8);
    // stream id of local slot s is rep0 + 1 + s; (sid_lo - SH) is a multiple of 8
    const long long sid_lo = rep0 + 1 + slot0;
    const long long oct_first = (sid_lo - SH) >> 3;
    constexpr int NOCT = SH ? 3 : 2;
    // validity of slot e (0..15) is row-independent: slot >= first_slot && slot < slots
    unsigned valid = 0;
#pragma unroll
    for (int e = 0; e < 16; ++e)
        if (slot0 + e >= first_slot && slot0 + e < slots) valid |= 1u << e;
    const bool point_slot = (slot0 == 0 && first_slot == 1);
    int sums[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) sums[e] = 0;

    for (long long row = row_begin + rl; row < row_begin + rows_per_block && row < n_pad; row += 32) {
        unsigned cnt[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) cnt[e] = 0;
        if (row < n) {
            const unsigned long long grow = (unsigned long long)(row + row_begin_global);   // streams are keyed by the GLOBAL row
            const uint32_t c1 = c1base | (uint32_t)(grow >> 32);
            if (!lambda_zero && valid) {
                uint32_t w[4 * NOCT];
#pragma unroll
                for (int gi = 0; gi < NOCT; ++gi) {
                    const long long oc = oct_first + gi;
                    const Philox4 r = philox4x32_10((uint32_t)grow, c1, (uint32_t)oc, STREAM_BODY ^ (uint32_t)(oc >> 32), k0, k1);
                    w[4 * gi] = r.x; w[4 * gi + 1] = r.y; w[4 * gi + 2] = r.z; w[4 * gi + 3] = r.w;
                }
                unsigned any = 0;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int h = SH + e;                                   // 16-bit lane h of the thread's uniform words
                    const uint32_t idx = (h & 1) ? (w[h >> 1] >> (32 - LUT_BITS)) : ((w[h >> 1] >> (16 - LUT_BITS)) & (LUT_SIZE - 1));
                    cnt[e] = lut[idx];
                    any |= cnt[e];
                }
                if (any & 0x80u) {   // some bucket straddles a threshold (AMBIG = 255; real counts are < 24)
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        if (cnt[e] != AMBIG) continue;
                        const int h = SH + e;
                        const uint32_t u16 = (h & 1) ? (w[h >> 1] >> 16) : (w[h >> 1] & 0xFFFFu);
                        cnt[e] = poisson_resolve(u16, reinterpret_cast<const PoissonDev*>(lut_g + LUT_SIZE), grow, c1,
                                                 (uint64_t)(rep0 + slot0 + e), k0, k1);
                    }
                }
                if (valid != 0xFFFFu) {   // first / last panel only: slots outside [first_slot, slots) stay empty
#pragma unroll
                    for (int e = 0; e < 16; ++e) cnt[e] = (valid & (1u << e)) ? cnt[e] : 0u;
                }
            }
            if (point_slot) cnt[0] = 1;  // point estimate
#pragma unroll
            for (int e = 0; e < 16; ++e) sums[e] += (int)cnt[e];
        }
        CountT* dst = C + ((long long)panel * n_pad + row) * BM + q * 16;
        if (sizeof(CountT) == 1) {
            uint4 v;
            v.x = cnt[0] | (cnt[1] << 8) | (cnt[2] << 16) | (cnt[3] << 24);
            v.y = cnt[4] | (cnt[5] << 8) | (cnt[6] << 16) | (cnt[7] << 24);
            v.z = cnt[8] | (cnt[9] << 8) | (cnt[10] << 16) | (cnt[11] << 24);
            v.w = cnt[12] | (cnt[13] << 8) | (cnt[14] << 16) | (cnt[15] << 24);
            *reinterpret_cast<uint4*>(dst) = v;
        } else {
            uint4 v0, v1;
            v0.x = cnt[0] | (cnt[1] << 16); v0.y = cnt[2] | (cnt[3] << 16);
            v0.z = cnt[4] | (cnt[5] << 16); v0.w = cnt[6] | (cnt[7] << 16);
            v1.x = cnt[8] | (cnt[9] << 16); v1.y = cnt[10] | (cnt[11] << 16);
            v1.z = cnt[12] | (cnt[13] << 16); v1.w = cnt[14] | (cnt[15] << 16);
            reinterpret_cast<uint4*>(dst)[0] = v0;
            reinterpret_cast<uint4*>(dst)[1] = v1;
        }
    }
    // column sums: reduce the 4 row-lanes of each warp that share q, then the 8 warps through shared memory,
    // then ONE global atomic per (block, slot): same-address global atomics serialise in L2
#pragma unroll
    for (int e = 0; e < 16; ++e) {
        int s = sums[e];
        s += __shfl_xor_sync(0xffffffffu, s, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if ((threadIdx.x & 31) < 8 && s != 0) atomicAdd(&ssum[q * 16 + e], s);
    }
    __syncthreads();
    if (threadIdx.x < BM) {
        const long long slot = (long long)panel * BM + threadIdx.x;
        const int s = ssum[threadIdx.x];
        if (s != 0 && slot < slots) atomicAdd(reinterpret_cast<unsigned long long*>(colsum + slot), (unsigned long long)s);
    }
}

template <typename CountT>
__device__ __forceinline__ bool bump_count(CountT* C, long long elem) {
    // increment one count through a 32-bit atomic on its containing word; true if it was saturated
    unsigned int* word = reinterpret_cast<unsigned int*>(C) + (elem * (long long)sizeof(CountT)) / 4;
    const int shift = (int)((elem * (long long)sizeof(CountT)) & 3) * 8;
    const unsigned old = atomicAdd(word, 1u << shift);
    const unsigned mask = sizeof(CountT) == 1 ? 0xFFu : 0xFFFFu;
    return ((old >> shift) & mask) == mask;
}

template <typename CountT>
__global__ void __launch_bounds__(256) counts_philox_fixup(CountT* __restrict__ C, long long n, long long n_pad,
                                                           long long slots, long long rep0, int first_slot, int group,
                                                           uint32_t k0, uint32_t k1,
                                                           const long long* __restrict__ colsum, int* __restrict__ flags,
                                                           long long n_global, long long row_begin_global) {
    const long long slot = first_slot + blockIdx.x;
    if (slot >= slots) return;
    const long long need = n_global - colsum[slot];    // colsum: summed over all row shards
    if (need < 0) { if (threadIdx.x == 0 && blockIdx.y == 0) atomicOr(&flags[0], 1); return; }
    const long long rep = rep0 + slot;
    const long long panel = slot / BM, col = slot % BM;
    const uint32_t c1base = ((uint32_t)group << 8);
    for (long long j = (long long)blockIdx.y * blockDim.x + threadIdx.x; j < need; j += (long long)gridDim.y * blockDim.x) {
        const Philox4 r = philox4x32_10((uint32_t)j, c1base | (uint32_t)((unsigned long long)j >> 32), (uint32_t)rep,
                                        STREAM_FIXUP ^ (uint32_t)((unsigned long long)rep >> 32), k0, k1);
        const unsigned long long U = ((unsigned long long)r.x << 32) | r.y;
        // uniform on [0, n_global), bias < n / 2^64; rows outside this shard belong to another GPU
        const long long row = (long long)__umul64hi(U, (unsigned long long)n_global) - row_begin_global;
        if (row < 0 || row >= n) continue;
        if (bump_count<CountT>(C, (panel * n_pad + row) * BM + col)) atomicOr(&flags[1], 1);
    }
}

template <typename CountT>
__global__ void __launch_bounds__(256) counts_point_kernel(CountT* __restrict__ C, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) C[i * BM] = 1;  // panel 0, slot 0
}

template <typename CountT>
__global__ void __launch_bounds__(256) counts_index_kernel(CountT* __restrict__ C, long long n, long long n_pad,
                                                           long long r0, int first_slot,
                                                           const uint32_t* __restrict__ idx, int* __restrict__ flags,
                                                           long long n_global, long long row_begin_global) {
    const long long r = r0 + blockIdx.y;  // replicate of this batch -> slot first_slot + r
    const long long slot = first_slot + r, panel = slot / BM, col = slot % BM;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_global; i += (long long)gridDim.x * blockDim.x) {
        long long row = idx[r * n_global + i];
        if (row >= n_global) { atomicOr(&flags[2], 1); continue; }
        row -= row_begin_global;
        if (row < 0 || row >= n) continue;             // drawn row lives on another GPU
        if (bump_count<CountT>(C, (panel * n_pad + row) * BM + col)) atomicOr(&flags[1], 1);
    }
}

// ---- Bayesian bootstrap weights ----
constexpr uint32_t STREAM_BAYES = 0x0BA7E5u;

// E = -log U with U = (u >> 9 + 1/2) 2^-23 in [2^-24, 1 - 2^-24]: exact in fp32, open at both ends, so E is a positive
// normal float (5.96e-8 <= E <= 16.6)
__device__ __forceinline__ float exp1_from_u32(uint32_t u) {
    return -logf(((float)(u >> 9) + 0.5f) * 0x1p-23f);
}

// Block = (leaf segment held here, panel); thread = (row lane rl = tid / 32, slot quad q = tid % 32): rows rl, rl + 8, ..
// of the leaf, slots 4q .. 4q + 3 of the panel (one 16-byte store per row).  Replicate r draws the 32-bit word of stream
// id sid = r + 1 (the slot of r when unsharded) from the Philox call keyed by sid / 4; SH = sid of the thread's first
// slot mod 4, uniform over the launch: the thread's four slots span one (SH == 0) or two calls.  Each (leaf, slot) sum
// adds the thread's rows in order, then the eight row lanes in order: fixed by the leaf alone.
template <int SH, bool EXPLICIT>
__global__ void __launch_bounds__(256) bayes_weights_kernel(const BayesArgs a, uint32_t k0, uint32_t k1) {
    __shared__ double red[8][BM];
    const int leaf = blockIdx.x, panel = blockIdx.y;
    const int q = threadIdx.x & 31, rl = threadIdx.x >> 5;
    const long long slot0 = (long long)panel * BM + 4 * q;
    const long long r_lo = (long long)leaf * a.seg_rows;
    const long long r_hi = r_lo + a.seg_rows < a.n_pad ? r_lo + a.seg_rows : a.n_pad;
    unsigned valid = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e)
        if (slot0 + e >= a.first_slot && slot0 + e < a.slots) valid |= 1u << e;
    const bool point_slot = slot0 == 0 && a.first_slot == 1;
    const long long quad0 = (a.rep0 + 1 + slot0 - SH) >> 2;
    constexpr int NQ = SH ? 2 : 1;
    const uint32_t c1base = (uint32_t)a.group << 8;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long row = r_lo + rl; row < r_hi; row += 8) {
        float E[4] = {0.f, 0.f, 0.f, 0.f};
        if (row < a.n) {
            const unsigned long long grow = (unsigned long long)(row + a.row_begin);   // keyed by the GLOBAL row
            if (EXPLICIT) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (!(valid & (1u << e))) continue;
                    E[e] = a.wt[(size_t)(slot0 + e - a.first_slot) * a.n_global + grow];
                    // the Gram kernel widens positive normal floats only; a caller's zero, denormal, negative, inf or NaN
                    // fails the call
                    if (!(E[e] >= 1.17549435e-38f && E[e] <= 3.40282347e38f)) { atomicOr(&a.flags[3], 1); E[e] = 0.f; }
                }
            } else if (valid) {
                const uint32_t c1 = c1base | (uint32_t)(grow >> 32);
                uint32_t w[4 * NQ];
#pragma unroll
                for (int h = 0; h < NQ; ++h) {
                    const long long qd = quad0 + h;
                    const Philox4 r = philox4x32_10((uint32_t)grow, c1, (uint32_t)qd, STREAM_BAYES ^ (uint32_t)((unsigned long long)qd >> 32), k0, k1);
                    w[4 * h] = r.x; w[4 * h + 1] = r.y; w[4 * h + 2] = r.z; w[4 * h + 3] = r.w;
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) E[e] = (valid & (1u << e)) ? exp1_from_u32(w[SH + e]) : 0.f;
            }
            if (point_slot) E[0] = 1.f;
        }
        *reinterpret_cast<float4*>(a.C + ((long long)panel * a.n_pad + row) * BM + 4 * q) = make_float4(E[0], E[1], E[2], E[3]);
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] += (double)E[e];
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) red[rl][4 * q + e] = acc[e];
    __syncthreads();
    if (threadIdx.x < BM) {
        double s = red[0][threadIdx.x];
#pragma unroll
        for (int l = 1; l < 8; ++l) s += red[l][threadIdx.x];
        a.part[(size_t)leaf * a.panels * BM + (size_t)panel * BM + threadIdx.x] = s;
    }
}

void bayes_weights_launch(const BayesArgs& a, cudaStream_t st) {
    if (a.segs <= 0 || a.panels <= 0) return;
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    const dim3 grid((unsigned)a.segs, (unsigned)a.panels);
    if (a.wt) {
        bayes_weights_kernel<0, true><<<grid, 256, 0, st>>>(a, k0, k1);
    } else {
        switch ((int)(((a.rep0 + 1) % 4 + 4) % 4)) {
        case 0: bayes_weights_kernel<0, false><<<grid, 256, 0, st>>>(a, k0, k1); break;
        case 1: bayes_weights_kernel<1, false><<<grid, 256, 0, st>>>(a, k0, k1); break;
        case 2: bayes_weights_kernel<2, false><<<grid, 256, 0, st>>>(a, k0, k1); break;
        default: bayes_weights_kernel<3, false><<<grid, 256, 0, st>>>(a, k0, k1); break;
        }
    }
    OB_CUDA(cudaGetLastError());
}

void counts_clear(const CountsArgs& a, cudaStream_t st) {
    OB_CUDA(cudaMemsetAsync(a.C, 0, (size_t)a.panels * a.n_pad * BM * a.count_bytes, st));
}

void counts_from_indices(const CountsArgs& a, const uint32_t* d_idx, int* d_flags, cudaStream_t st) {
    counts_clear(a, st);
    const int pb = (int)((a.n + 255) / 256);
    const int pbg = (int)std::max<long long>((a.n_global + 255) / 256, 1);
    const long long reps = a.slots - a.first_slot;
    if (a.first_slot == 1 && pb > 0) {
        if (a.count_bytes == 1) counts_point_kernel<uint8_t><<<pb, 256, 0, st>>>((uint8_t*)a.C, a.n);
        else counts_point_kernel<uint16_t><<<pb, 256, 0, st>>>((uint16_t*)a.C, a.n);
        OB_CUDA(cudaGetLastError());
    }
    for (long long done = 0; done < reps; done += 32768) {  // gridDim.y <= 65535
        const long long nb = std::min<long long>(reps - done, 32768);
        dim3 grid((unsigned)std::min<long long>(pbg, 1024), (unsigned)nb);
        if (a.count_bytes == 1)
            counts_index_kernel<uint8_t><<<grid, 256, 0, st>>>((uint8_t*)a.C, a.n, a.n_pad, done, a.first_slot, d_idx, d_flags,
                                                               a.n_global, a.row_begin);
        else
            counts_index_kernel<uint16_t><<<grid, 256, 0, st>>>((uint16_t*)a.C, a.n, a.n_pad, done, a.first_slot, d_idx, d_flags,
                                                                a.n_global, a.row_begin);
        OB_CUDA(cudaGetLastError());
    }
}

static PoissonTable make_table(long long n) {
    PoissonTable t{};
    const long double delta = ceill(8.0L * sqrtl((long double)n));
    if (delta >= (long double)n) { t.lambda_zero = 1; return t; }
    const long double lam = ((long double)n - delta) / (long double)n;
    long double p = expl(-lam), cdf = 0.0L;
    const long double two64 = 18446744073709551616.0L;
    for (int k = 0; k < KMAX; ++k) {
        cdf += p;
        long double v = floorl(cdf * two64);
        t.T[k] = (v >= two64 || cdf >= 1.0L) ? 0xFFFFFFFFFFFFFFFFull : (unsigned long long)v;
        t.T16[k] = (unsigned short)(t.T[k] >> 48);
        p = p * lam / (long double)(k + 1);
    }
    t.lambda_zero = 0;
    return t;
}

size_t counts_lut_bytes() { return LUT_SIZE + ((sizeof(PoissonDev) + 255) / 256) * 256; }

void counts_philox_body_launch(const CountsArgs& a, long long* d_colsum, unsigned char* d_lut, cudaStream_t st) {
    const PoissonTable tab = make_table(a.n_global);       // lambda from the whole group's row count
    counts_lut_kernel<<<LUT_SIZE / 256, 256, 0, st>>>(tab, d_lut);
    OB_CUDA(cudaGetLastError());
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    const int rows_per_block = 2048;
    dim3 grid((unsigned)((a.n_pad + rows_per_block - 1) / rows_per_block), (unsigned)a.panels);
    const int sh = (int)((((a.rep0 + 1) % 8) + 8) % 8);
    auto body = [&](auto ct) {
        using CT = decltype(ct);
#define OB_BODY(SHV) counts_philox_body<CT, SHV><<<grid, 256, 0, st>>>((CT*)a.C, a.n, a.n_pad, a.slots, a.rep0, \
            a.first_slot, a.group, k0, k1, tab.lambda_zero, d_lut, d_colsum, rows_per_block, a.row_begin)
        switch (sh) {
        case 0: OB_BODY(0); break; case 1: OB_BODY(1); break; case 2: OB_BODY(2); break; case 3: OB_BODY(3); break;
        case 4: OB_BODY(4); break; case 5: OB_BODY(5); break; case 6: OB_BODY(6); break; default: OB_BODY(7);
        }
#undef OB_BODY
    };
    if (a.count_bytes == 1) body(uint8_t{}); else body(uint16_t{});
    OB_CUDA(cudaGetLastError());
}

void counts_philox_fixup_launch(const CountsArgs& a, const long long* d_colsum, int* d_flags, cudaStream_t st) {
    const long long nrep = a.slots - a.first_slot;
    if (nrep <= 0) return;
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    dim3 fgrid((unsigned)nrep, 16);
    if (a.count_bytes == 1)
        counts_philox_fixup<uint8_t><<<fgrid, 256, 0, st>>>((uint8_t*)a.C, a.n, a.n_pad, a.slots, a.rep0, a.first_slot,
                                                            a.group, k0, k1, d_colsum, d_flags, a.n_global, a.row_begin);
    else
        counts_philox_fixup<uint16_t><<<fgrid, 256, 0, st>>>((uint16_t*)a.C, a.n, a.n_pad, a.slots, a.rep0, a.first_slot,
                                                             a.group, k0, k1, d_colsum, d_flags, a.n_global, a.row_begin);
    OB_CUDA(cudaGetLastError());
}

}  // namespace ob
