// csrc/gram.cu -- replicate Gram / cross-product accumulation  G_b = sum_i c[i,b] w_i z_i  on the
// FP64 tensor cores (DMMA.8x8x4), replacing per replicate the gather + X'WX + X'Wy + column means
// of the reference (builder.rs:822-829 sample_n_literal, prepare_data :294-378, ols.rs:68-89,
// estimation.rs:56-71).
//
// Contraction:  [slots x n] (multiplicities, A operand)  x  [n x P'] (Z, B operand), per group.
//   * A[i][b] = c[i,b]: counts arrive as uint8/uint16 tiles by TMA bulk copy and are widened once per
//     CTA tile into an fp64 shared-memory tile (table lookup / exact magic-number conversion).  Sample
//     weights live in the B operand: the design rows are sqrt(w)-scaled once at pack time (ols.rs:68-78).
//   * Z is never materialised (110 GB at n=1e7,K=51): z_i[(j,l)] = x_ij * x_il is formed in
//     registers from the staged design rows while loading B fragments (one DMUL per fragment
//     element, 1/64 of the DMMA work).  Column (j,l) order = row-major upper triangle of
//     [x|y][x|y]^T, so G, X'Wy, the column sums (means) and sum(w) all come out of one pass.
//   * CTA tile 128 slots x 128 columns, 8 warps (1 x 8), warp tile 128 x 16 = 16 x 2 DMMA sub-tiles,
//     KT = 32 rows per stage, 3-stage TMA/mbarrier pipeline.  The last column tile is cut to one, two or three
//     quanta of 32 columns (one 8-column DMMA sub-tile per scheduler) when that is all it needs: K = 17 costs 1.5
//     tiles, K = 31 4.25, K = 51 with two four-level categoricals 10.75 (structural zeros are not computed).
//   * Split-n: the rows of a group are cut into <= 256 fixed leaf segments whose size depends only on the
//     group's GLOBAL row count.  Work unit = (group, panel, segment, column tile): accumulated from zero,
//     flushed as one partial tile.  A persistent grid of one CTA per SM walks cost-balanced contiguous
//     unit ranges; gram_reduce sums a tile's leaf partials by a fixed aligned binary tree.  The summation
//     tree of every Gram entry is therefore fixed by (n_g, K) alone: results are bit-identical run to
//     run and do not depend on how replicates are batched, or on how replicates (mode R) or rows (mode
//     N: each GPU reduces an aligned subtree, gram_combine evaluates the top levels) are sharded.
#include "common.cuh"
#include "internal.h"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace ob {

// Every warp reads A fragments of 8 k-rows x (MI*8) slots, so the fp64 A tile is fragment-major:
//   As[k][lg][i] = A[k][m = 8 i + lg],  offset k * LDA2 + lg * LGS + i
// -> the MI values a thread needs for one k-step are contiguous: MI/2 x LDS.128 instead of MI x LDS.64.
// LGS = 18 and LDA2 = 148 (LDA2 / 2 = 2 mod 8) keep both the LDS.128 fragment loads and the STS.128 widening
// stores bank-conflict free.
constexpr int LGS = 18;
constexpr int LDA2 = 148;
constexpr int A_TILE = KT * LDA2;   // doubles per A buffer

struct GramKernelParams {
    const double* X[2];     // per group: (sqrt(w)-scaled) design rows [n_pad][ldx]
    const void* C[2];
    long long n_pad[2];
    int segs[2];            // row segments (leaves) held here, per group: stride of the partial-tile index
    int seg_lo[2], seg_n[2];// leaves [seg_lo, seg_lo + seg_n) this LAUNCH covers (all of them, or the part of the design that has
                            // already arrived when the upload is still in flight: ob_design_pack_async)
    int seg_rows[2];        // rows per segment (multiple of KT)
    long long units0;       // units of group 0 = panels * ntiles * segs[0]
    long long units_total;
    int ldx, panels, ntiles;
    int nfull, tail_q;      // column tiling: nfull tiles of BN columns + (tail_q ? one tile of tail_q * BQ columns : none)
    int tail_mi;            // warp-specialised kernel: 8-slot groups of the LAST panel that hold valid slots, rounded up to
                            // a multiple of 4 (16 = the panel is full): its units skip the DMMAs of the empty groups
    double* partials;       // [units_total][BM*BN], unit-major (a tail tile uses the first BM * tail_q * BQ doubles, that row stride)
    const uint16_t* pairs;
};

// Widening of the count tile.  Thread (r = tid / 8, lg = tid % 8) converts slots m = 8 i + lg of row r, two i per
// step (one STS.128 at As[r][lg][2e]), so the eight steps of the NEXT stage are interleaved with the eight k-steps
// of the current stage's DMMA loop.  uint8 counts go through a 256-entry fp64 table in shared memory (no FP64-pipe
// work: that pipe is what the DMMAs need); uint16 counts use the exact magic-number conversion (2^52 + c) - 2^52.
// Sample weights are NOT applied here: the design rows are already sqrt(w)-scaled (ols.rs:68-78), so A is the
// bare multiplicity.  fp32 Bayesian-bootstrap weights (resample.cu) are widened by integer bit operations alone: for a
// positive normal float the fp64 exponent is the fp32 one rebiased by 1023 - 127 = 896 and the 23 mantissa bits move up
// by 29, so the value is exact and the FP64 pipe stays free for the DMMAs; 0.0f (padding rows, empty slots) stays 0.0.
template <typename CountT>
__device__ __forceinline__ double count_to_f64(CountT c, const double* __restrict__ tab) {
    if constexpr (std::is_same<CountT, float>::value) {
        const uint32_t f = __float_as_uint(c);
        return __hiloint2double(f ? (int)((f >> 3) + (896u << 20)) : 0, (int)(f << 29));
    } else if constexpr (sizeof(CountT) == 1) {
        return tab[(unsigned)c];
    } else {
        return __hiloint2double(0x43300000, (int)(unsigned)c) - 4503599627370496.0;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Warp-specialised CTA: 8 consumer warps issue nothing but fragment loads and DMMAs; a
// producer warpgroup (4 warps) owns the TMA issue and the widening of the count tiles.  Ring of WS_R slots, each holding a stage's
// raw counts, design rows and widened fp64 A tile; three mbarriers per slot:
//   full[s]      TMA bytes landed             (producer lane 0 arms it; producer and consumers wait)
//   ready[s]     A tile widened               (one arrival per producer warp; consumers wait)
//   consumed[s]  stage finished by a warp     (one arrival per consumer warp; producer waits before reusing the slot)
// Stage numbers run on across work units, so the producer prefetches and widens the next unit's first stages while
// the consumers finish the current one: no per-unit pipeline fill, no CTA-wide barrier in the loop.
constexpr int WS_R = 3;   // ring depth; designs too wide for three stages in shared memory (K + T > ~120) run with two
constexpr int WS_PRODUCER_WARPS = 4;                       // one warpgroup, so that setmaxnreg can rebalance registers
constexpr int WS_THREADS = GRAM_THREADS + 32 * WS_PRODUCER_WARPS;
// register budget: 384 threads x 168 at launch; the producer warpgroup drops to 56, the two consumer warpgroups rise to 224
#define OB_WS_CONSUMER_REGS 224
#define OB_WS_PRODUCER_REGS 56

struct GramUnit { const double* Xg; const void* Cg; double* out; int nstages, nt, mi, tq; };   // tq: quanta of the tile (4 = full)

// Unit sequence of the warp-specialised kernel: four cost classes, each in (group, segment, panel, tile) order --
// wide tiles of full panels, wide tiles of the tail panel, tail tiles of full panels, tail tiles of the tail panel.  CTA b takes positions b, b + grid, ...: equal shares of every class, lockstep through consecutive units.
__host__ __device__ __forceinline__ bool ws_decode(const GramKernelParams& p, long long i, int ldx, size_t count_bytes, GramUnit& u) {
    const int pt = p.tail_mi < 16 ? 1 : 0, pf = p.panels - pt;            // tail / full panels of this batch
    const long long segs01 = (long long)p.seg_n[0] + p.seg_n[1];
    const long long n0 = segs01 * pf * p.nfull, n1 = segs01 * pt * p.nfull;
    const long long n2 = p.tail_q ? segs01 * pf : 0, n3 = p.tail_q ? segs01 * pt : 0;
    if (i >= n0 + n1 + n2 + n3) return false;
    int np, p0, nt_cnt, nt0;          // panels / first panel / tiles per sweep / first tile of the class
    if (i < n0) { np = pf; p0 = 0; nt_cnt = p.nfull; nt0 = 0; }
    else if ((i -= n0) < n1) { np = pt; p0 = pf; nt_cnt = p.nfull; nt0 = 0; }
    else if ((i -= n1) < n2) { np = pf; p0 = 0; nt_cnt = 1; nt0 = p.nfull; }
    else { i -= n2; np = pt; p0 = pf; nt_cnt = 1; nt0 = p.nfull; }
    const long long per_seg = (long long)np * nt_cnt;
    const long long g0 = (long long)p.seg_n[0] * per_seg;
    const int g = i >= g0 ? 1 : 0;
    const long long r = i - (g ? g0 : 0);
    const int sidx = (int)(r / per_seg);
    const long long r2 = r - (long long)sidx * per_seg;
    const int seg = (g ? p.seg_lo[1] : p.seg_lo[0]) + sidx;
    const int panel = p0 + (int)(r2 / nt_cnt), nt = nt0 + (int)(r2 % nt_cnt);
    const int segs = g ? p.segs[1] : p.segs[0], seg_rows = g ? p.seg_rows[1] : p.seg_rows[0];
    const long long n_pad = g ? p.n_pad[1] : p.n_pad[0];
    const long long row0 = (long long)seg * seg_rows;
    const long long row1 = row0 + seg_rows < n_pad ? row0 + seg_rows : n_pad;
    u.nstages = (int)((row1 - row0) / KT);
    u.nt = nt; u.tq = (p.tail_q && nt == p.nfull) ? p.tail_q : 4;
    u.mi = panel >= pf ? p.tail_mi : 16;
    u.Xg = (g ? p.X[1] : p.X[0]) + row0 * ldx;
    u.Cg = reinterpret_cast<const unsigned char*>(g ? p.C[1] : p.C[0]) + (((long long)panel * n_pad + row0) * BM) * (long long)count_bytes;
    u.out = p.partials + (size_t)((g ? p.units0 : 0) + ((long long)panel * segs + seg) * p.ntiles + nt) * (BM * BN);
    return true;
}

// MI = 8-slot groups of the panel this warp accumulates (16 = all 128 slots; 4 / 8 / 12 for a partly filled tail panel)
// sub0: first of the warp's NI 8-column sub-tiles within the tile; tw: the tile's width (the partial tile's row stride)
template <typename CountT, int LDXC, int NI, int MI, int R>
__device__ __forceinline__ void ws_consume_unit(const GramKernelParams& p, const GramUnit& u, const double* As, const double* Xs,
                                                uint64_t* full, uint64_t* ready, uint64_t* consumed, int ldx_rt, uint32_t& jc,
                                                int sub0, int tw) {
    constexpr int KSTEPS = KT / 4;
    const int lane = threadIdx.x & 31;
    const int lk = lane & 3, lg = lane >> 2;
    const int ldx = LDXC ? LDXC : ldx_rt;
    int oj[NI], ol[NI];
#pragma unroll
    for (int s = 0; s < NI; ++s) {
        const int col = u.nt * BN + (sub0 + s) * 8 + lg;
        const uint32_t pr = *reinterpret_cast<const uint32_t*>(p.pairs + 2 * col);
        oj[s] = pr & 0xFFFFu; ol[s] = pr >> 16;
    }
    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int s = 0; s < NI; ++s) { acc[i][s][0] = 0.0; acc[i][s][1] = 0.0; }

    for (int s = 0; s < u.nstages; ++s) {
        const uint32_t slot = jc % R, par = (jc / R) & 1u;
        mbar_wait(&full[slot], par);       // design rows of this stage (TMA writes become visible to this thread)
        mbar_wait(&ready[slot], par);      // widened A tile
        const double* abase = As + (size_t)slot * A_TILE + lk * LDA2 + lg * LGS;
        const double* xbase = Xs + (size_t)slot * KT * ldx + lk * ldx;
#pragma unroll
        for (int kk = 0; kk < KSTEPS; ++kk) {
            double a[MI], b[NI];
            const double* arow = abase + kk * 4 * LDA2;
            const double* xrow = xbase + kk * 4 * ldx;
#pragma unroll
            for (int i = 0; i < MI; i += 2) {
                const double2 v = *reinterpret_cast<const double2*>(arow + i);
                a[i] = v.x; a[i + 1] = v.y;
            }
#pragma unroll
            for (int t = 0; t < NI; ++t) b[t] = xrow[oj[t]] * xrow[ol[t]];
#pragma unroll
            for (int i = 0; i < MI; ++i)
#pragma unroll
                for (int t = 0; t < NI; ++t) dmma884(acc[i][t][0], acc[i][t][1], a[i], b[t]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&consumed[slot]);
        ++jc;
    }
    // rows of slot groups >= MI are not written: those slots do not exist (the solve never reads them)
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int t = 0; t < NI; ++t) {
            const int m = i * 8 + lg, n = (sub0 + t) * 8 + 2 * lk;
            *reinterpret_cast<double2*>(u.out + m * tw + n) = make_double2(acc[i][t][0], acc[i][t][1]);
        }
}

template <typename CountT, int LDXC, int NI, int R>
__device__ __forceinline__ void ws_consume_dispatch(const GramKernelParams& p, const GramUnit& u, const double* As, const double* Xs,
                                                    uint64_t* full, uint64_t* ready, uint64_t* consumed, int ldx_rt, uint32_t& jc,
                                                    int sub0, int tw) {
    switch (u.mi) {
    case 4: ws_consume_unit<CountT, LDXC, NI, 4, R>(p, u, As, Xs, full, ready, consumed, ldx_rt, jc, sub0, tw); break;
    case 8: ws_consume_unit<CountT, LDXC, NI, 8, R>(p, u, As, Xs, full, ready, consumed, ldx_rt, jc, sub0, tw); break;
    case 12: ws_consume_unit<CountT, LDXC, NI, 12, R>(p, u, As, Xs, full, ready, consumed, ldx_rt, jc, sub0, tw); break;
    default: ws_consume_unit<CountT, LDXC, NI, 16, R>(p, u, As, Xs, full, ready, consumed, ldx_rt, jc, sub0, tw); break;
    }
}

// A consumer warp with no columns in a one-quantum tail tile keeps step with the ring: stage j's `consumed` arrival
// only once stage j's TMA has landed, i.e. after the slot's previous use has been released by all eight warps.
template <int R>
__device__ __forceinline__ void ws_idle_unit(const GramUnit& u, uint64_t* full, uint64_t* consumed, uint32_t& jc) {
    const int lane = threadIdx.x & 31;
    for (int s = 0; s < u.nstages; ++s) {
        const uint32_t slot = jc % R, par = (jc / R) & 1u;
        mbar_wait(&full[slot], par);
        __syncwarp();
        if (lane == 0) mbar_arrive(&consumed[slot]);
        ++jc;
    }
}

template <typename CountT, int LDXC, int R = WS_R>
__global__ void __launch_bounds__(WS_THREADS, 1) gram_ws_kernel(const GramKernelParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ldx = LDXC ? LDXC : p.ldx;
    double* As = reinterpret_cast<double*>(smem_raw);                           // [R][A_TILE]
    double* Tab = As + R * A_TILE;                                           // [256]
    double* Xs = Tab + 256;                                                     // [R][KT*ldx]
    CountT* Cr = reinterpret_cast<CountT*>(Xs + (size_t)R * KT * ldx);       // [R][KT*BM]
    uint64_t* full = reinterpret_cast<uint64_t*>(Cr + (size_t)R * KT * BM);  // [R]
    uint64_t* ready = full + R;
    uint64_t* consumed = ready + R;
    if (tid < 256) Tab[tid] = (double)tid;
    if (tid == 0) {
        for (int s = 0; s < R; ++s) { mbar_init(&full[s], 1); mbar_init(&ready[s], WS_PRODUCER_WARPS); mbar_init(&consumed[s], GRAM_THREADS / 32); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp < GRAM_THREADS / 32) {
        // ---------------- consumers ----------------
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(OB_WS_CONSUMER_REGS));
        uint32_t jc = 0;
        GramUnit u;
        for (long long i = blockIdx.x; ws_decode(p, i, ldx, sizeof(CountT), u); i += gridDim.x) {
            // the tile's quanta give every scheduler (warps w and w + 4) tq sub-tiles: 2 + 2, 2 + 1, 1 + 1 or 1 + 0
            const int tw = u.tq * BQ, hi = warp >> 2;
            int ni, sub0;
            if (u.tq == 4) { ni = 2; sub0 = warp * 2; }
            else if (u.tq == 2) { ni = 1; sub0 = warp; }
            else if (u.tq == 3) { ni = hi ? 1 : 2; sub0 = hi ? 4 + warp : warp * 2; }
            else { ni = hi ? 0 : 1; sub0 = warp; }
            if (ni == 2) ws_consume_dispatch<CountT, LDXC, 2, R>(p, u, As, Xs, full, ready, consumed, ldx, jc, sub0, tw);
            else if (ni == 1) ws_consume_dispatch<CountT, LDXC, 1, R>(p, u, As, Xs, full, ready, consumed, ldx, jc, sub0, tw);
            else ws_idle_unit<R>(u, full, consumed, jc);
        }
    } else {
        // ---------------- producers: TMA issue (warp 0 lane 0) + widening (4 warps x 8 rows) ----------------
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(OB_WS_PRODUCER_REGS));
        const int pw = warp - GRAM_THREADS / 32;
        const uint32_t stage_bytes = (uint32_t)(KT * ldx * sizeof(double) + KT * BM * sizeof(CountT));
        // two cursors over the (unit, stage) sequence: `is` = next stage to issue, `wi` = next stage to widen
        long long is_i = blockIdx.x, wi_i = blockIdx.x;
        int is_s = 0, wi_s = 0;
        GramUnit is_u, wi_u;
        bool is_ok = ws_decode(p, is_i, ldx, sizeof(CountT), is_u);
        bool wi_ok = ws_decode(p, wi_i, ldx, sizeof(CountT), wi_u);
        uint32_t ji = 0, jw = 0;
        auto issue_next = [&]() {   // stage ji -> slot ji % R
            const uint32_t slot = ji % R;
            if (pw == 0 && lane == 0) {
                fence_proxy_async();
                mbar_expect_tx(&full[slot], stage_bytes);
                tma_load_1d(Xs + (size_t)slot * KT * ldx, is_u.Xg + (long long)is_s * KT * ldx, KT * ldx * sizeof(double), &full[slot]);
                tma_load_1d(Cr + (size_t)slot * KT * BM, reinterpret_cast<const CountT*>(is_u.Cg) + (long long)is_s * KT * BM,
                            KT * BM * sizeof(CountT), &full[slot]);
            }
            ++ji;
            if (++is_s == is_u.nstages) { is_s = 0; is_i += gridDim.x; is_ok = ws_decode(p, is_i, ldx, sizeof(CountT), is_u); }
        };
        while (is_ok && ji < (uint32_t)R) issue_next();
        while (wi_ok) {
            const uint32_t slot = jw % R, par = (jw / R) & 1u;
            mbar_wait(&full[slot], par);
            // widen Cr[slot] (32 rows x 128 slots) -> As[slot], fragment-major; producer warp pw takes rows 8 pw .. 8 pw + 7
            {
                const CountT* src = Cr + (size_t)slot * KT * BM;
                double* dst = As + (size_t)slot * A_TILE;
                // item = (e, r, lg): slots m = 8 (2e) + lg and 8 (2e+1) + lg of row r -> one STS.128 at dst[r][lg][2e];
                // consecutive lanes take consecutive lg (then r): conflict-free stores (LGS = 18, LDA2 = 148)
#pragma unroll 4
                for (int it = lane; it < (KT / WS_PRODUCER_WARPS) * 8 * 8; it += 32) {
                    const int e = it >> 6, rem = it & 63, r = pw * (KT / WS_PRODUCER_WARPS) + (rem >> 3), lgq = rem & 7;
                    const CountT* sp = src + r * BM + lgq;
                    double2 o;
                    o.x = count_to_f64<CountT>(sp[e * 16], Tab);
                    o.y = count_to_f64<CountT>(sp[e * 16 + 8], Tab);
                    *reinterpret_cast<double2*>(dst + r * LDA2 + lgq * LGS + e * 2) = o;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&ready[slot]);
            ++jw;
            if (++wi_s == wi_u.nstages) { wi_s = 0; wi_i += gridDim.x; wi_ok = ws_decode(p, wi_i, ldx, sizeof(CountT), wi_u); }
            // refill: stage ji reuses the slot of stage ji - R, which the consumers must have finished (only the issuing
            // warp waits; the other producer warps meet the new stage at its full[] barrier)
            if (is_ok && ji <= jw + (uint32_t)(R - 2)) {
                const uint32_t prev = ji - R;
                if (pw == 0) mbar_wait(&consumed[prev % R], (prev / R) & 1u);
                issue_next();
            }
        }
    }
}

static constexpr size_t gram_ws_smem(int ldx, int count_bytes, int ring = WS_R) {
    return sizeof(double) * ((size_t)ring * A_TILE + 256 + (size_t)ring * KT * ldx) + (size_t)ring * KT * BM * count_bytes +
           sizeof(uint64_t) * 3 * ring;
}
constexpr size_t GRAM_SMEM_MAX = 227 * 1024;
// ring depth of the fp32-weight kernel at a specialised row stride: three stages up to ldx 84, two beyond
constexpr int gram_ring_f32(int ldx) { return gram_ws_smem(ldx, 4, WS_R) <= GRAM_SMEM_MAX ? WS_R : 2; }

// The Gram CTA fits in shared memory at this row stride and count width (two ring stages when three do not fit):
// ldx <= 284 (K + outcomes <= 280) with uint8 counts, ldx <= 268 (K + outcomes <= 268) with uint16 counts, ldx <= 236
// (K + outcomes <= 236) with fp32 Bayesian-bootstrap weights.
bool gram_fits(int ldx, int count_bytes) { return gram_ws_smem(ldx, count_bytes, 2) <= GRAM_SMEM_MAX; }

// Aligned binary summation tree over LEN consecutive leaves starting at `lo` (lo < cnt): leaves >= cnt are absent
// and skipped.  The tree shape depends on the leaf indices only, so any aligned sub-range reduced on another GPU
// (mode N) yields the very same intermediate sums.
template <int LEN>
__device__ __forceinline__ double2 tree_sum(const double2* __restrict__ base, size_t stride, int lo, int cnt);

// a 64-leaf subtree as a real call: keeps the 128- and 256-leaf trees from being flattened into hundreds of loads in
// flight at once (255 registers + spills); the tree shape is the same
__device__ __noinline__ double2 tree_sum64_call(const double2* __restrict__ base, size_t stride, int lo, int cnt);

template <int LEN>
__device__ __forceinline__ double2 tree_sum(const double2* __restrict__ base, size_t stride, int lo, int cnt) {
    if constexpr (LEN == 1) {
        return base[(size_t)lo * stride];
    } else if constexpr (LEN == 128) {
        double2 a = tree_sum64_call(base, stride, lo, cnt);
        if (lo + 64 < cnt) {
            const double2 b = tree_sum64_call(base, stride, lo + 64, cnt);
            a.x += b.x; a.y += b.y;
        }
        return a;
    } else {
        double2 a = tree_sum<LEN / 2>(base, stride, lo, cnt);
        if (lo + LEN / 2 < cnt) {
            const double2 b = tree_sum<LEN / 2>(base, stride, lo + LEN / 2, cnt);
            a.x += b.x; a.y += b.y;
        }
        return a;
    }
}

__device__ __noinline__ double2 tree_sum64_call(const double2* __restrict__ base, size_t stride, int lo, int cnt) {
    return tree_sum<64>(base, stride, lo, cnt);
}

__device__ __forceinline__ double2 tree_sum_span(const double2* __restrict__ base, size_t stride, int cnt, int span) {
    switch (span) {
    case 256: return tree_sum<256>(base, stride, 0, cnt);
    case 128: return tree_sum<128>(base, stride, 0, cnt);
    case 64: return tree_sum<64>(base, stride, 0, cnt);
    case 32: return tree_sum<32>(base, stride, 0, cnt);
    case 16: return tree_sum<16>(base, stride, 0, cnt);
    case 8: return tree_sum<8>(base, stride, 0, cnt);
    case 4: return tree_sum<4>(base, stride, 0, cnt);
    case 2: return tree_sum<2>(base, stride, 0, cnt);
    default: return tree_sum<1>(base, stride, 0, cnt);
    }
}

// out[g][panel*BM + m][colmap[nt*BN + n]] = tree sum over the tile's leaf partials held here (span = MAX_SEGS / world);
// the cells of the upper triangle that are not computed (structural zeros) have been zero-filled by the launcher
__global__ void __launch_bounds__(256) gram_reduce_kernel(const double* __restrict__ partials, int segs0, int segs1,
                                                          double* __restrict__ gram, int panels, int ntiles, int span,
                                                          int Pld, int tail_q, const int32_t* __restrict__ colmap) {
    const int tile_id = blockIdx.x;
    const int tiles_g = panels * ntiles;
    const int g = tile_id / tiles_g, t = tile_id - g * tiles_g;
    const int panel = t / ntiles, nt = t - panel * ntiles;
    const int cnt = g ? segs1 : segs0;
    // partial of (g, panel, nt, seg) sits at unit base_g + (panel * segs_g + seg) * ntiles + nt
    const size_t first = (g ? (size_t)tiles_g * segs0 : 0) + (size_t)panel * cnt * ntiles + nt;
    const size_t slots_pad = (size_t)panels * BM;
    const int tw = (tail_q && nt == ntiles - 1) ? tail_q * BQ : BN;     // this tile's width
    for (int e = threadIdx.x + blockIdx.y * blockDim.x; e < BM * tw / 2; e += blockDim.x * gridDim.y) {
        double2 s = make_double2(0.0, 0.0);
        if (cnt > 0) s = tree_sum_span(reinterpret_cast<const double2*>(partials + first * (BM * BN)) + e, (size_t)ntiles * (BM * BN / 2), cnt, span);
        const int m = (2 * e) / tw, n = (2 * e) % tw;
        double* dst = gram + ((size_t)g * slots_pad + (size_t)panel * BM + m) * (size_t)Pld;
        const int c0 = colmap[nt * BN + n], c1 = colmap[nt * BN + n + 1];
        if (c0 >= 0) dst[c0] = s.x;
        if (c1 >= 0) dst[c1] = s.y;
    }
}

// Per-slot sums of the Bayesian-bootstrap weights: out[g][slot] = tree sum over the group's leaf partials held here,
// part [segs0 + segs1][slots_pad] (group 0's leaves first).  The same aligned tree as gram_reduce, so the sums do not
// depend on batching, and mode N combines the per-rank sums with gram_combine_kernel into the single-GPU values.
__global__ void __launch_bounds__(256) leaf_sum_kernel(const double* __restrict__ part, int segs0, int segs1, long long half,
                                                       int span, double* __restrict__ out) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < 2 * half; e += (long long)gridDim.x * blockDim.x) {
        const int g = e >= half ? 1 : 0;
        const int cnt = g ? segs1 : segs0;
        const double2* base = reinterpret_cast<const double2*>(part + (g ? (size_t)segs0 * 2 * half : 0)) + (e - (g ? half : 0));
        reinterpret_cast<double2*>(out)[e] = cnt > 0 ? tree_sum_span(base, (size_t)half, cnt, span) : make_double2(0.0, 0.0);
    }
}

// mode N: the upper levels of the same tree, over the per-rank sums gathered from all GPUs
__global__ void __launch_bounds__(256) gram_combine_kernel(const double* __restrict__ gathered, int world, int ranks0,
                                                           int ranks1, long long per_group2, double* __restrict__ gram) {
    // gathered [world][2][per_group] doubles; per_group2 = per_group / 2 double2 elements
    const long long total = 2 * per_group2;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int g = e >= per_group2 ? 1 : 0;
        const int cnt = g ? ranks1 : ranks0;
        double2 s = make_double2(0.0, 0.0);
        if (cnt > 0) s = tree_sum_span(reinterpret_cast<const double2*>(gathered) + e, (size_t)total, cnt, world);
        reinterpret_cast<double2*>(gram)[e] = s;
    }
}

GramColumns gram_columns(int K, int T, int n_cont, const std::vector<int>& cat_levels) {
    // dummy block of every design column (-1: intercept / continuous): two different columns of one block never are
    // non-zero on the same row
    std::vector<int> block((size_t)K, -1);
    {
        int64_t dummies = 0;
        for (int m : cat_levels) dummies += m > 1 ? m - 1 : 0;
        if (!cat_levels.empty() && 1 + (int64_t)n_cont + dummies == K) {
            int c = 1 + n_cont;
            for (size_t q = 0; q < cat_levels.size(); ++q)
                for (int lvl = 1; lvl < cat_levels[q]; ++lvl) block[(size_t)c++] = (int)q;
        }
    }
    GramColumns gc;
    std::vector<uint16_t> pj, pl; std::vector<int32_t> cm;
    for (int j = 0; j < K; ++j) {
        const int64_t base = pair_base(K, T, j);
        for (int l = j; l < K; ++l) {
            if (l > j && block[(size_t)j] >= 0 && block[(size_t)j] == block[(size_t)l]) continue;     // structural zero
            pj.push_back((uint16_t)j); pl.push_back((uint16_t)l); cm.push_back((int32_t)(base + (l - j)));
        }
        for (int o = 0; o < T; ++o) { pj.push_back((uint16_t)j); pl.push_back((uint16_t)(K + o)); cm.push_back((int32_t)(base + (K - j) + o)); }
    }
    pj.push_back((uint16_t)K); pl.push_back((uint16_t)K); cm.push_back((int32_t)(num_pairs(K, T) - 1));    // (y_0, y_0)
    gc.Pc = (int)cm.size();
    gram_col_tiling(gc.Pc, gc.nfull, gc.tail_q);
    gc.ntiles = gc.nfull + (gc.tail_q > 0);
    const size_t cols = (size_t)gc.ntiles * BN;
    gc.pairs.assign(cols * 2, (uint16_t)K);          // padding columns: harmless duplicates of (y_0, y_0), never stored
    gc.colmap.assign(cols, -1);
    for (size_t c = 0; c < cm.size(); ++c) { gc.pairs[2 * c] = pj[c]; gc.pairs[2 * c + 1] = pl[c]; gc.colmap[c] = cm[c]; }
    return gc;
}

// The outcome columns of gram_columns alone: (j, y_t) in the full table's order, then (y_0, y_0).  Every column's sum is
// the same as in the full launch: its DMMA sequence and leaf tree depend on (n_g, K) only, not on the tile it sits in.
GramColumns gram_outcome_columns(int K, int T) {
    GramColumns gc;
    std::vector<uint16_t> pj, pl; std::vector<int32_t> cm;
    for (int j = 0; j < K; ++j) {
        const int64_t base = pair_base(K, T, j);
        for (int o = 0; o < T; ++o) { pj.push_back((uint16_t)j); pl.push_back((uint16_t)(K + o)); cm.push_back((int32_t)(base + (K - j) + o)); }
    }
    pj.push_back((uint16_t)K); pl.push_back((uint16_t)K); cm.push_back((int32_t)(num_pairs(K, T) - 1));
    gc.Pc = (int)cm.size();
    gram_col_tiling(gc.Pc, gc.nfull, gc.tail_q);
    gc.ntiles = gc.nfull + (gc.tail_q > 0);
    const size_t cols = (size_t)gc.ntiles * BN;
    gc.pairs.assign(cols * 2, (uint16_t)K);
    gc.colmap.assign(cols, -1);
    for (size_t c = 0; c < cm.size(); ++c) { gc.pairs[2 * c] = pj[c]; gc.pairs[2 * c + 1] = pl[c]; gc.colmap[c] = cm[c]; }
    return gc;
}

std::vector<int32_t> gram_cache_map(int K, int T) {
    std::vector<int32_t> m;
    m.reserve((size_t)gram_cache_xx_cells(K) + gram_cache_y_cells(K, T));
    for (int j = 0; j < K; ++j)
        for (int l = j; l < K; ++l) m.push_back((int32_t)(pair_base(K, T, j) + (l - j)));
    for (int j = 0; j < K; ++j)
        for (int o = 0; o < T; ++o) m.push_back((int32_t)(pair_base(K, T, j) + (K - j) + o));
    m.push_back((int32_t)(num_pairs(K, T) - 1));
    return m;
}

// cell e of the copy -> (group, batch slot, cache cell c); TO_CACHE: batch Gram -> cache, else cache -> batch Gram
template <bool TO_CACHE>
__device__ __forceinline__ void gram_cache_copy_cells(const GramCacheCopy& a) {
    const long long ncell = a.c_hi - a.c_lo, per_g = a.nslots * ncell, total = 2 * per_g;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int g = e >= per_g ? 1 : 0;
        const long long r = e - (g ? per_g : 0);
        const long long s = r / ncell;
        const int c = a.c_lo + (int)(r - s * ncell);
        double* gcell = a.gram + ((size_t)g * a.slots_pad + (size_t)s) * (size_t)a.Pld + a.map[c];
        const size_t slot = (size_t)g * a.cslots + (size_t)(a.slot_lo + s);
        double* ccell = c < a.nx ? a.xx + slot * a.nx + c : a.yy + slot * a.ny + (c - a.nx);
        if (TO_CACHE) *ccell = *gcell; else *gcell = *ccell;
    }
}
__global__ void __launch_bounds__(256) gram_cache_extract_kernel(const GramCacheCopy a) { gram_cache_copy_cells<true>(a); }
__global__ void __launch_bounds__(256) gram_cache_assemble_kernel(const GramCacheCopy a) { gram_cache_copy_cells<false>(a); }

static void gram_cache_copy(const GramCacheCopy& a, bool to_cache, cudaStream_t st) {
    const long long total = 2 * a.nslots * (long long)(a.c_hi - a.c_lo);
    if (total <= 0) return;
    const unsigned blocks = (unsigned)std::min<long long>((total + 255) / 256, 148 * 8);
    if (to_cache) gram_cache_extract_kernel<<<blocks, 256, 0, st>>>(a);
    else gram_cache_assemble_kernel<<<blocks, 256, 0, st>>>(a);
    OB_CUDA(cudaGetLastError());
}
void gram_cache_extract_launch(const GramCacheCopy& a, cudaStream_t st) { gram_cache_copy(a, true, st); }
void gram_cache_assemble_launch(const GramCacheCopy& a, cudaStream_t st) { gram_cache_copy(a, false, st); }

GramPlan gram_make_plan(int K, int T, int ldx, int panels, const GroupData gd[2], int count_bytes, int num_sms,
                        const GramColumns& cols) {
    GramPlan pl;
    pl.K = K; pl.T = T; pl.ldx = ldx; pl.panels = panels;
    pl.nfull = cols.nfull; pl.tail_q = cols.tail_q; pl.ntiles = cols.ntiles;
    pl.Pld = gram_pld(K, T);
    int64_t total = 0;
    pl.leaf_span = gd[0].shard.leaf_span;
    for (int g = 0; g < 2; ++g) {
        pl.n_pad[g] = gd[g].n_pad;
        pl.segs[g] = gd[g].shard.leaf_hi - gd[g].shard.leaf_lo;     // leaves held here (fixed by the global row count)
        pl.seg_rows[g] = gd[g].shard.seg_rows;
        pl.units[g] = (int64_t)pl.segs[g] * panels * pl.ntiles;
        total += pl.units[g];
    }
    pl.grid = (int)std::min<int64_t>(num_sms, std::max<int64_t>(total, 1));
    pl.ring = gram_ws_smem(pl.ldx, count_bytes, WS_R) <= GRAM_SMEM_MAX ? WS_R : 2;
    pl.smem_bytes = gram_ws_smem(pl.ldx, count_bytes, pl.ring);
    pl.num_partials = (int64_t)total;
    return pl;
}

static GramKernelParams gram_params(const GramPlan& pl, const GramArgs& a, const int seg_lo[2], const int seg_n[2]) {
    GramKernelParams p;
    for (int g = 0; g < 2; ++g) {
        p.X[g] = a.X[g]; p.C[g] = a.C[g];
        p.n_pad[g] = pl.n_pad[g]; p.segs[g] = pl.segs[g]; p.seg_rows[g] = pl.seg_rows[g];
        p.seg_lo[g] = seg_lo ? seg_lo[g] : 0; p.seg_n[g] = seg_n ? seg_n[g] : pl.segs[g];
    }
    p.units0 = pl.units[0];
    p.units_total = pl.units[0] + pl.units[1];
    p.ldx = pl.ldx; p.panels = pl.panels; p.ntiles = pl.ntiles;
    p.nfull = pl.nfull; p.tail_q = pl.tail_q;
    p.partials = a.partials; p.pairs = a.d_pairs;
    p.tail_mi = a.tail_mi >= 1 && a.tail_mi <= 16 ? a.tail_mi : 16;
    return p;
}

// The contraction over the leaves [seg_lo[g], seg_lo[g] + seg_n[g]) of each group (null = all leaves held here):
// writes those leaves' partial tiles.  A design whose upload is still in flight is contracted in two such launches
// (the rows that have arrived, then the rest); the partial tiles, hence every sum, are the same as from one launch.
void gram_launch_leaves(const GramPlan& pl, const GramArgs& a, const int seg_lo[2], const int seg_n[2], cudaStream_t st) {
    const GramKernelParams p = gram_params(pl, a, seg_lo, seg_n);
    const int64_t units = ((int64_t)p.seg_n[0] + p.seg_n[1]) * pl.panels * pl.ntiles;
    if (units <= 0) return;
    const int grid = (int)std::min<int64_t>(pl.grid, units);
    const size_t ws_smem = pl.smem_bytes;
    if (!gram_fits(pl.ldx, a.count_bytes))
        throw StatusError{OB_ERR_UNSUPPORTED, "design too wide for the Gram kernel's shared-memory ring (K + outcomes <= 280 with "
                                              "8-bit multiplicities, <= 268 with 16-bit, <= 236 with fp32 Bayesian weights)"};
    auto launch_ws = [&](auto kernel) {
        OB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws_smem));
        kernel<<<grid, WS_THREADS, ws_smem, st>>>(p);
    };
    // row stride specialisations (ldx = 4 mod 8): the common design widths get immediate shared-memory offsets
#define OB_GRAM_WS_CASE(L) case L: if (a.count_bytes == 4) launch_ws(gram_ws_kernel<float, L, gram_ring_f32(L)>); \
                                   else if (a.count_bytes == 1) launch_ws(gram_ws_kernel<uint8_t, L>); else launch_ws(gram_ws_kernel<uint16_t, L>); break;
    switch (pl.ldx) {
        OB_GRAM_WS_CASE(12) OB_GRAM_WS_CASE(20) OB_GRAM_WS_CASE(28) OB_GRAM_WS_CASE(36) OB_GRAM_WS_CASE(44) OB_GRAM_WS_CASE(52)
        OB_GRAM_WS_CASE(60) OB_GRAM_WS_CASE(68) OB_GRAM_WS_CASE(76) OB_GRAM_WS_CASE(84) OB_GRAM_WS_CASE(92)
        default:      // wider designs: run-time row stride; two ring stages when three do not fit
            if (a.count_bytes == 4) { if (pl.ring == WS_R) launch_ws(gram_ws_kernel<float, 0, WS_R>); else launch_ws(gram_ws_kernel<float, 0, 2>); }
            else if (pl.ring == WS_R) { if (a.count_bytes == 1) launch_ws(gram_ws_kernel<uint8_t, 0, WS_R>); else launch_ws(gram_ws_kernel<uint16_t, 0, WS_R>); }
            else { if (a.count_bytes == 1) launch_ws(gram_ws_kernel<uint8_t, 0, 2>); else launch_ws(gram_ws_kernel<uint16_t, 0, 2>); }
    }
#undef OB_GRAM_WS_CASE
    OB_CUDA(cudaGetLastError());
}

// fixed-tree sum of every tile's leaf partials -> gram [2][panels*BM][Pld]
void gram_reduce_launch(const GramPlan& pl, const GramArgs& a, cudaStream_t st) {
    // cells the contraction does not compute (structural zeros, row padding up to Pld) are 0.0
    OB_CUDA(cudaMemsetAsync(a.gram, 0, sizeof(double) * 2 * (size_t)pl.panels * BM * (size_t)pl.Pld, st));
    dim3 rgw(2 * pl.panels * pl.ntiles, 16);
    gram_reduce_kernel<<<rgw, 256, 0, st>>>(a.partials, pl.segs[0], pl.segs[1], a.gram, pl.panels, pl.ntiles, pl.leaf_span,
                                            pl.Pld, pl.tail_q, a.d_colmap);
    OB_CUDA(cudaGetLastError());
}

void gram_launch(const GramPlan& pl, const GramArgs& a, cudaStream_t st, cudaEvent_t ev_main_begin, cudaEvent_t ev_main_end) {
    if (ev_main_begin) OB_CUDA(cudaEventRecord(ev_main_begin, st));
    gram_launch_leaves(pl, a, nullptr, nullptr, st);
    if (ev_main_end) OB_CUDA(cudaEventRecord(ev_main_end, st));
    gram_reduce_launch(pl, a, st);
}

void leaf_sum_launch(const double* part, const int segs[2], int64_t slots_pad, int span, double* out, cudaStream_t st) {
    const long long half = slots_pad / 2;
    const unsigned blocks = (unsigned)std::min<long long>((2 * half + 255) / 256, 148 * 8);
    leaf_sum_kernel<<<std::max(blocks, 1u), 256, 0, st>>>(part, segs[0], segs[1], half, span, out);
    OB_CUDA(cudaGetLastError());
}

void gram_combine_launch(const double* gathered, int world, const int ranks_with_rows[2], int64_t per_group_elems,
                         double* gram, cudaStream_t st) {
    const long long per2 = per_group_elems / 2;
    const unsigned blocks = (unsigned)std::min<long long>((2 * per2 + 255) / 256, 148 * 8);
    gram_combine_kernel<<<std::max(blocks, 1u), 256, 0, st>>>(gathered, world, ranks_with_rows[0], ranks_with_rows[1], per2, gram);
    OB_CUDA(cudaGetLastError());
}

// Host-side walk of the warp-specialised kernel's unit schedule (no device needed): for every CTA the units it takes,
// as (group, panel, tile, segment, stages, mi, tail quanta: 0 = a full tile).  Lets the CPU tests check that every unit is covered exactly once
// and that CTAs get equal shares of every cost class, for any shape.
int64_t gram_schedule_debug(int K, int panels, int64_t slots_last_panel, const GroupData gd[2], int grid, int64_t* out7, int64_t cap) {
    const GramColumns cols = gram_columns(K, 1, K - 1, std::vector<int>());
    GramPlan pl = gram_make_plan(K, 1, design_ldx(K + 1), panels, gd, 1, grid, cols);
    GramKernelParams p{};
    for (int g = 0; g < 2; ++g) { p.n_pad[g] = pl.n_pad[g]; p.segs[g] = pl.segs[g]; p.seg_rows[g] = pl.seg_rows[g]; p.seg_lo[g] = 0; p.seg_n[g] = pl.segs[g]; }
    p.units0 = pl.units[0]; p.units_total = pl.units[0] + pl.units[1];
    p.ldx = pl.ldx; p.panels = pl.panels; p.ntiles = pl.ntiles; p.nfull = pl.nfull; p.tail_q = pl.tail_q;
    p.tail_mi = (int)std::min<int64_t>(16, ((slots_last_panel + 7) / 8 + 3) / 4 * 4);
    p.partials = nullptr;
    int64_t count = 0;
    for (int b = 0; b < grid; ++b) {
        GramUnit u;
        for (long long i = b; ws_decode(p, i, pl.ldx, 1, u); i += grid) {
            if (count < cap) {
                // recover (g, panel, nt, seg) from the partial-tile index the unit writes to
                const long long idx = (long long)(u.out - (double*)nullptr) / (BM * BN);
                const int g = idx >= p.units0 ? 1 : 0;
                const long long r = idx - (g ? p.units0 : 0);
                const int segs = p.segs[g];
                const long long sweep = r / p.ntiles;
                int64_t* o = out7 + 8 * count;
                o[0] = b; o[1] = g; o[2] = sweep / segs; o[3] = r % p.ntiles; o[4] = sweep % segs; o[5] = u.nstages; o[6] = u.mi; o[7] = u.tq < 4 ? u.tq : 0;
            }
            ++count;
        }
    }
    return count;
}

}  // namespace ob
