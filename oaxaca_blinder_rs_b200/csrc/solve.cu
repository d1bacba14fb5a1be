// csrc/solve.cu -- per-replicate (W)LS solves + decomposition epilogue, one CTA per replicate slot.
//
// Input: the replicate's sufficient statistics from gram.cu (upper triangle of [x|y][x|y]^T sums).
// Restates, per slot:
//   ols()                    ols.rs:96-115   n_obs <= k guard, Cholesky (nalgebra column algorithm:
//                                            pivot <= 0 or NaN -> failure), solve
//   column means             estimation.rs:56-71  = G[0][j] / G[0][0] (intercept column carries the sums)
//   Yun normalisation        normalization.rs:5-51
//   beta* selection          builder.rs:538-621 (GroupA / GroupB / Pooled with indicator at 1+n_cont / Cotton)
//   two/three-fold, detailed decomposition.rs:56-122
//   Yun base-category rows   builder.rs:634-674 (three_fold stays uncorrected)
//   total gap                builder.rs:676-684
// A failing replicate gets a status code and NaN statistics; the host drops it (builder.rs:831-837).
#include "common.cuh"
#include "internal.h"

#include <cmath>

namespace ob {

constexpr int SOLVE_THREADS = 128;

struct SolveParams {
    const double* gram; long long slots_pad; int Pld; long long slots;
    int K, n_cont, ref_kind, T;
    int n_norm; const int* norm_m; const int* norm_off; const int* norm_idx; const int* norm_has_base;
    int n_base, S, weighted;
    double na, nb;
    const long long* rows;   // [2][slots_pad] per-slot group row counts (clustered designs), null: na / nb
    const double* esum;      // [2][slots_pad] per-slot sums of the raw Bayesian weights E, null: multiplicities
    double* stats; int* status; double* beta_a; double* beta_b; double* point_extra;
    double* gscratch;        // per-slot matrix buffer in global memory when it does not fit shared memory, else null
};

__device__ __forceinline__ int ld_of(int N) { return N | 1; }  // odd stride: conflict-free column walks

// In-place Cholesky of the N x N matrix (lower triangle used), nalgebra semantics. Returns false on failure.
__device__ bool chol_factor(double* G, int N, int ld, int* fail) {
    for (int j = 0; j < N; ++j) {
        // col_j(i >= j) -= sum_{k<j} L[i][k] L[j][k], k ascending (axpy order of nalgebra)
        for (int i = j + threadIdx.x; i < N; i += blockDim.x) {
            double s = G[i * ld + j];
            const double* Li = G + i * ld;
            const double* Lj = G + j * ld;
            for (int k = 0; k < j; ++k) s -= Li[k] * Lj[k];
            G[i * ld + j] = s;
        }
        __syncthreads();
        const double d = G[j * ld + j];
        if (!(d > 0.0)) {
            if (threadIdx.x == 0) *fail = 1;
            __syncthreads();
            return false;
        }
        const double r = sqrt(d);
        __syncthreads();
        for (int i = j + threadIdx.x; i < N; i += blockDim.x) G[i * ld + j] = (i == j) ? r : G[i * ld + j] / r;
        __syncthreads();
    }
    return true;
}

// L L^T x = b in place, by warp 0 (lane-parallel dot products).
__device__ void chol_solve(const double* L, int N, int ld, double* b) {
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        for (int i = 0; i < N; ++i) {
            double s = 0.0;
            for (int k = lane; k < i; k += 32) s += L[i * ld + k] * b[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) b[i] = (b[i] - s) / L[i * ld + i];
            __syncwarp();
        }
        for (int i = N - 1; i >= 0; --i) {
            double s = 0.0;
            for (int k = i + 1 + lane; k < N; k += 32) s += L[k * ld + i] * b[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) b[i] = (b[i] - s) / L[i * ld + i];
            __syncwarp();
        }
    }
    __syncthreads();
}

__device__ void yun_shift(const SolveParams& p, double* beta, int shift_from, double* base) {
    for (int v = 0; v < p.n_norm; ++v) {  // normalization.rs:13-49
        base[v] = 0.0;
        const int a = p.norm_off[v], b = p.norm_off[v + 1];
        if (a == b) continue;
        double sum = 0.0;
        for (int t = a; t < b; ++t) {
            int i = p.norm_idx[t];
            if (shift_from >= 0 && i >= shift_from) ++i;
            sum += beta[i];
        }
        const int m = p.norm_m[v];
        if (m == 0) continue;
        const double mu = sum / (double)m;
        base[v] = -mu;
        beta[0] += mu;
        for (int t = a; t < b; ++t) {
            int i = p.norm_idx[t];
            if (shift_from >= 0 && i >= shift_from) ++i;
            beta[i] -= mu;
        }
    }
}

// index of pair (i,j), i <= j < K, among the packed Gram columns (internal.h: pair_base)
__device__ __forceinline__ long long gidx(int K, int T, int i, int j) {
    return (long long)i * (K + T) - (long long)i * (i - 1) / 2 + (j - i);
}
__device__ __forceinline__ double gsym(const double* g, int K, int T, int i, int j) { return i <= j ? g[gidx(K, T, i, j)] : g[gidx(K, T, j, i)]; }

// One system at a time in the matrix buffer M -- group A, group B, then (Pooled) the stacked system with the group
// indicator -- so that the buffer is a single (K+1) x (K+1) matrix: shared memory up to K+1 = 164, a per-slot global
// scratch beyond (p.gscratch).  Each factor is used for all T right-hand sides before the buffer is reused.
__global__ void __launch_bounds__(SOLVE_THREADS) solve_kernel(const SolveParams p) {
    extern __shared__ __align__(16) double sm[];
    const int K = p.K, T = p.T, Kp = K + 1;
    const int ld = ld_of(K), ldp = ld_of(Kp);
    const long long slot = blockIdx.x;
    const int tid = threadIdx.x;
    const bool pooled = p.ref_kind == OB_REF_POOLED;
    const int msize = pooled ? Kp * ldp : K * ld;

    double* vec = sm;
    double* M = p.gscratch ? p.gscratch + (size_t)slot * msize : sm;
    if (!p.gscratch) vec = sm + msize;
    double* xa = vec;            double* xb = xa + Kp;
    double* bs = xb + Kp;        double* rawA = bs + Kp; double* rawB = rawA + Kp;
    double* baseA = rawB + Kp;   double* baseB = baseA + p.n_norm + 1; double* baseS = baseB + p.n_norm + 1;
    double* BA = baseS + p.n_norm + 1;     // [T][Kp] solutions of group A
    double* BB = BA + (size_t)T * Kp;      // [T][Kp]
    double* BP = BB + (size_t)T * Kp;      // [T][Kp] pooled (only when pooled)
    __shared__ int fail;
    __shared__ double sums[4];   // sum(cw) per group and, per outcome, sum(cwy)

    const double* gA = p.gram + (size_t)slot * p.Pld;
    const double* gB = p.gram + ((size_t)p.slots_pad + slot) * p.Pld;
    if (tid == 0) { fail = 0; sums[0] = gA[0]; sums[2] = gB[0]; }
    for (int j = tid; j < K; j += blockDim.x) {  // estimation.rs:56-71: the intercept row of the Gram carries the column sums
        xa[j] = gA[j] / gA[0];
        xb[j] = gB[j] / gB[0];
    }
    int status = OB_OK;
    // ols.rs:96-105: n_obs (row count, not sum of weights) must exceed k; group A is fitted first
    double na = p.na, nb = p.nb;
    if (p.rows) {
        // a clustered replicate: its own group sizes, checked in the reference's order -- an empty group first
        // (builder.rs:431-435), then group A's fit, group B's n-guard at its own fit (sys == 1 below)
        na = (double)p.rows[slot]; nb = (double)p.rows[p.slots_pad + slot];
        if (na == 0.0 || nb == 0.0) status = OB_ERR_INVALID_GROUP;
        else if (na <= (double)K) status = OB_ERR_INSUFFICIENT_DATA;
    } else if (na <= (double)K || nb <= (double)K) status = OB_ERR_INSUFFICIENT_DATA;
    const int ind = 1 + p.n_cont;       // builder.rs:548-566: position of the group indicator in the pooled design
    // Bayesian bootstrap: the Gram holds sums over raw weights E; the replicate's weights are pi = n_g E / sum_g E.  beta
    // and the means of one group do not change when its weights scale by a common factor; where the groups meet (the
    // stacked Pooled system, the weighted Cotton / Weighted omega) each group's cells are scaled by s_g = n_g / sum_g E.
    double sA = 1.0, sB = 1.0;
    if (p.esum) { sA = na / p.esum[slot]; sB = nb / p.esum[p.slots_pad + slot]; }

    for (int sys = 0; sys < (pooled ? 3 : 2); ++sys) {
        const int N = sys == 2 ? Kp : K, ldm = sys == 2 ? ldp : ld;
        double* B = sys == 0 ? BA : (sys == 1 ? BB : BP);
        const double* g = sys == 1 ? gB : gA;
        __syncthreads();
        if (sys == 1 && p.rows && nb <= (double)K) status = OB_ERR_INSUFFICIENT_DATA;
        if (status != OB_OK) break;
        if (sys < 2) {
            // unpack X'WX of the group from the packed columns
            for (int i = 0; i < K; ++i) {
                const long long base_idx = gidx(K, T, i, i) - i;
                for (int l = i + tid; l < K; l += blockDim.x) {
                    const double v = g[base_idx + l];
                    M[i * ldm + l] = v; M[l * ldm + i] = v;
                }
            }
            for (int e = tid; e < T * K; e += blockDim.x) {  // X'Wy of outcome t: pair (j, y_t) at pair_base(j) + (K - j) + t
                const int t = e / K, j = e - t * K;
                B[t * Kp + j] = g[gidx(K, T, j, j) + (K - j) + t];
            }
        } else {
            if (na + nb <= (double)Kp) { status = OB_ERR_INSUFFICIENT_DATA; break; }
            // rows of A and B stacked, indicator (1 on A rows) at column ind
            for (int e = tid; e < Kp * Kp; e += blockDim.x) {
                const int i = e / Kp, j = e - i * Kp;
                const int si = i < ind ? i : i - 1, sj = j < ind ? j : j - 1;  // source design columns
                double v;
                if (i == ind && j == ind) v = gA[0];
                else if (i == ind) v = gA[sj];        // sum over A rows of w * 1 * x_sj
                else if (j == ind) v = gA[si];
                else v = p.esum ? sA * gsym(gA, K, T, si, sj) + sB * gsym(gB, K, T, si, sj) : gsym(gA, K, T, si, sj) + gsym(gB, K, T, si, sj);
                if (p.esum && (i == ind || j == ind)) v *= sA;
                M[i * ldm + j] = v;
            }
            for (int e = tid; e < T * Kp; e += blockDim.x) {
                const int t = e / Kp, i = e - t * Kp;
                const int si = i < ind ? i : i - 1;
                const long long ya = gidx(K, T, 0, 0) + K + t;             // (0, y_t): sum over A rows of w y_t
                const double a = gA[gidx(K, T, si, si) + (K - si) + t], b = gB[gidx(K, T, si, si) + (K - si) + t];
                if (p.esum) B[e] = (i == ind) ? sA * gA[ya] : sA * a + sB * b;
                else B[e] = (i == ind) ? gA[ya] : a + b;
            }
        }
        __syncthreads();
        if (!chol_factor(M, N, ldm, &fail)) { status = OB_ERR_NALGEBRA; break; }
        for (int t = 0; t < T; ++t) chol_solve(M, N, ldm, B + (size_t)t * Kp);
    }
    __syncthreads();

    const int D = K + p.n_base;
    for (int t = 0; t < T; ++t) {
        double* out = p.stats + ((size_t)slot * T + t) * p.S;
        const size_t brow = ((size_t)slot * T + t) * K;
        // ---- scalar epilogue ----
        int st_t = status;
        if (tid == 0 && st_t == OB_OK) {
            double* ba = BA + (size_t)t * Kp; double* bb = BB + (size_t)t * Kp; double* rP = BP + (size_t)t * Kp;
            sums[1] = gA[K + t]; sums[3] = gB[K + t];                      // pair (0, y_t)
            for (int j = 0; j < K; ++j) { rawA[j] = ba[j]; rawB[j] = bb[j]; }
            if (p.n_norm > 0) { yun_shift(p, ba, -1, baseA); yun_shift(p, bb, -1, baseB); }   // estimation.rs:76-91
            switch (p.ref_kind) {  // builder.rs:538-621
            case OB_REF_GROUP_A:
                for (int j = 0; j < K; ++j) bs[j] = ba[j];
                for (int v = 0; v < p.n_norm; ++v) baseS[v] = baseA[v];
                break;
            case OB_REF_GROUP_B:
                for (int j = 0; j < K; ++j) bs[j] = bb[j];
                for (int v = 0; v < p.n_norm; ++v) baseS[v] = baseB[v];
                break;
            case OB_REF_POOLED: {
                if (p.n_norm > 0) yun_shift(p, rP, ind, baseS);           // builder.rs:568-579
                for (int j = 0; j < ind; ++j) bs[j] = rP[j];              // remove_row(ind) :580-589
                for (int j = ind; j < K; ++j) bs[j] = rP[j + 1];
                break;
            }
            default: {  // Weighted | Cotton: builder.rs:591-620
                const double n_a = p.weighted ? (p.esum ? sA * sums[0] : sums[0]) : na;
                const double n_b = p.weighted ? (p.esum ? sB * sums[2] : sums[2]) : nb;
                const double total = n_a + n_b;
                if (total == 0.0) { st_t = OB_ERR_INVALID_GROUP; break; }
                const double wA = n_a / total, wB = 1.0 - wA;
                for (int v = 0; v < p.n_norm; ++v) baseS[v] = baseA[v] * wA + baseB[v] * wB;
                for (int j = 0; j < K; ++j) bs[j] = ba[j] * wA + bb[j] * wB;
                break;
            }
            }
            if (st_t == OB_OK) {
                // decomposition.rs:56-89
                double en = 0.0, co = 0.0, in = 0.0, ex = 0.0, fa = 0.0, fb = 0.0;
                for (int j = 0; j < K; ++j) {
                    const double dx = xa[j] - xb[j], db = ba[j] - bb[j];
                    en += dx * bb[j]; co += xb[j] * db; in += dx * db;
                    ex += dx * bs[j]; fa += xa[j] * ba[j]; fb += xb[j] * bb[j];
                }
                double two0 = ex, two1 = (fa - fb) - ex;
                for (int j = 0; j < K; ++j) {  // decomposition.rs:92-122
                    out[5 + j] = (xa[j] - xb[j]) * bs[j];
                    out[5 + D + j] = xa[j] * (ba[j] - bs[j]) + xb[j] * (bs[j] - bb[j]);
                }
                int row = K;
                for (int v = 0; v < p.n_norm; ++v) {  // builder.rs:634-674
                    if (!p.norm_has_base[v]) continue;
                    double sa = 0.0, sb = 0.0;
                    for (int q = p.norm_off[v]; q < p.norm_off[v + 1]; ++q) { sa += xa[p.norm_idx[q]]; sb += xb[p.norm_idx[q]]; }
                    const double xab = 1.0 - sa, xbb = 1.0 - sb;
                    const double un = xab * (baseA[v] - baseS[v]) + xbb * (baseS[v] - baseB[v]);
                    const double e2 = (xab - xbb) * baseS[v];
                    out[5 + D + row] = un; out[5 + row] = e2;
                    two0 += e2; two1 += un;
                    ++row;
                }
                out[0] = two0; out[1] = two1; out[2] = en; out[3] = co; out[4] = in;
                if (p.beta_a) for (int j = 0; j < K; ++j) p.beta_a[brow + j] = ba[j];
                if (p.beta_b) for (int j = 0; j < K; ++j) p.beta_b[brow + j] = bb[j];
                if (p.point_extra && slot == 0) {
                    double* pe = p.point_extra + (size_t)t * (5 * K + 1);
                    for (int j = 0; j < K; ++j) {
                        pe[j] = xa[j]; pe[K + j] = xb[j]; pe[2 * K + j] = bs[j];
                        pe[3 * K + j] = rawA[j]; pe[4 * K + j] = rawB[j];
                    }
                    pe[5 * K] = sums[1] / sums[0] - sums[3] / sums[2];    // builder.rs:676-684
                }
            }
        }
        if (tid == 0) {
            if (st_t != OB_OK) {
                const double nan = __longlong_as_double(0x7ff8000000000000LL);
                for (int j = 0; j < p.S; ++j) out[j] = nan;
                if (p.beta_a) for (int j = 0; j < K; ++j) p.beta_a[brow + j] = nan;
                if (p.beta_b) for (int j = 0; j < K; ++j) p.beta_b[brow + j] = nan;
            }
            if (t == 0 || st_t != OB_OK) p.status[slot] = st_t;     // one status per slot (the fits fail or succeed together)
        }
    }
}

// shared memory of one solve CTA: the vectors always, the matrix buffer while it fits (else per-slot global scratch)
static size_t solve_vec_doubles(int K, int n_norm, int T) { return (size_t)5 * (K + 1) + (size_t)3 * (n_norm + 1) + (size_t)3 * T * (K + 1); }
static size_t solve_mat_doubles(int K, bool pooled) { const int Kp = K + 1; return pooled ? (size_t)Kp * (Kp | 1) : (size_t)K * (K | 1); }
constexpr size_t SOLVE_SMEM_MAX = 227 * 1024;

size_t solve_smem_bytes(int K, bool pooled, int n_norm) {
    return (solve_vec_doubles(K, n_norm, 1) + solve_mat_doubles(K, pooled)) * sizeof(double);
}

size_t solve_scratch_bytes(int K, bool pooled, int n_norm, int T, int64_t slots) {
    const size_t in_smem = (solve_vec_doubles(K, n_norm, T) + solve_mat_doubles(K, pooled)) * sizeof(double);
    return in_smem <= SOLVE_SMEM_MAX ? 0 : sizeof(double) * solve_mat_doubles(K, pooled) * (size_t)slots;
}

void solve_launch(const SolveArgs& a, cudaStream_t st) {
    SolveParams p;
    p.gram = a.gram; p.slots_pad = a.slots_pad; p.Pld = a.Pld; p.slots = a.slots;
    p.K = a.K; p.n_cont = a.n_cont; p.ref_kind = a.ref_kind; p.T = a.T;
    p.n_norm = a.n_norm; p.norm_m = a.d_norm_m; p.norm_off = a.d_norm_off; p.norm_idx = a.d_norm_idx;
    p.norm_has_base = a.d_norm_has_base; p.n_base = a.n_base; p.S = a.S; p.weighted = a.weighted;
    p.na = a.na; p.nb = a.nb; p.rows = a.rows; p.esum = a.esum;
    p.stats = a.stats; p.status = a.status; p.beta_a = a.beta_a; p.beta_b = a.beta_b; p.point_extra = a.point_extra;
    const bool pooled = a.ref_kind == OB_REF_POOLED;
    const bool global = solve_scratch_bytes(a.K, pooled, a.n_norm, a.T, 1) != 0;
    if (global && !a.scratch) throw StatusError{OB_ERR_INVALID_ARG, "solve scratch missing for a design this wide"};
    p.gscratch = global ? a.scratch : nullptr;
    const size_t smem = (solve_vec_doubles(a.K, a.n_norm, a.T) + (global ? 0 : solve_mat_doubles(a.K, pooled))) * sizeof(double);
    if (smem > SOLVE_SMEM_MAX) throw StatusError{OB_ERR_UNSUPPORTED, "design too wide for the solve kernel"};
    OB_CUDA(cudaFuncSetAttribute(solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    solve_kernel<<<(unsigned)a.slots, SOLVE_THREADS, smem, st>>>(p);
    OB_CUDA(cudaGetLastError());
}

}  // namespace ob
