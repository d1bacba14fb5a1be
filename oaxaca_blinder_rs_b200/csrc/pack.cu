// csrc/pack.cu -- design-matrix pack: frame columns -> per-group row-major designs in HBM.
//
// Done ONCE per dataset, replacing what the reference redoes for every replicate: split_groups
// (builder.rs:61-102: string unique/sort/equal/filter), prepare_data (builder.rs:294-378: intercept,
// predictor select, dummy columns, three n x K copies) and the sqrt(w) scaling copy (ols.rs:68-78).
//
//   X_g[r][:] = [1 | continuous.. | dummies.. | outcome | 0-pad]      r = rank of the row inside group g
// Row order inside a group is frame order (stable), as df.filter() gives (builder.rs:85-94), so
// row positions agree with the oracle's and with an external resample index stream.
// Dummy for code c >= 1 of categorical q: design column dummy_start[q] + c - 1 (builder.rs:402-409).
//
// HBM-bound: reads 8 B x (n_cont + 2) + 4 B x n_cat + 1 B per row, writes 8 B x ldx per row.
// Three launches: per-block group counts -> single-block exclusive scan -> staged transpose/scatter.
#include "common.cuh"
#include "internal.h"

#include <algorithm>

namespace ob {

constexpr int PK_ROWS = 128;   // rows per block
constexpr int PK_THREADS = 256;

__global__ void __launch_bounds__(PK_THREADS) pack_count_kernel(const uint8_t* __restrict__ group,
                                                                const double* __restrict__ w, long long n,
                                                                long long* __restrict__ block_counts,
                                                                int* __restrict__ flags) {
    __shared__ int ca, cb;
    if (threadIdx.x == 0) { ca = 0; cb = 0; }
    __syncthreads();
    const long long row0 = (long long)blockIdx.x * PK_ROWS;
    int a = 0, b = 0;
    for (int t = threadIdx.x; t < PK_ROWS; t += PK_THREADS) {
        const long long i = row0 + t;
        if (i < n) {
            const uint8_t g = group[i];
            a += g == 0; b += g == 1;
            if (w && g <= 1 && w[i] < 0.0) atomicOr(&flags[0], 1);   // ols.rs:60-66
        }
    }
    if (a) atomicAdd(&ca, a);
    if (b) atomicAdd(&cb, b);
    __syncthreads();
    if (threadIdx.x == 0) { block_counts[2 * blockIdx.x] = ca; block_counts[2 * blockIdx.x + 1] = cb; }
}

// exclusive scan of block_counts [nblocks][2] in place; totals[2] receives the group sizes
__global__ void __launch_bounds__(1024) pack_scan_kernel(long long* __restrict__ bc, int nblocks, long long* totals) {
    __shared__ long long part[2][1024];
    const int t = threadIdx.x;
    const int per = (nblocks + 1023) / 1024;
    const int lo = t * per, hi = min(lo + per, nblocks);
    long long sa = 0, sb = 0;
    for (int i = lo; i < hi; ++i) { sa += bc[2 * i]; sb += bc[2 * i + 1]; }
    part[0][t] = sa; part[1][t] = sb;
    __syncthreads();
    if (t < 2) {  // 1024-element serial scan per group: negligible
        long long run = 0;
        for (int i = 0; i < 1024; ++i) { const long long v = part[t][i]; part[t][i] = run; run += v; }
        totals[t] = run;
    }
    __syncthreads();
    long long ra = part[0][t], rb = part[1][t];
    for (int i = lo; i < hi; ++i) {
        const long long va = bc[2 * i], vb = bc[2 * i + 1];
        bc[2 * i] = ra; bc[2 * i + 1] = rb;
        ra += va; rb += vb;
    }
}

struct PackKernelParams {
    long long n; int n_cont, n_cat, K, ldx;
    const double* const* cont; const int32_t* const* cat; const int32_t* cat_levels; const int32_t* dummy_start;
    const double* y; const double* w; const uint8_t* group;
    const long long* block_base;   // [nblocks][2] exclusive scan
    int blk0;                      // first block of this launch (chunked pack: ob_design_pack_async)
    double* XA; double* XB; double* wA; double* wB;
    double* XsA; double* XsB;      // sqrt(w)-scaled copies (weighted designs) or nullptr
    uint32_t* srcA; uint32_t* srcB;
    int* flags;
    // row-shard window (ob_design_pack_row_shard_async; identity for an ordinary pack): a row of group g with rank q inside
    // the packed frame slice belongs at shard row q + shift[g]; rows falling outside [0, n_local[g]) are another rank's and
    // go to the export buffers instead (low side first, then high side), to be exchanged over the communicator
    long long shift[2], n_local[2], lo_add[2], hi_base[2];
    double* EX[2]; double* Ew[2]; uint32_t* Esrc[2];
    uint32_t src_add;              // frame row of the slice's first row
    int tile_cols;                 // design columns staged per pass (all V unless [PK_ROWS][V | 1] exceeds shared memory)
};

__global__ void __launch_bounds__(PK_THREADS) pack_scatter_kernel(const PackKernelParams p) {
    extern __shared__ __align__(16) double tile[];      // [PK_ROWS][tile_cols | 1] (odd stride: conflict-free column writes)
    __shared__ int lrank[PK_ROWS];                      // local rank within the row's group, -1 = ignored row
    __shared__ uint8_t lgrp[PK_ROWS];
    __shared__ int srcA[PK_ROWS], srcB[PK_ROWS];
    __shared__ int cnt[2];
    __shared__ const double* scont[288];                // column base pointers: no dependent global load per element
    const int V = p.K + 1, ts = V | 1;
    const int blk = blockIdx.x + p.blk0;
    const long long row0 = (long long)blk * PK_ROWS;
    const int rows = (int)min((long long)PK_ROWS, p.n - row0);
    const int tid = threadIdx.x;

    // stable local ranks: warp 0..3 each own 32 rows; ballot + prefix over warps
    __shared__ int wcount[4][2];
    if (tid < PK_ROWS) {
        const int g = (tid < rows) ? p.group[row0 + tid] : 255;
        lgrp[tid] = (uint8_t)g;
        const unsigned ma = __ballot_sync(0xffffffffu, g == 0), mb = __ballot_sync(0xffffffffu, g == 1);
        const unsigned below = (1u << (tid & 31)) - 1u;
        lrank[tid] = g == 0 ? __popc(ma & below) : (g == 1 ? __popc(mb & below) : -1);
        if ((tid & 31) == 0) { wcount[tid >> 5][0] = __popc(ma); wcount[tid >> 5][1] = __popc(mb); }
    } else {
        for (int c = tid - PK_ROWS; c < p.n_cont; c += PK_THREADS - PK_ROWS) scont[c] = p.cont[c];
    }
    __syncthreads();
    if (tid < PK_ROWS && lrank[tid] >= 0) {
        const int g = lgrp[tid];
        int off = 0;
        for (int wv = 0; wv < (tid >> 5); ++wv) off += wcount[wv][g];
        const int r = lrank[tid] + off;
        lrank[tid] = r;
        (g == 0 ? srcA : srcB)[r] = tid;
    }
    if (tid == 0) {
        cnt[0] = wcount[0][0] + wcount[1][0] + wcount[2][0] + wcount[3][0];
        cnt[1] = wcount[0][1] + wcount[1][1] + wcount[2][1] + wcount[3][1];
    }
    const long long baseA = p.block_base[2 * blk], baseB = p.block_base[2 * blk + 1];
    const int warp = tid >> 5, lane = tid & 31;
    // design columns [c0, c1) per pass: all V in one pass unless the tile would not fit in shared memory (wide designs)
    for (int c0 = 0; c0 < V; c0 += p.tile_cols) {
        const int c1 = min(V, c0 + p.tile_cols), ts = (c1 - c0) | 1;
        const bool last = c1 == V;
        if (c0 > 0) __syncthreads();          // every warp has written out the previous pass's tile
        // ---- stage the block's rows: column-wise coalesced reads -> tile[row][col - c0] ----
        // continuous predictors (design columns 1 .. n_cont, the bulk of the bytes): 4 independent loads in flight per thread
        {
            const int q0 = max(c0 - 1, 0), q1 = min(c1 - 1, p.n_cont);
            const int lim = (q1 > q0 ? q1 - q0 : 0) * PK_ROWS;
            for (int base = tid; base < lim; base += PK_THREADS * 4) {
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int e = base + u * PK_THREADS;
                    const int c = q0 + e / PK_ROWS, t = e % PK_ROWS;
                    v[u] = (e < lim && t < rows) ? scont[c][row0 + t] : 0.0;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int e = base + u * PK_THREADS;
                    if (e < lim) { const int c = q0 + e / PK_ROWS, t = e % PK_ROWS; tile[t * ts + 1 + c - c0] = v[u]; }
                }
            }
        }
        // intercept, outcome, dummies
        for (int t = tid; t < PK_ROWS; t += PK_THREADS) {
            if (c0 == 0) tile[t * ts] = t < rows ? 1.0 : 0.0;                   // __ob_intercept__ (builder.rs:330)
            if (last) tile[t * ts + p.K - c0] = t < rows ? p.y[row0 + t] : 0.0;
        }
        for (int e = tid; e < p.n_cat * PK_ROWS; e += PK_THREADS) {
            const int q = e / PK_ROWS, t = e - q * PK_ROWS;
            const int levels = p.cat_levels[q], start = p.dummy_start[q];
            // no dummy of q in this pass (a one-level categorical has none: its codes are checked in the last pass)
            if (!(last && levels <= 1) && (start + levels - 1 <= c0 || start >= c1)) continue;
            int code = 0;
            if (t < rows) {
                code = p.cat[q][row0 + t];
                if (code < 0 || code >= levels) { atomicOr(&p.flags[1], 1); code = 0; }
            }
            for (int lv = 1; lv < levels; ++lv) {                             // builder.rs:402-409: level lv -> column start + lv - 1
                const int c = start + lv - 1;
                if (c >= c0 && c < c1) tile[t * ts + c - c0] = (t < rows && code == lv) ? 1.0 : 0.0;
            }
        }
        __syncthreads();
        // ---- write out: one warp per packed row, lanes over the pass's contiguous columns; the sqrt(w)-scaled copy
        //      (ols.rs:68-78) is written in the same pass ----
        const int cend = last ? p.ldx : c1;                                    // pad columns [V, ldx) are written as zeros
        for (int g = 0; g < 2; ++g) {
            double* X = g ? p.XB : p.XA;
            double* Xs = g ? p.XsB : p.XsA;
            double* W = g ? p.wB : p.wA;
            uint32_t* SRC = g ? p.srcB : p.srcA;
            const int* src = g ? srcB : srcA;
            const long long base = g ? baseB : baseA;
            for (int r = warp; r < cnt[g]; r += PK_THREADS / 32) {
                const int t = src[r];
                const double wv = p.w ? p.w[row0 + t] : 1.0;
                if (last && wv < 0.0 && lane == 0) atomicOr(&p.flags[0], 1);   // ols.rs:60-66 (the chunked pack has no earlier look at w)
                const double sw = sqrt(wv);
                long long pos = base + r + p.shift[g];
                const bool mine = pos >= 0 && pos < p.n_local[g];
                double* xdst = X; double* xsdst = Xs; double* wdst = W; uint32_t* sdst = SRC;
                if (!mine) {      // another rank's row: export buffer, no scaled copy (the receiver scales what it imports)
                    pos = pos < 0 ? pos + p.lo_add[g] : p.hi_base[g] + (pos - p.n_local[g]);
                    xdst = p.EX[g]; xsdst = nullptr; wdst = p.Ew[g]; sdst = p.Esrc[g];
                }
                double* xr = xdst + pos * p.ldx;
                for (int c = c0 + lane; c < cend; c += 32) {
                    const double v = c < V ? tile[t * ts + c - c0] : 0.0;
                    xr[c] = v;
                    if (xsdst) xsdst[pos * p.ldx + c] = sw * v;
                }
                if (last && lane == 0) {
                    if (p.w) wdst[pos] = wv;
                    sdst[pos] = p.src_add + (uint32_t)(row0 + t);      // frame row of the packed row (ob_design_update_outcome)
                }
            }
        }
    }
}

int pack_num_blocks(int64_t n) { return (int)((n + PK_ROWS - 1) / PK_ROWS); }

void pack_count_scan(const PackArgs& a, long long* d_block_counts, long long* d_totals, int* d_flags, cudaStream_t st) {
    const int nb = pack_num_blocks(a.n);
    if (nb == 0) { OB_CUDA(cudaMemsetAsync(d_totals, 0, 2 * sizeof(long long), st)); return; }
    pack_count_kernel<<<nb, PK_THREADS, 0, st>>>(a.d_group, a.d_w, a.n, d_block_counts, d_flags);
    OB_CUDA(cudaGetLastError());
    pack_scan_kernel<<<1, 1024, 0, st>>>(d_block_counts, nb, d_totals);
    OB_CUDA(cudaGetLastError());
}

void pack_scatter(const PackArgs& a, const long long* d_block_base, GroupData ga, GroupData gb, int* d_flags,
                  cudaStream_t st, int blk0, int blk1, const PackWindow* win) {
    const int nb = (blk1 < 0 ? pack_num_blocks(a.n) : blk1) - blk0;
    if (nb <= 0) return;
    PackKernelParams p;
    p.n = a.n; p.n_cont = a.n_cont; p.n_cat = a.n_cat; p.K = a.K; p.ldx = a.ldx;
    p.cont = a.d_cont; p.cat = a.d_cat; p.cat_levels = a.d_cat_levels; p.dummy_start = a.d_dummy_start;
    p.y = a.d_y; p.w = a.d_w; p.group = a.d_group; p.block_base = d_block_base;
    p.XA = ga.X; p.XB = gb.X; p.wA = ga.w; p.wB = gb.w; p.XsA = ga.Xs; p.XsB = gb.Xs;
    p.srcA = ga.src; p.srcB = gb.src; p.flags = d_flags; p.blk0 = blk0;
    for (int g = 0; g < 2; ++g) {
        p.shift[g] = win ? win->shift[g] : 0;
        p.n_local[g] = win ? win->n_local[g] : 0x7fffffffffffffffLL;
        p.lo_add[g] = win ? win->lo_add[g] : 0;
        p.hi_base[g] = win ? win->hi_base[g] : 0;
        p.EX[g] = win ? win->EX[g] : nullptr; p.Ew[g] = win ? win->Ew[g] : nullptr; p.Esrc[g] = win ? win->Esrc[g] : nullptr;
    }
    p.src_add = win ? win->src_add : 0u;
    // the widest odd tile row that fits next to the kernel's static shared memory; wider designs are staged in passes
    cudaFuncAttributes fa;
    OB_CUDA(cudaFuncGetAttributes(&fa, pack_scatter_kernel));
    const int max_ts = (int)((227 * 1024 - fa.sharedSizeBytes) / (sizeof(double) * PK_ROWS));
    const int V = a.K + 1;
    p.tile_cols = std::min(V, (max_ts - 1) | 1);
    const size_t smem = sizeof(double) * (size_t)PK_ROWS * (p.tile_cols | 1);
    OB_CUDA(cudaFuncSetAttribute(pack_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pack_scatter_kernel<<<nb, PK_THREADS, smem, st>>>(p);
    OB_CUDA(cudaGetLastError());
}

// ---- WLS pre-scaling: the reference runs OLS on sqrt(w)-scaled rows (ols.rs:68-78); done once here ----
__global__ void __launch_bounds__(256) scale_rows_kernel(const double* __restrict__ X, const double* __restrict__ w,
                                                         double* __restrict__ Xs, long long total, int ldx) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long row = e / ldx;
        Xs[e] = sqrt(w[row]) * X[e];
    }
}

void scale_rows_launch(const GroupData& g, int ldx, cudaStream_t st) {
    if (!g.Xs) return;
    const long long total = g.n_pad * (long long)ldx;
    scale_rows_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, 148 * 32), 256, 0, st>>>(g.X, g.w, g.Xs, total, ldx);
    OB_CUDA(cudaGetLastError());
}

void scale_rows_range_launch(const GroupData& g, int ldx, int64_t row0, int64_t rows, cudaStream_t st) {
    if (!g.Xs || rows <= 0) return;
    const long long total = rows * (long long)ldx;
    scale_rows_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, 148 * 32), 256, 0, st>>>(g.X + row0 * ldx, g.w + row0, g.Xs + row0 * ldx,
                                                                                                  total, ldx);
    OB_CUDA(cudaGetLastError());
}

__global__ void __launch_bounds__(256) iota_kernel(uint32_t* __restrict__ dst, long long n, uint32_t first) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = first + (uint32_t)i;
}

__global__ void __launch_bounds__(256) add_u32_kernel(uint32_t* __restrict__ p, long long n, uint32_t add) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] += add;
}

void add_u32_launch(uint32_t* p, int64_t n, uint32_t add, cudaStream_t st) {
    if (n == 0 || add == 0) return;
    add_u32_kernel<<<(unsigned)std::min<long long>((n + 255) / 256, 148 * 16), 256, 0, st>>>(p, n, add);
    OB_CUDA(cudaGetLastError());
}

void iota_launch(uint32_t* dst, int64_t n, uint32_t first, cudaStream_t st) {
    if (n == 0) return;
    iota_kernel<<<(unsigned)std::min<long long>((n + 255) / 256, 148 * 16), 256, 0, st>>>(dst, n, first);
    OB_CUDA(cudaGetLastError());
}

// ---- outcome refresh (callers that re-run the decomposition on the same X with another y: JMP's two runs,
//      jmp.rs:44-106; the engine's perturbed-wage sweeps, engine/src/analysis.rs:871-914) ----
__global__ void __launch_bounds__(256) update_outcome_kernel(double* __restrict__ X, double* __restrict__ Xs,
                                                             const double* __restrict__ w, const uint32_t* __restrict__ src,
                                                             const double* __restrict__ y, long long n, int K, int ldx) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (long long)gridDim.x * blockDim.x) {
        const double v = y[src[r]];
        X[r * ldx + K] = v;
        if (Xs) Xs[r * ldx + K] = sqrt(w[r]) * v;
    }
}

void update_outcome_launch(const GroupData& g, int K, int ldx, const double* d_y_frame, cudaStream_t st) {
    if (g.n == 0) return;
    update_outcome_kernel<<<(unsigned)std::min<long long>((g.n + 255) / 256, 148 * 16), 256, 0, st>>>(g.X, g.Xs, g.w, g.src, d_y_frame,
                                                                                                     g.n, K, ldx);
    OB_CUDA(cudaGetLastError());
}

// ---- re-layout of a packed design to a wider row stride (room for more outcome columns): design columns copied,
//      everything from column K on zeroed ----
__global__ void __launch_bounds__(256) relayout_kernel(const double* __restrict__ src, int ld_src, double* __restrict__ dst, int ld_dst,
                                                       long long rows, int K) {
    const long long total = rows * ld_dst;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / ld_dst; const int c = (int)(e - r * ld_dst);
        dst[e] = c < K ? src[r * ld_src + c] : 0.0;
    }
}

void relayout_launch(const double* src, int ld_src, double* dst, int ld_dst, int64_t rows, int K, cudaStream_t st) {
    if (rows == 0) return;
    const long long total = rows * (long long)ld_dst;
    relayout_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, 148 * 32), 256, 0, st>>>(src, ld_src, dst, ld_dst, rows, K);
    OB_CUDA(cudaGetLastError());
}

// ---- point-estimate residuals r = y - X beta (ols.rs:118-119), one warp per row ----
__global__ void __launch_bounds__(256) residuals_kernel(const double* __restrict__ X, long long n, int K, int ycol, int ldx,
                                                        const double* __restrict__ beta, double* __restrict__ out) {
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n) return;
    const double* row = X + warp * ldx;
    double s = 0.0;
    for (int j = lane; j < K; j += 32) s += row[j] * beta[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[warp] = row[ycol] - s;
}

void residuals_launch(const GroupData& g, int K, int ycol, int ldx, const double* d_beta, double* d_out, cudaStream_t st) {
    if (g.n == 0) return;
    const long long threads = g.n * 32;
    residuals_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(g.X, g.n, K, ycol, ldx, d_beta, d_out);
    OB_CUDA(cudaGetLastError());
}

}  // namespace ob
