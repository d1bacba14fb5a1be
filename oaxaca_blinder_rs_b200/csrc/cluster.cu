// csrc/cluster.cu -- cluster bootstrap: resample whole clusters (firms, households, panel units) instead of rows.
//
// A clustered replicate is still a column of row multiplicities: if unit u is drawn c_u times, every row of u has
// multiplicity c_u.  So the resampler draws a multiplicity matrix over UNITS, U[panel][unit][BM], with the row kernels of
// resample.cu (n = M units instead of n_g rows), and counts_expand_kernel turns it into the row matrix C the Gram
// contraction reads: C[panel][row][:] = U[panel][uid[row]][:].  The contraction, its column table and the reduction do not
// change; only the group row counts become per replicate (rows[2][slots], summed here, read by the solve).
//
// Attach (ob_design_attach_clusters): a code per frame row is gathered through each group's frame-row map (src), checked
// against [0, n_codes), the codes present in a stratum are marked and an exclusive scan over the code space gives the unit
// index (units ordered by ascending code).  BY_GROUP: one stratum per group, a unit is a (cluster, group) pair.  JOINT: one
// stratum over both groups.
#include "common.cuh"
#include "internal.h"

#include <algorithm>

namespace ob {

// uid[row] = codes_frame[src[row]] (the raw code for now), present[code] = 1; flags[0] |= 1 on a code out of range
__global__ void __launch_bounds__(256) cluster_gather_kernel(const int32_t* __restrict__ codes_frame, const uint32_t* __restrict__ src,
                                                             long long n, int32_t n_codes, uint32_t* __restrict__ uid,
                                                             uint8_t* __restrict__ present, int* __restrict__ flags) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int32_t c = codes_frame[src[i]];
        if (c < 0 || c >= n_codes) { atomicOr(flags, 1); uid[i] = 0; continue; }
        uid[i] = (uint32_t)c;
        present[c] = 1;
    }
}

// unit[code] = number of present codes below it (exclusive scan of the marks, one block); *units = the total
constexpr int SCAN_THREADS = 1024;
__global__ void __launch_bounds__(SCAN_THREADS) cluster_scan_kernel(const uint8_t* __restrict__ present, int32_t n_codes,
                                                                    uint32_t* __restrict__ unit, long long* __restrict__ units) {
    __shared__ long long part[SCAN_THREADS];
    const long long per = ((long long)n_codes + SCAN_THREADS - 1) / SCAN_THREADS;
    const long long lo = (long long)threadIdx.x * per, hi = lo + per < n_codes ? lo + per : n_codes;
    long long s = 0;
    for (long long c = lo; c < hi; ++c) s += present[c];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int off = 1; off < SCAN_THREADS; off <<= 1) {     // Hillis-Steele inclusive scan of the per-thread counts
        const long long v = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    long long base = part[threadIdx.x] - s;
    for (long long c = lo; c < hi; ++c) { unit[c] = (uint32_t)base; base += present[c]; }
    if (threadIdx.x == SCAN_THREADS - 1) *units = part[SCAN_THREADS - 1];
}

__global__ void __launch_bounds__(256) cluster_remap_kernel(uint32_t* __restrict__ uid, long long n, const uint32_t* __restrict__ unit) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        uid[i] = unit[uid[i]];
}

static int grid_for(long long n) { return (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, 148LL * 16)); }

void cluster_gather_launch(const int32_t* d_codes_frame, const uint32_t* src, int64_t n, int32_t n_codes, uint32_t* uid,
                           uint8_t* present, int* d_flags, cudaStream_t st) {
    if (n == 0) return;
    cluster_gather_kernel<<<grid_for(n), 256, 0, st>>>(d_codes_frame, src, n, n_codes, uid, present, d_flags);
    OB_CUDA(cudaGetLastError());
}

void cluster_scan_launch(const uint8_t* present, int32_t n_codes, uint32_t* unit, long long* d_units, cudaStream_t st) {
    cluster_scan_kernel<<<1, SCAN_THREADS, 0, st>>>(present, n_codes, unit, d_units);
    OB_CUDA(cudaGetLastError());
}

void cluster_remap_launch(uint32_t* uid, int64_t n, const uint32_t* unit, cudaStream_t st) {
    if (n == 0) return;
    cluster_remap_kernel<<<grid_for(n), 256, 0, st>>>(uid, n, unit);
    OB_CUDA(cudaGetLastError());
}

// C[panel][row][q*16 ..] = U[panel][uid[row]][q*16 ..], 16 counts per thread with 16-byte loads and stores; pad rows
// [n, n_pad) are written as zero.  The per-slot row sums (the group's rows in each replicate) are reduced like the column
// sums of counts_philox_body: shuffle over the warp's row lanes, shared memory over the block, one atomic per block and
// slot into rows[slot].
template <typename CountT>
__global__ void __launch_bounds__(256) counts_expand_kernel(CountT* __restrict__ C, const CountT* __restrict__ U,
                                                            const uint32_t* __restrict__ uid, long long n, long long n_pad,
                                                            long long u_pad, long long slots, int rows_per_block,
                                                            long long* __restrict__ rows) {
    __shared__ unsigned ssum[BM];      // <= rows_per_block * 65535 < 2^32
    if (threadIdx.x < BM) ssum[threadIdx.x] = 0;
    __syncthreads();
    constexpr int VEC = 16 * sizeof(CountT) / 16;      // uint4 per thread and row: 1 (8-bit) or 2 (16-bit)
    const int panel = blockIdx.y;
    const int q = threadIdx.x & 7, rl = threadIdx.x >> 3;
    const long long row_begin = (long long)blockIdx.x * rows_per_block;
    const CountT* Up = U + (long long)panel * u_pad * BM + q * 16;
    unsigned sums[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) sums[e] = 0;
    for (long long row = row_begin + rl; row < row_begin + rows_per_block && row < n_pad; row += 32) {
        uint4 v[VEC];
        if (row < n) {
            const uint4* s = reinterpret_cast<const uint4*>(Up + (long long)uid[row] * BM);
#pragma unroll
            for (int k = 0; k < VEC; ++k) v[k] = __ldg(s + k);
            const uint32_t* w = reinterpret_cast<const uint32_t*>(v);
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const int bit = e * (int)sizeof(CountT) * 8;
                sums[e] += (w[bit >> 5] >> (bit & 31)) & (sizeof(CountT) == 1 ? 0xFFu : 0xFFFFu);
            }
        } else {
#pragma unroll
            for (int k = 0; k < VEC; ++k) v[k] = make_uint4(0, 0, 0, 0);
        }
        uint4* d = reinterpret_cast<uint4*>(C + ((long long)panel * n_pad + row) * BM + q * 16);
#pragma unroll
        for (int k = 0; k < VEC; ++k) d[k] = v[k];
    }
#pragma unroll
    for (int e = 0; e < 16; ++e) {
        unsigned s = sums[e];
        s += __shfl_xor_sync(0xffffffffu, s, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if ((threadIdx.x & 31) < 8 && s != 0) atomicAdd(&ssum[q * 16 + e], s);
    }
    __syncthreads();
    if (threadIdx.x < BM) {
        const long long slot = (long long)panel * BM + threadIdx.x;
        const unsigned s = ssum[threadIdx.x];
        if (s != 0 && slot < slots) atomicAdd(reinterpret_cast<unsigned long long*>(rows + slot), (unsigned long long)s);
    }
}

void counts_expand_launch(const ExpandArgs& a, cudaStream_t st) {
    if (a.n_pad == 0) return;
    const int rows_per_block = 2048;
    dim3 grid((unsigned)((a.n_pad + rows_per_block - 1) / rows_per_block), (unsigned)a.panels);
    if (a.count_bytes == 1)
        counts_expand_kernel<uint8_t><<<grid, 256, 0, st>>>((uint8_t*)a.C, (const uint8_t*)a.U, a.uid, a.n, a.n_pad, a.u_pad,
                                                            a.slots, rows_per_block, a.rows);
    else
        counts_expand_kernel<uint16_t><<<grid, 256, 0, st>>>((uint16_t*)a.C, (const uint16_t*)a.U, a.uid, a.n, a.n_pad, a.u_pad,
                                                             a.slots, rows_per_block, a.rows);
    OB_CUDA(cudaGetLastError());
}

}  // namespace ob
