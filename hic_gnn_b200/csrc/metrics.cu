// dSCC (Spearman correlation of the i<j wish distances and reconstructed distances) at map sizes where neither the
// N x N distance matrix nor the P = N(N-1)/2 gathered vectors of the reference can exist (SURVEY.md section 8 row f-3).
//
// Reference: scipy.stats.spearmanr(dist_truth, dist_out) on the triu_indices gathers, every iteration in
// HiC_GAT_generalize_directly.py:210-242 and once per model in HiC-GNN_main.py:135-139 -- 16 B of int64 indices per pair,
// two P-vectors and an O(P log P) sort: 20 GB + minutes at 50k loci.
//
// Here: Spearman = Pearson of the average ranks.  Ranks are taken from two FINE HISTOGRAMS (B bins each) built in one
// streaming pass over the target rows (d is recomputed from the coordinates, never stored): the rank of a value is the
// mid-rank of its bin, i.e. the bin is treated as one tie group.  That is exact for the big tie group of a Hi-C wish matrix
// (every zero-contact pair has t == 1.0 and falls into one bin) and perturbs every other rank by at most half a bin population
// (relative 1/(2B) ~ 1e-7 at B = 2^22), far inside the 1e-3 the parity contract asks of the final dSCC.  A second streaming pass
// accumulates sum_k rank_t(k) * rank_d(k) in f64.  Both passes are row-block local: a sharded caller all-reduces the histograms
// and the cross sum.
#include <algorithm>

#include "common.cuh"

namespace hicgat {
namespace {

constexpr int kRows = 32;   // rows per block tile
constexpr int kThreadsM = 256;

__device__ __forceinline__ int bin_of(float v, float scale, int nbins) {
    int b = (int)(v * scale);
    return b < 0 ? 0 : (b >= nbins ? nbins - 1 : b);
}

// |x_j - x_i| in f32, the one distance every dSCC kernel bins
__device__ __forceinline__ float pair_dist(float xj, float yj, float zj, float xi, float yi, float zi) {
    const float dx = xj - xi, dy = yj - yi, dz = zj - zi;
    return sqrtf(dx * dx + dy * dy + dz * dz);
}

// A block tile is kRows rows from i0 by kThreadsM columns; it holds pairs i < j unless it lies on or below the diagonal.
__device__ __forceinline__ bool tile_below_diagonal(int i0) { return (int)(blockIdx.x + 1) * kThreadsM - 1 <= i0; }

// coordinates of the tile's rows into shared memory (rows past n repeat row n - 1; they are never paired)
__device__ __forceinline__ void load_tile_rows(float (*s_x)[3], const float* __restrict__ coords, int i0, int n) {
    if (threadIdx.x < kRows * 3) {
        const int r = min(i0 + threadIdx.x / 3, n - 1);
        s_x[threadIdx.x / 3][threadIdx.x % 3] = coords[(size_t)r * 3 + threadIdx.x % 3];
    }
}

// grid = (column tiles of 256, row tiles of 32); upper triangle only (i < j)
template <bool CROSS>
__global__ void __launch_bounds__(kThreadsM) rank_pass_kernel(const float* __restrict__ coords, const float* __restrict__ target, int64_t pitch, int n, int r0, int r1,
                                                              float d_scale, float t_scale, int nbins, unsigned long long* __restrict__ hist_d,
                                                              unsigned long long* __restrict__ hist_t, const double* __restrict__ rank_d,
                                                              const double* __restrict__ rank_t, double* __restrict__ cross) {
    __shared__ float s_x[kRows][3];
    __shared__ double s_red[kThreadsM / 32];
    const int i0 = r0 + blockIdx.y * kRows;
    const int j = blockIdx.x * kThreadsM + threadIdx.x;
    if (tile_below_diagonal(i0)) return;
    load_tile_rows(s_x, coords, i0, n);
    __syncthreads();
    double acc = 0.0;
    if (j < n) {
        const float xj = coords[(size_t)j * 3], yj = coords[(size_t)j * 3 + 1], zj = coords[(size_t)j * 3 + 2];
        const int rows = min(kRows, r1 - i0);
        for (int u = 0; u < rows; ++u) {
            const int i = i0 + u;
            if (i >= j) break;
            const float d = pair_dist(xj, yj, zj, s_x[u][0], s_x[u][1], s_x[u][2]);
            const float t = __ldg(target + (size_t)(i - r0) * pitch + j);
            const int bd = bin_of(d, d_scale, nbins), bt = bin_of(t, t_scale, nbins);
            if constexpr (CROSS) {
                acc += rank_d[bd] * rank_t[bt];
            } else {
                atomicAdd(hist_d + bd, 1ull);
                atomicAdd(hist_t + bt, 1ull);
            }
        }
    }
    if constexpr (CROSS) {
        acc = warp_sum(acc);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kThreadsM / 32; ++w) s += s_red[w];
            if (s != 0.0) atomicAdd(cross, s);
        }
    }
}

// Implicit (sparse) target: every pair i<j of rows [r0,r1) goes into hist_d (no target stream).
__global__ void __launch_bounds__(kThreadsM) dist_hist_kernel(const float* __restrict__ coords, int n, int r0, int r1, float d_scale, int nbins,
                                                              unsigned long long* __restrict__ hist_d) {
    __shared__ float s_x[kRows][3];
    const int i0 = r0 + blockIdx.y * kRows;
    const int j = blockIdx.x * kThreadsM + threadIdx.x;
    if (tile_below_diagonal(i0)) return;
    load_tile_rows(s_x, coords, i0, n);
    __syncthreads();
    if (j >= n) return;
    const float xj = coords[(size_t)j * 3], yj = coords[(size_t)j * 3 + 1], zj = coords[(size_t)j * 3 + 2];
    const int rows = min(kRows, r1 - i0);
    for (int u = 0; u < rows; ++u) {
        if (i0 + u >= j) break;
        atomicAdd(hist_d + bin_of(pair_dist(xj, yj, zj, s_x[u][0], s_x[u][1], s_x[u][2]), d_scale, nbins), 1ull);
    }
}

// bins of the reconstructed distance of the stored pairs (i < j) of CSR rows [r0, r1): one thread per stored entry
__global__ void __launch_bounds__(256) edge_dist_bins_kernel(const float* __restrict__ coords, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                             int r0, int r1, float d_scale, int nbins, int32_t* __restrict__ bins) {
    const int i = r0 + blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= r1) return;
    const float xi = coords[(size_t)i * 3], yi = coords[(size_t)i * 3 + 1], zi = coords[(size_t)i * 3 + 2];
    for (int k = rowptr[i] + lane; k < rowptr[i + 1]; k += 32) {
        const int j = col[k];
        bins[k] = j > i ? bin_of(pair_dist(coords[(size_t)j * 3], coords[(size_t)j * 3 + 1], coords[(size_t)j * 3 + 2], xi, yi, zi), d_scale, nbins) : -1;
    }
}


// ------------------------------------------------------------------ per-step dSCC on the device (hicgat_dscc_*)
constexpr int kScanThreads = 256;
constexpr int kScanPer = 16;                              // bins per thread of the mid-rank scan
constexpr int kScanBins = kScanThreads * kScanPer;        // bins per scan block
constexpr int kFinishThreads = 1024;
constexpr int kCsrRowsPerBlock = 8;                       // one warp per CSR row

// Sum of v over the block (every thread passes its value; all threads must call it), in an order fixed by the launch shape.
template <int THREADS>
__device__ __forceinline__ double block_sum_fixed(double v, double* s_red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) s += s_red[w];
    }
    __syncthreads();
    return s;  // valid in thread 0
}

// hist[bin] += 1 for every lane with bin >= 0 (all 32 lanes call it).  When every valid lane of the warp holds the same bin (the t == 1.0
// group of a wish matrix; a collapsed structure) one lane adds their count; otherwise each lane adds 1.  A shuffle and a vote per
// call: __match_any_sync on every pair cost more than it saved on spread-out distances (DESIGN.md section 6d).
__device__ __forceinline__ void hist_add_warp(unsigned long long* __restrict__ hist, int bin) {
    const unsigned valid = __ballot_sync(0xffffffffu, bin >= 0);
    if (valid == 0u) return;
    const int first = __shfl_sync(0xffffffffu, bin, __ffs(valid) - 1);
    if (__all_sync(0xffffffffu, bin < 0 || bin == first)) {
        if ((int)(threadIdx.x & 31) == __ffs(valid) - 1) atomicAdd(hist + bin, (unsigned long long)__popc(valid));
    } else if (bin >= 0) {
        atomicAdd(hist + bin, 1ull);
    }
}

// d_scale = (float)(nbins / dmax), dmax = sqrt(sum span^2) (1 + 1e-6) + 1e-30 in f64 of the f32 bounding box: the host rule of
// metrics.dscc_streamed, with explicitly rounded operations so that no contraction changes a bit.  One block.
__global__ void __launch_bounds__(kFinishThreads) dscc_scale_kernel(const float* __restrict__ coords, int n, int nbins, float* __restrict__ d_scale) {
    __shared__ float s_mn[3][kFinishThreads / 32], s_mx[3][kFinishThreads / 32];
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = threadIdx.x; i < n; i += kFinishThreads) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const float v = coords[(size_t)i * 3 + q];
            mn[q] = fminf(mn[q], v);
            mx[q] = fmaxf(mx[q], v);
        }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        for (int o = 16; o > 0; o >>= 1) {
            mn[q] = fminf(mn[q], __shfl_xor_sync(0xffffffffu, mn[q], o));
            mx[q] = fmaxf(mx[q], __shfl_xor_sync(0xffffffffu, mx[q], o));
        }
        if ((threadIdx.x & 31) == 0) {
            s_mn[q][threadIdx.x >> 5] = mn[q];
            s_mx[q][threadIdx.x >> 5] = mx[q];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ss = 0.0;
        for (int q = 0; q < 3; ++q) {
            float a = s_mn[q][0], b = s_mx[q][0];
            for (int w = 1; w < kFinishThreads / 32; ++w) {
                a = fminf(a, s_mn[q][w]);
                b = fmaxf(b, s_mx[q][w]);
            }
            const double span = (double)__fsub_rn(b, a);
            ss = __dadd_rn(ss, __dmul_rn(span, span));
        }
        const double dmax = __dadd_rn(__dmul_rn(__dsqrt_rn(ss), 1.0 + 1e-6), 1e-30);
        *d_scale = __double2float_rn(__ddiv_rn((double)nbins, dmax));
    }
}

// Histogram of the pairs i < j with i in rows [r0, r1) of an n x n map: of the reconstructed distance (TARGET = false, scale read from
// the device) or of the dense target (TARGET = true; row i at target + (i - r0) pitch).  Same tiles as rank_pass_kernel; a warp whose
// pairs all share a bin (the t == 1.0 group of a wish matrix, a collapsed structure) adds once instead of serialising 32 atomics on one
// address.
template <bool TARGET>
__global__ void __launch_bounds__(kThreadsM) dscc_hist_kernel(const float* __restrict__ coords, const float* __restrict__ target, int64_t pitch, int n,
                                                              int r0, int r1, const float* __restrict__ d_scale_p, float t_scale, int nbins,
                                                              unsigned long long* __restrict__ hist) {
    __shared__ float s_x[kRows][3];
    const int i0 = r0 + blockIdx.y * kRows;
    const int j = blockIdx.x * kThreadsM + threadIdx.x;
    if (tile_below_diagonal(i0)) return;
    if (!TARGET) load_tile_rows(s_x, coords, i0, n);
    __syncthreads();
    const bool col_ok = j < n;
    float xj = 0.f, yj = 0.f, zj = 0.f, d_scale = 0.f;
    if (!TARGET) {
        d_scale = *d_scale_p;
        if (col_ok) xj = coords[(size_t)j * 3], yj = coords[(size_t)j * 3 + 1], zj = coords[(size_t)j * 3 + 2];
    }
    const int rows = min(kRows, r1 - i0);
    for (int u = 0; u < rows; ++u) {  // warp-uniform trip count: every lane takes part in the match
        const int i = i0 + u;
        int b = -1;
        if (col_ok && i < j) {
            b = TARGET ? bin_of(__ldg(target + (size_t)(i - r0) * pitch + j), t_scale, nbins)
                       : bin_of(pair_dist(xj, yj, zj, s_x[u][0], s_x[u][1], s_x[u][2]), d_scale, nbins);
        }
        hist_add_warp(hist, b);
    }
}

// per scan block: the number of pairs in its kScanBins bins (exact in u64)
__global__ void __launch_bounds__(kScanThreads) dscc_bin_block_sums_kernel(const unsigned long long* __restrict__ hist, int nbins,
                                                                           unsigned long long* __restrict__ block_sums) {
    __shared__ unsigned long long s_red[kScanThreads / 32];
    const int64_t base = (int64_t)blockIdx.x * kScanBins;
    unsigned long long c = 0;
    for (int k = threadIdx.x; k < kScanBins; k += kScanThreads)
        if (base + k < nbins) c += hist[base + k];
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long s = 0;
        for (int w = 0; w < kScanThreads / 32; ++w) s += s_red[w];
        block_sums[blockIdx.x] = s;
    }
}

// Mid-ranks of a histogram: rank[b] = (pairs in bins < b) + (hist[b] + 1) / 2, exact in f64 (integers and halves below 2^53), so the
// table equals metrics._midranks bit for bit.  Per block: partial[0][blk] = sum_b h (rank - mean)^2, partial[1][blk] = sum_b h rank.
__global__ void __launch_bounds__(kScanThreads) dscc_midrank_kernel(const unsigned long long* __restrict__ hist, int nbins,
                                                                    const unsigned long long* __restrict__ block_sums, double mean,
                                                                    double* __restrict__ rank, double* __restrict__ partials) {
    __shared__ unsigned long long s_scan[kScanThreads];
    __shared__ double s_red[kScanThreads / 32];
    // pairs in every earlier scan block
    unsigned long long before = 0;
    for (int k = threadIdx.x; k < (int)blockIdx.x; k += kScanThreads) before += block_sums[k];
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if ((threadIdx.x & 31) == 0) s_scan[threadIdx.x >> 5] = before;
    __syncthreads();
    unsigned long long offset = 0;
    for (int w = 0; w < kScanThreads / 32; ++w) offset += s_scan[w];
    __syncthreads();
    // this thread's kScanPer consecutive bins, then an exclusive scan of the per-thread totals (Hillis-Steele in shared memory)
    const int64_t b0 = (int64_t)blockIdx.x * kScanBins + (int64_t)threadIdx.x * kScanPer;
    unsigned long long h[kScanPer], tot = 0;
#pragma unroll
    for (int k = 0; k < kScanPer; ++k) {
        h[k] = b0 + k < nbins ? hist[b0 + k] : 0ull;
        tot += h[k];
    }
    s_scan[threadIdx.x] = tot;
    __syncthreads();
    for (int o = 1; o < kScanThreads; o <<= 1) {
        const unsigned long long add = threadIdx.x >= o ? s_scan[threadIdx.x - o] : 0ull;
        __syncthreads();
        s_scan[threadIdx.x] += add;
        __syncthreads();
    }
    unsigned long long below = offset + s_scan[threadIdx.x] - tot;
    double var = 0.0, hr = 0.0;
#pragma unroll
    for (int k = 0; k < kScanPer; ++k) {
        if (b0 + k < nbins) {
            const double hk = (double)h[k];
            const double r = (double)below + (hk + 1.0) / 2.0;
            rank[b0 + k] = r;
            const double e = r - mean;
            var += hk * e * e;
            hr += hk * r;
            below += h[k];
        }
    }
    const double sv = block_sum_fixed<kScanThreads>(var, s_red);
    const double sh = block_sum_fixed<kScanThreads>(hr, s_red);
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = sv;
        partials[gridDim.x + blockIdx.x] = sh;
    }
}

// Dense target, rows [r0, r1) (row i at target + (i - r0) pitch): partial[tile] = sum over the tile's pairs i < j of
// rank_d[bin(d_ij)] * rank_t[bin(t_ij)]; every tile of the block writes its slot.
__global__ void __launch_bounds__(kThreadsM) dscc_cross_dense_kernel(const float* __restrict__ coords, const float* __restrict__ target, int64_t pitch, int n,
                                                                     int r0, int r1, const float* __restrict__ d_scale_p, float t_scale, int nbins,
                                                                     const double* __restrict__ rank_d, const double* __restrict__ rank_t,
                                                                     double* __restrict__ partials) {
    __shared__ float s_x[kRows][3];
    __shared__ double s_red[kThreadsM / 32];
    const int i0 = r0 + blockIdx.y * kRows;
    const int j = blockIdx.x * kThreadsM + threadIdx.x;
    const size_t slot = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    if (tile_below_diagonal(i0)) {
        if (threadIdx.x == 0) partials[slot] = 0.0;
        return;
    }
    load_tile_rows(s_x, coords, i0, n);
    __syncthreads();
    double acc = 0.0;
    if (j < n) {
        const float d_scale = *d_scale_p;
        const float xj = coords[(size_t)j * 3], yj = coords[(size_t)j * 3 + 1], zj = coords[(size_t)j * 3 + 2];
        const int rows = min(kRows, r1 - i0);
        for (int u = 0; u < rows; ++u) {
            const int i = i0 + u;
            if (i >= j) break;
            const float d = pair_dist(xj, yj, zj, s_x[u][0], s_x[u][1], s_x[u][2]);
            const float t = __ldg(target + (size_t)(i - r0) * pitch + j);
            acc += rank_d[bin_of(d, d_scale, nbins)] * rank_t[bin_of(t, t_scale, nbins)];
        }
    }
    const double s = block_sum_fixed<kThreadsM>(acc, s_red);
    if (threadIdx.x == 0) partials[slot] = s;
}

// Implicit target: over the stored CSR entries k = (i, j), j > i, of rows [r0, r1) (one warp per row), partial[0][blk] =
// sum rank_t_csr[k] rank_d[bin(d_ij)] and partial[1][blk] = sum rank_d[bin(d_ij)]; the fill group's share follows from them
// (dscc_finish_kernel).
__global__ void __launch_bounds__(kCsrRowsPerBlock * 32) dscc_cross_csr_kernel(const float* __restrict__ coords, const int32_t* __restrict__ rowptr,
                                                                               const int32_t* __restrict__ col, const double* __restrict__ rank_t_csr,
                                                                               int r0, int r1, const float* __restrict__ d_scale_p, int nbins,
                                                                               const double* __restrict__ rank_d, double* __restrict__ partials) {
    __shared__ double s_red[kCsrRowsPerBlock];
    const int i = r0 + blockIdx.x * kCsrRowsPerBlock + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    double sx = 0.0, sd = 0.0;
    if (i < r1) {
        const float d_scale = *d_scale_p;
        const float xi = coords[(size_t)i * 3], yi = coords[(size_t)i * 3 + 1], zi = coords[(size_t)i * 3 + 2];
        for (int k = rowptr[i] + lane; k < rowptr[i + 1]; k += 32) {
            const int j = col[k];
            if (j <= i) continue;
            const double rd = rank_d[bin_of(pair_dist(coords[(size_t)j * 3], coords[(size_t)j * 3 + 1], coords[(size_t)j * 3 + 2], xi, yi, zi), d_scale, nbins)];
            sx += rank_t_csr[k] * rd;
            sd += rd;
        }
    }
    const double tx = block_sum_fixed<kCsrRowsPerBlock * 32>(sx, s_red);
    const double td = block_sum_fixed<kCsrRowsPerBlock * 32>(sd, s_red);
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = tx;
        partials[gridDim.x + blockIdx.x] = td;
    }
}

__device__ double block_sum_strided(const double* __restrict__ v, int64_t count, double* s_red) {
    double a = 0.0;
    for (int64_t k = threadIdx.x; k < count; k += kFinishThreads) a += v[k];
    return block_sum_fixed<kFinishThreads>(a, s_red);
}

// out[q] = sum of v[q count .. (q + 1) count) in a fixed order for q < nsums, out[q] = 0 for nsums <= q < nout.  One block.
__global__ void __launch_bounds__(kFinishThreads) dscc_sum_kernel(const double* __restrict__ v, int64_t count, int nsums, int nout, double* __restrict__ out) {
    __shared__ double s_red[kFinishThreads / 32];
    for (int q = 0; q < nout; ++q) {
        const double s = q < nsums ? block_sum_strided(v + q * count, count, s_red) : 0.0;
        if (threadIdx.x == 0) out[q] = s;
    }
}

// rho = (cross - P mean^2) / sqrt(var_d var_t), NaN unless var_d var_t is finite and > 0; cross_sum = the rank-summed f64[2] of the block
// cross sums.  Implicit target: cross = cross_sum[0] + rank_fill (sum_all h rank_d - cross_sum[1]), cross_sum[1] = sum_stored rank_d.
// One block.
__global__ void __launch_bounds__(kFinishThreads) dscc_finish_kernel(const double* __restrict__ scan_partials, int nscan,
                                                                     const double* __restrict__ cross_sum, int implicit,
                                                                     const double* __restrict__ var_t, const double* __restrict__ rank_fill,
                                                                     double npairs, double* __restrict__ rho) {
    __shared__ double s_red[kFinishThreads / 32];
    const double var_d = block_sum_strided(scan_partials, nscan, s_red);
    double cross = cross_sum[0];
    if (implicit) {
        const double sum_hr = block_sum_strided(scan_partials + nscan, nscan, s_red);
        if (threadIdx.x == 0) cross += *rank_fill * (sum_hr - cross_sum[1]);
    }
    if (threadIdx.x == 0) {
        const double mean = (npairs + 1.0) / 2.0;
        const double vv = var_d * *var_t;
        const double r = (cross - npairs * mean * mean) / sqrt(vv);
        *rho = (vv > 0.0 && isfinite(vv) && isfinite(r)) ? r : __longlong_as_double(0x7ff8000000000000ll);
    }
}

}  // namespace
}  // namespace hicgat

using namespace hicgat;

static int rank_pass(bool cross, const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, float d_scale, float t_scale,
                     int nbins, unsigned long long* hist_d, unsigned long long* hist_t, const double* rank_d, const double* rank_t, double* cross_out,
                     cudaStream_t stream) {
    HICGAT_REQUIRE(n > 0 && n < (1ll << 30) && r0 >= 0 && r1 >= r0 && r1 <= n && nbins > 0, "hicgat_rank_*: bad n/r0/r1/nbins");
    HICGAT_REQUIRE(coords && (target || r0 == r1) && pitch >= n, "hicgat_rank_*: null pointer / bad pitch");
    if (r1 == r0) return HICGAT_OK;
    dim3 grid((unsigned)((n + kThreadsM - 1) / kThreadsM), (unsigned)((r1 - r0 + kRows - 1) / kRows));
    if (cross) rank_pass_kernel<true><<<grid, kThreadsM, 0, stream>>>(coords, target, pitch, (int)n, (int)r0, (int)r1, d_scale, t_scale, nbins, nullptr, nullptr, rank_d, rank_t, cross_out);
    else rank_pass_kernel<false><<<grid, kThreadsM, 0, stream>>>(coords, target, pitch, (int)n, (int)r0, (int)r1, d_scale, t_scale, nbins, hist_d, hist_t, nullptr, nullptr, nullptr);
    HICGAT_CHECK_LAUNCH("rank_pass_kernel");
    return HICGAT_OK;
}

extern "C" int hicgat_rank_histograms(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, float d_scale,
                                      float t_scale, int nbins, uint64_t* hist_d, uint64_t* hist_t, hicgat_stream_t stream) {
    HICGAT_REQUIRE(hist_d && hist_t, "hicgat_rank_histograms: null histogram");
    return rank_pass(false, coords, target, pitch, n, r0, r1, d_scale, t_scale, nbins, reinterpret_cast<unsigned long long*>(hist_d),
                     reinterpret_cast<unsigned long long*>(hist_t), nullptr, nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int hicgat_rank_cross_sum(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, float d_scale,
                                     float t_scale, int nbins, const double* rank_d, const double* rank_t, double* cross, hicgat_stream_t stream) {
    HICGAT_REQUIRE(rank_d && rank_t && cross, "hicgat_rank_cross_sum: null pointer");
    return rank_pass(true, coords, target, pitch, n, r0, r1, d_scale, t_scale, nbins, nullptr, nullptr, rank_d, rank_t, cross, static_cast<cudaStream_t>(stream));
}

extern "C" int hicgat_dist_histogram(const float* coords, int64_t n, int64_t r0, int64_t r1, float d_scale, int nbins, uint64_t* hist_d,
                                     hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(coords && hist_d && n > 0 && n < (1ll << 30) && r0 >= 0 && r1 >= r0 && r1 <= n && nbins > 0, "hicgat_dist_histogram: bad arguments");
    if (r1 == r0) return HICGAT_OK;
    dim3 grid((unsigned)((n + kThreadsM - 1) / kThreadsM), (unsigned)((r1 - r0 + kRows - 1) / kRows));
    dist_hist_kernel<<<grid, kThreadsM, 0, stream>>>(coords, (int)n, (int)r0, (int)r1, d_scale, nbins, reinterpret_cast<unsigned long long*>(hist_d));
    HICGAT_CHECK_LAUNCH("dist_hist_kernel");
    return HICGAT_OK;
}

extern "C" int hicgat_edge_dist_bins(const float* coords, const int32_t* rowptr, const int32_t* col, int64_t n, int64_t r0, int64_t r1, float d_scale,
                                     int nbins, int32_t* bins, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(coords && rowptr && bins && n > 0 && r0 >= 0 && r1 >= r0 && r1 <= n && nbins > 0, "hicgat_edge_dist_bins: bad arguments");
    if (r1 == r0) return HICGAT_OK;
    edge_dist_bins_kernel<<<(unsigned)((r1 - r0 + 7) / 8), 256, 0, stream>>>(coords, rowptr, col, (int)r0, (int)r1, d_scale, nbins, bins);
    HICGAT_CHECK_LAUNCH("edge_dist_bins_kernel");
    return HICGAT_OK;
}

// ------------------------------------------------------------------ hicgat_dscc_*
namespace {
constexpr int64_t kDsccMaxN = 65535ll * kRows;  // grid.y of the tile kernels

struct DsccWorkspace {
    unsigned long long* hist;
    double* rank_d;
    float* d_scale;
    unsigned long long* block_sums;
    double* scan_partials;   // [2][nscan]
    double* cross_partials;  // [2][ncross]
    double* cross_sum;       // [2]: the block cross sum of the (0, n) entry points
    int nscan;
    int64_t ncross;
    size_t bytes;
};

DsccWorkspace dscc_layout(int64_t n, int nbins, void* base) {
    DsccWorkspace w{};
    w.nscan = (int)((nbins + (int64_t)kScanBins - 1) / kScanBins);
    const int64_t tiles = ((n + kThreadsM - 1) / kThreadsM) * ((n + kRows - 1) / kRows);
    w.ncross = std::max<int64_t>(tiles, (n + kCsrRowsPerBlock - 1) / kCsrRowsPerBlock);
    char* p = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* q = p + off;
        off = align_up(off + bytes, 256);
        return q;
    };
    w.hist = reinterpret_cast<unsigned long long*>(take((size_t)nbins * 8));
    w.rank_d = reinterpret_cast<double*>(take((size_t)nbins * 8));
    w.d_scale = reinterpret_cast<float*>(take(sizeof(float)));
    w.block_sums = reinterpret_cast<unsigned long long*>(take((size_t)w.nscan * 8));
    w.scan_partials = reinterpret_cast<double*>(take((size_t)w.nscan * 16));
    w.cross_partials = reinterpret_cast<double*>(take((size_t)w.ncross * 16));
    w.cross_sum = reinterpret_cast<double*>(take(16));
    w.bytes = off;
    return w;
}

bool dscc_sizes_ok(int64_t n, int nbins) { return n > 0 && n <= kDsccMaxN && nbins > 0; }
bool dscc_rows_ok(int64_t n, int64_t r0, int64_t r1, int nbins) { return dscc_sizes_ok(n, nbins) && r0 >= 0 && r0 <= r1 && r1 <= n; }

// zero hist, then add the pairs i < j of rows [r0, r1): distances (of_target = false, scale from the workspace) or the dense block
int dscc_block_hist(bool of_target, const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, const float* d_scale,
                    float t_scale, int nbins, unsigned long long* hist, cudaStream_t stream) {
    HICGAT_CUDA(cudaMemsetAsync(hist, 0, (size_t)nbins * 8, stream));
    if (r1 == r0) return HICGAT_OK;
    const dim3 grid((unsigned)((n + kThreadsM - 1) / kThreadsM), (unsigned)((r1 - r0 + kRows - 1) / kRows));
    if (of_target) dscc_hist_kernel<true><<<grid, kThreadsM, 0, stream>>>(nullptr, target, pitch, (int)n, (int)r0, (int)r1, nullptr, t_scale, nbins, hist);
    else dscc_hist_kernel<false><<<grid, kThreadsM, 0, stream>>>(coords, nullptr, 0, (int)n, (int)r0, (int)r1, d_scale, 0.f, nbins, hist);
    HICGAT_CHECK_LAUNCH("dscc_hist_kernel");
    return HICGAT_OK;
}

// mid-rank table of a (summed) histogram of all P = n (n - 1) / 2 pairs + per-scan-block partials of var and sum h rank (w.scan_partials)
int dscc_hist_midranks(const unsigned long long* hist, int64_t n, int nbins, double* rank, const DsccWorkspace& w, cudaStream_t stream) {
    dscc_bin_block_sums_kernel<<<w.nscan, kScanThreads, 0, stream>>>(hist, nbins, w.block_sums);
    HICGAT_CHECK_LAUNCH("dscc_bin_block_sums_kernel");
    const double npairs = (double)n * (double)(n - 1) / 2.0;
    dscc_midrank_kernel<<<w.nscan, kScanThreads, 0, stream>>>(hist, nbins, w.block_sums, (npairs + 1.0) / 2.0, rank, w.scan_partials);
    HICGAT_CHECK_LAUNCH("dscc_midrank_kernel");
    return HICGAT_OK;
}

// the block's per-tile (per-CSR-block) partials [2][count] -> cross f64[2] (cross[1] = 0 for a dense target)
int dscc_cross_total(int64_t count, bool implicit, double* cross, const DsccWorkspace& w, cudaStream_t stream) {
    dscc_sum_kernel<<<1, kFinishThreads, 0, stream>>>(w.cross_partials, count, implicit ? 2 : 1, 2, cross);
    HICGAT_CHECK_LAUNCH("dscc_sum_kernel");
    return HICGAT_OK;
}
}  // namespace

#define DSCC_WORKSPACE(name)                                                                                                   \
    const DsccWorkspace w = dscc_layout(n, nbins, workspace);                                                                  \
    HICGAT_REQUIRE(workspace_bytes >= w.bytes, name ": workspace of %zu bytes, %zu needed", workspace_bytes, w.bytes);         \
    cudaStream_t stream = static_cast<cudaStream_t>(stream_)

extern "C" size_t hicgat_dscc_workspace_bytes(int64_t n, int nbins) {
    if (!dscc_sizes_ok(n, nbins)) return 0;
    return dscc_layout(n, nbins, nullptr).bytes;
}

// ---- the phases of one evaluation over target rows [r0, r1)
extern "C" int hicgat_dscc_dist_hist_rows(const float* coords, int64_t n, int64_t r0, int64_t r1, int nbins, uint64_t* hist_d, void* workspace,
                                          size_t workspace_bytes, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_rows_ok(n, r0, r1, nbins), "hicgat_dscc_dist_hist_rows: bad n/r0/r1/nbins (need 0 <= r0 <= r1 <= n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(coords && hist_d && workspace, "hicgat_dscc_dist_hist_rows: null pointer");
    DSCC_WORKSPACE("hicgat_dscc_dist_hist_rows");
    dscc_scale_kernel<<<1, kFinishThreads, 0, stream>>>(coords, (int)n, nbins, w.d_scale);  // from all n loci: the same bins on every rank
    HICGAT_CHECK_LAUNCH("dscc_scale_kernel");
    return dscc_block_hist(false, coords, nullptr, 0, n, r0, r1, w.d_scale, 0.f, nbins, reinterpret_cast<unsigned long long*>(hist_d), stream);
}

extern "C" int hicgat_dscc_target_hist_rows(const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, float t_scale, int nbins,
                                            uint64_t* hist_t, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_rows_ok(n, r0, r1, nbins), "hicgat_dscc_target_hist_rows: bad n/r0/r1/nbins (need 0 <= r0 <= r1 <= n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(target && hist_t && pitch >= n, "hicgat_dscc_target_hist_rows: null pointer / bad pitch");
    return dscc_block_hist(true, nullptr, target, pitch, n, r0, r1, nullptr, t_scale, nbins, reinterpret_cast<unsigned long long*>(hist_t),
                           static_cast<cudaStream_t>(stream_));
}

extern "C" int hicgat_dscc_hist_ranks(const uint64_t* hist, int64_t n, int nbins, double* rank, double* var, void* workspace, size_t workspace_bytes,
                                      hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_sizes_ok(n, nbins), "hicgat_dscc_hist_ranks: bad n/nbins (need 0 < n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(hist && rank && var && workspace, "hicgat_dscc_hist_ranks: null pointer");
    DSCC_WORKSPACE("hicgat_dscc_hist_ranks");
    const int rc = dscc_hist_midranks(reinterpret_cast<const unsigned long long*>(hist), n, nbins, rank, w, stream);
    if (rc != HICGAT_OK) return rc;
    dscc_sum_kernel<<<1, kFinishThreads, 0, stream>>>(w.scan_partials, w.nscan, 1, 1, var);
    HICGAT_CHECK_LAUNCH("dscc_sum_kernel");
    return HICGAT_OK;
}

extern "C" int hicgat_dscc_cross_dense_rows(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, float t_scale,
                                            int nbins, const uint64_t* hist_d, const double* rank_t, double* cross, void* workspace,
                                            size_t workspace_bytes, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_rows_ok(n, r0, r1, nbins), "hicgat_dscc_cross_dense_rows: bad n/r0/r1/nbins (need 0 <= r0 <= r1 <= n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(coords && target && hist_d && rank_t && cross && workspace && pitch >= n, "hicgat_dscc_cross_dense_rows: null pointer / bad pitch");
    DSCC_WORKSPACE("hicgat_dscc_cross_dense_rows");
    int rc = dscc_hist_midranks(reinterpret_cast<const unsigned long long*>(hist_d), n, nbins, w.rank_d, w, stream);
    if (rc != HICGAT_OK) return rc;
    const dim3 grid((unsigned)((n + kThreadsM - 1) / kThreadsM), (unsigned)((r1 - r0 + kRows - 1) / kRows));
    if (r1 > r0) {
        dscc_cross_dense_kernel<<<grid, kThreadsM, 0, stream>>>(coords, target, pitch, (int)n, (int)r0, (int)r1, w.d_scale, t_scale, nbins, w.rank_d, rank_t,
                                                                w.cross_partials);
        HICGAT_CHECK_LAUNCH("dscc_cross_dense_kernel");
    }
    return dscc_cross_total((int64_t)grid.x * grid.y, false, cross, w, stream);
}

extern "C" int hicgat_dscc_cross_implicit_rows(const float* coords, const int32_t* rowptr, const int32_t* col, const double* rank_t_csr, int64_t n,
                                               int64_t r0, int64_t r1, int nbins, const uint64_t* hist_d, double* cross, void* workspace,
                                               size_t workspace_bytes, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_rows_ok(n, r0, r1, nbins), "hicgat_dscc_cross_implicit_rows: bad n/r0/r1/nbins (need 0 <= r0 <= r1 <= n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(coords && rowptr && col && rank_t_csr && hist_d && cross && workspace, "hicgat_dscc_cross_implicit_rows: null pointer");
    DSCC_WORKSPACE("hicgat_dscc_cross_implicit_rows");
    int rc = dscc_hist_midranks(reinterpret_cast<const unsigned long long*>(hist_d), n, nbins, w.rank_d, w, stream);
    if (rc != HICGAT_OK) return rc;
    const int blocks = (int)((r1 - r0 + kCsrRowsPerBlock - 1) / kCsrRowsPerBlock);
    if (blocks > 0) {
        dscc_cross_csr_kernel<<<blocks, kCsrRowsPerBlock * 32, 0, stream>>>(coords, rowptr, col, rank_t_csr, (int)r0, (int)r1, w.d_scale, nbins, w.rank_d,
                                                                            w.cross_partials);
        HICGAT_CHECK_LAUNCH("dscc_cross_csr_kernel");
    }
    return dscc_cross_total(blocks, true, cross, w, stream);
}

extern "C" int hicgat_dscc_finish(const double* cross_sum, int64_t n, int nbins, int implicit, const double* rank_fill, const double* var_t, double* rho,
                                  void* workspace, size_t workspace_bytes, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_sizes_ok(n, nbins), "hicgat_dscc_finish: bad n/nbins (need 0 < n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(cross_sum && var_t && rho && workspace && (rank_fill || !implicit), "hicgat_dscc_finish: null pointer");
    DSCC_WORKSPACE("hicgat_dscc_finish");
    dscc_finish_kernel<<<1, kFinishThreads, 0, stream>>>(w.scan_partials, w.nscan, cross_sum, implicit ? 1 : 0, var_t, rank_fill,
                                                         (double)n * (double)(n - 1) / 2.0, rho);
    HICGAT_CHECK_LAUNCH("dscc_finish_kernel");
    return HICGAT_OK;
}

// ---- the full target: the phases over rows (0, n) with the workspace's own histogram and cross sum
extern "C" int hicgat_dscc_target_ranks(const float* target, int64_t pitch, int64_t n, float t_scale, int nbins, double* rank_t, double* var_t,
                                        void* workspace, size_t workspace_bytes, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_sizes_ok(n, nbins), "hicgat_dscc_target_ranks: bad n/nbins (need 0 < n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(target && rank_t && var_t && workspace && pitch >= n, "hicgat_dscc_target_ranks: null pointer / bad pitch");
    DSCC_WORKSPACE("hicgat_dscc_target_ranks");
    const int rc = hicgat_dscc_target_hist_rows(target, pitch, n, 0, n, t_scale, nbins, reinterpret_cast<uint64_t*>(w.hist), stream);
    if (rc != HICGAT_OK) return rc;
    return hicgat_dscc_hist_ranks(reinterpret_cast<const uint64_t*>(w.hist), n, nbins, rank_t, var_t, workspace, workspace_bytes, stream);
}

extern "C" int hicgat_dscc_dense(const float* coords, const float* target, int64_t pitch, int64_t n, float t_scale, int nbins, const double* rank_t,
                                 const double* var_t, double* rho, void* workspace, size_t workspace_bytes, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_sizes_ok(n, nbins), "hicgat_dscc_dense: bad n/nbins (need 0 < n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(coords && target && rank_t && var_t && rho && workspace && pitch >= n, "hicgat_dscc_dense: null pointer / bad pitch");
    DSCC_WORKSPACE("hicgat_dscc_dense");
    uint64_t* hist = reinterpret_cast<uint64_t*>(w.hist);
    int rc = hicgat_dscc_dist_hist_rows(coords, n, 0, n, nbins, hist, workspace, workspace_bytes, stream);
    if (rc == HICGAT_OK) rc = hicgat_dscc_cross_dense_rows(coords, target, pitch, n, 0, n, t_scale, nbins, hist, rank_t, w.cross_sum, workspace, workspace_bytes, stream);
    if (rc == HICGAT_OK) rc = hicgat_dscc_finish(w.cross_sum, n, nbins, 0, nullptr, var_t, rho, workspace, workspace_bytes, stream);
    return rc;
}

extern "C" int hicgat_dscc_implicit(const float* coords, const int32_t* rowptr, const int32_t* col, const double* rank_t_csr, int64_t n,
                                    const double* rank_fill, const double* var_t, int nbins, double* rho, void* workspace, size_t workspace_bytes,
                                    hicgat_stream_t stream_) {
    HICGAT_REQUIRE(dscc_sizes_ok(n, nbins), "hicgat_dscc_implicit: bad n/nbins (need 0 < n <= %lld, nbins > 0)", (long long)kDsccMaxN);
    HICGAT_REQUIRE(coords && rowptr && col && rank_t_csr && rank_fill && var_t && rho && workspace, "hicgat_dscc_implicit: null pointer");
    DSCC_WORKSPACE("hicgat_dscc_implicit");
    uint64_t* hist = reinterpret_cast<uint64_t*>(w.hist);
    int rc = hicgat_dscc_dist_hist_rows(coords, n, 0, n, nbins, hist, workspace, workspace_bytes, stream);
    if (rc == HICGAT_OK) rc = hicgat_dscc_cross_implicit_rows(coords, rowptr, col, rank_t_csr, n, 0, n, nbins, hist, w.cross_sum, workspace, workspace_bytes, stream);
    if (rc == HICGAT_OK) rc = hicgat_dscc_finish(w.cross_sum, n, nbins, 1, rank_fill, var_t, rho, workspace, workspace_bytes, stream);
    return rc;
}
