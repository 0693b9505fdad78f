// Dense-tile path of the GATConv message passing for near-dense graphs (the 1 Mb / 100 kb maps:
// >= ~50 % of all pairs are edges).  Same arithmetic as conv.cu (torch-geometric 1.7.2 GATConv,
// ctor sites models.py:619,1013; SURVEY.md Appendix A.3), different loop order:
//
//   CSR path   : warp per row, gathers xl[col] edge by edge -> nnz * H*C * 4 B of L2 gather traffic
//                (12.8 GB at 2.5k dense loci), FFMA-starved.
//   dense path : per head, the attention matrix P_h [N x N] is never stored; tiles of it are
//                regenerated from the rank-1 logits  z_ij = a_src[j] + a_dst[i], the row statistics
//                (max_i, 1/sum_i) and a bit mask of the pattern, and fed to register-tiled fp32
//                FFMA GEMMs (64x128 CTA tile, 8x8 per thread):
//     fwd   : out_h   = P_h    @ XL_h            K = N sources
//     bwd-1 : dA_h    = G_h    @ XL_h^T          K = C; epilogue turns dA into dz (softmax + LeakyReLU
//                                                backward, row term <g_i, out_i - bias>) and reduces it to
//                                                per-tile partial row sums (d a_dst) and column sums (d a_src)
//     bwd-2 : dXL_h   = P_h^T  @ G_h  (+ d a_src * att_l + d a_dst * att_r)
// Tensor cores are not used: the reference computes in fp32 and parity is 1e-5 (TF32 is 1e-3).
#include "common.cuh"

namespace hicgat {
namespace {

constexpr int BM = 64, BN = 128, BK = 16;   // CTA tile (rows x cols) and k-step
constexpr int TM = 8, TN = 8;               // per-thread outputs: rows {ty*4..+3, 32+ty*4..+3}, cols {tx*4..+3, 64+tx*4..+3}
constexpr int kThreads = (BM / TM) * (BN / TN);  // 8 x 16 = 128

template <int BM_>
struct Tiles {
    float a[2][BK][BM_];
    float b[2][BK][BN];
};

__device__ __forceinline__ float lrelu(float z, float slope) { return z > 0.f ? z : z * slope; }

// acc[r][c] += sum_k a[k][row(r)] * b[k][col(c)] over one staged k-step.  BM_ = 64: 8 rows per thread
// {ty*4..+3, 32+ty*4..+3}; BM_ = 32: 4 rows per thread {ty*4..+3}.  Columns {tx*4..+3, 64+tx*4..+3}.
template <int BM_>
__device__ __forceinline__ void mma_step(float (&acc)[BM_ / 8][TN], const float (*__restrict__ as)[BM_], const float (*__restrict__ bs)[BN], int ty, int tx) {
    constexpr int TM_ = BM_ / 8;
#pragma unroll
    for (int k = 0; k < BK; ++k) {
        float a[TM_];
        const float4 a0 = *reinterpret_cast<const float4*>(&as[k][ty * 4]);
        a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
        if constexpr (TM_ == 8) {
            const float4 a1 = *reinterpret_cast<const float4*>(&as[k][32 + ty * 4]);
            a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
        }
        const float4 b0 = *reinterpret_cast<const float4*>(&bs[k][tx * 4]);
        const float4 b1 = *reinterpret_cast<const float4*>(&bs[k][64 + tx * 4]);
        const float b[TN] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int r = 0; r < TM_; ++r)
#pragma unroll
            for (int c = 0; c < TN; ++c) acc[r][c] = fmaf(a[r], b[c], acc[r][c]);
    }
}
__device__ __forceinline__ int out_row(int ty, int r) { return (r < 4 ? 0 : 32) + ty * 4 + (r & 3); }
__device__ __forceinline__ int out_col(int tx, int c) { return (c < 4 ? 0 : 64) + tx * 4 + (c & 3); }

struct DenseArgs {
    int n, H, C;           // loci, heads, channels per head
    int words;             // mask words per row
    const uint32_t* mask;  // [n][words]  bit j of row i: edge (i, j) of the self-loop pattern (symmetric)
    const float* a_src;    // [n][H]
    const float* a_dst;    // [n][H]
    const float* rmax;     // [n][H] row max of leaky_relu(z)
    const float* rinv;     // [n][H] 1 / (row sum of exp + 1e-16)
    float slope;
};

// attention weight a_ij (normalised) for head h; bit = edge present
__device__ __forceinline__ float att_weight(bool bit, float asj, float adi, float mx, float inv, float slope) {
    return bit ? __expf(lrelu(asj + adi, slope) - mx) * inv : 0.f;  // argument <= 0: ex2.approx, rel. error ~5e-7
}

// ------------------------------------------------------------------ row statistics (CSR, warp per row)
template <int H>
__global__ void __launch_bounds__(256) gat_row_stats_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                            const float* __restrict__ a_src, const float* __restrict__ a_dst, float slope, int n,
                                                            float* __restrict__ rmax, float* __restrict__ rinv) {
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const int rs = rowptr[i], re = rowptr[i + 1];
    float adst[H], m[H], s[H];
#pragma unroll
    for (int h = 0; h < H; ++h) { adst[h] = a_dst[i * H + h]; m[h] = -INFINITY; s[h] = 0.f; }
    for (int k = rs + lane; k < re; k += 32) {
        const int j = col[k];
#pragma unroll
        for (int h = 0; h < H; ++h) m[h] = fmaxf(m[h], lrelu(a_src[j * H + h] + adst[h], slope));
    }
#pragma unroll
    for (int h = 0; h < H; ++h) m[h] = warp_max(m[h]);
    for (int k = rs + lane; k < re; k += 32) {
        const int j = col[k];
#pragma unroll
        for (int h = 0; h < H; ++h) s[h] += expf(lrelu(a_src[j * H + h] + adst[h], slope) - m[h]);
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float t = warp_sum(s[h]);
        if (lane == 0) { rmax[i * H + h] = m[h]; rinv[i * H + h] = 1.0f / (t + 1e-16f); }
    }
}

__global__ void __launch_bounds__(256) mask_from_csr_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int n, int words,
                                                            uint32_t* __restrict__ mask) {
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    for (int k = rowptr[i] + lane; k < rowptr[i + 1]; k += 32) {
        const int j = col[k];
        atomicOr(mask + (size_t)i * words + (j >> 5), 1u << (j & 31));  // integer OR: order-independent
    }
}

// ------------------------------------------------------------------ generated attention tiles
// A-tile of P (rows = targets i, k = sources j):      as[k][m] = a_{i0+m, j0+k}           (fwd)
// A-tile of P^T (rows = sources j, k = targets i):    as[k][m] = a_{i0'+k, j0'+m}         (bwd-2)
// thread t fills row m = t % BM_ for the k-group t / BM_ (BK * BM_ / 128 consecutive k)
template <bool TRANSPOSED, int BM_>
__device__ __forceinline__ void gen_att_tile(float (*__restrict__ as)[BM_], const DenseArgs& A, int h, int m0, int k0, int t) {
    constexpr int KG = BK * BM_ / kThreads;  // 8 (BM_ = 64) or 4 (BM_ = 32) sources per thread
    const int m = t % BM_, kb = (t / BM_) * KG;
    const int gm = m0 + m;  // fwd: target i ; transposed: source j
    float fixed_s = 0.f, fixed_d = 0.f, mx = 0.f, inv = 0.f;
    uint32_t bits = 0;
    if (gm < A.n) {
        if (!TRANSPOSED) { fixed_d = A.a_dst[gm * A.H + h]; mx = A.rmax[gm * A.H + h]; inv = A.rinv[gm * A.H + h]; }
        else fixed_s = A.a_src[gm * A.H + h];
        // the pattern is symmetric (set_diag of a symmetrised map): bit (gm, gk) serves both orientations
        const int gk0 = k0 + kb;  // multiple of KG: the KG bits sit inside one mask word
        if (gk0 < A.n) bits = (A.mask[(size_t)gm * A.words + (gk0 >> 5)] >> (gk0 & 31)) & ((1u << KG) - 1u);
    }
#pragma unroll
    for (int q = 0; q < KG; ++q) {
        const int gk = k0 + kb + q;
        float v = 0.f;
        if (gk < A.n && ((bits >> q) & 1u)) {
            if (!TRANSPOSED) v = att_weight(true, A.a_src[gk * A.H + h], fixed_d, mx, inv, A.slope);
            else v = att_weight(true, fixed_s, A.a_dst[gk * A.H + h], A.rmax[gk * A.H + h], A.rinv[gk * A.H + h], A.slope);
        }
        as[kb + q][m] = v;
    }
}

// B-tile from a row-major [n][ld] matrix, rows = k (sources / targets), cols = channels c0..c0+127
// thread t loads 4 float4 per k-step: row k = t/32 + 4*q (q=0..3), cols (t%32)*4
__device__ __forceinline__ void load_rows_tile(float4 (&reg)[4], const float* __restrict__ X, int ld, int n, int k0, int c0, int t) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int gk = k0 + (t >> 5) + 4 * q;
        reg[q] = gk < n ? __ldg(reinterpret_cast<const float4*>(X + (size_t)gk * ld + c0 + (t & 31) * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
__device__ __forceinline__ void store_rows_tile(float (*__restrict__ bs)[BN], const float4 (&reg)[4], int t) {
#pragma unroll
    for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(&bs[(t >> 5) + 4 * q][(t & 31) * 4]) = reg[q];
}

// out[i, h*C + c] = sum_j a_ij xl[j, h*C + c] + bias          (TRANSPOSED = false, X = xl)
// dxl[j, h*C + c] = sum_i a_ij g[i, h*C + c] + d_a_src[j] att_l[c] + d_a_dst[j] att_r[c]   (TRANSPOSED = true, X = g)
template <bool TRANSPOSED, int BM_>
__global__ void __launch_bounds__(kThreads) gat_dense_spmm_kernel(const DenseArgs A, const float* __restrict__ X, const float* __restrict__ v0,
                                                                  const float* __restrict__ v1, const float* __restrict__ s0,
                                                                  const float* __restrict__ s1, float* __restrict__ out, float* __restrict__ part,
                                                                  int kper) {
    // gridDim.z > 1: split-K over the sources/targets; CTA z accumulates k in [z*kper, (z+1)*kper) and writes its
    // raw tile to part[z]; gat_dense_combine_kernel adds the splits in order and applies the epilogue
    constexpr int TM_ = BM_ / 8;
    __shared__ __align__(16) Tiles<BM_> T;
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int F = A.H * A.C;
    const int ctiles = A.C / BN;                 // column tiles per head
    const int h = blockIdx.y / ctiles, c0 = h * A.C + (blockIdx.y % ctiles) * BN;
    const int m0 = blockIdx.x * BM_;
    float acc[TM_][TN];
#pragma unroll
    for (int r = 0; r < TM_; ++r)
#pragma unroll
        for (int c = 0; c < TN; ++c) acc[r][c] = 0.f;

    float4 breg[4];
    const int kbeg = blockIdx.z * kper, kend = min(A.n, kbeg + kper);  // kper is a multiple of BK
    const int ksteps = (kend - kbeg + BK - 1) / BK;
    gen_att_tile<TRANSPOSED, BM_>(T.a[0], A, h, m0, kbeg, t);
    load_rows_tile(breg, X, F, A.n, kbeg, c0, t);
    store_rows_tile(T.b[0], breg, t);
    __syncthreads();
    for (int ks = 0; ks < ksteps; ++ks) {
        const int cur = ks & 1, nxt = cur ^ 1;
        const bool more = ks + 1 < ksteps;
        if (more) load_rows_tile(breg, X, F, A.n, kbeg + (ks + 1) * BK, c0, t);   // in flight during the FMAs
        mma_step<BM_>(acc, T.a[cur], T.b[cur], ty, tx);
        if (more) {
            gen_att_tile<TRANSPOSED, BM_>(T.a[nxt], A, h, m0, kbeg + (ks + 1) * BK, t);
            store_rows_tile(T.b[nxt], breg, t);
        }
        __syncthreads();
    }
    if (gridDim.z > 1) {  // raw partial tile; epilogue in the combine kernel
        float* dst = part + (size_t)blockIdx.z * A.n * F;
#pragma unroll
        for (int r = 0; r < TM_; ++r) {
            const int gm = m0 + (TM_ == 8 ? out_row(ty, r) : ty * 4 + r);
            if (gm >= A.n) continue;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int gc = c0 + half * 64 + tx * 4;
                *reinterpret_cast<float4*>(dst + (size_t)gm * F + gc) =
                    make_float4(acc[r][half * 4 + 0], acc[r][half * 4 + 1], acc[r][half * 4 + 2], acc[r][half * 4 + 3]);
            }
        }
        return;
    }
#pragma unroll
    for (int r = 0; r < TM_; ++r) {
        const int gm = m0 + (TM_ == 8 ? out_row(ty, r) : ty * 4 + r);
        if (gm >= A.n) continue;
        float e0 = 0.f, e1 = 0.f;
        if (TRANSPOSED) { e0 = s0[gm * A.H + h]; e1 = s1[gm * A.H + h]; }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int gc = c0 + half * 64 + tx * 4;
            float4 o = make_float4(acc[r][half * 4 + 0], acc[r][half * 4 + 1], acc[r][half * 4 + 2], acc[r][half * 4 + 3]);
            const float4 p = __ldg(reinterpret_cast<const float4*>(v0 + gc));
            if (!TRANSPOSED) { o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w; }  // + bias
            else {
                const float4 q = __ldg(reinterpret_cast<const float4*>(v1 + gc));
                o.x += e0 * p.x + e1 * q.x; o.y += e0 * p.y + e1 * q.y; o.z += e0 * p.z + e1 * q.z; o.w += e0 * p.w + e1 * q.w;
            }
            *reinterpret_cast<float4*>(out + (size_t)gm * F + gc) = o;
        }
    }
}

// out[m, c] = sum_z part[z][m, c] (+ bias[c])  or  (+ s0[m,h] v0[c] + s1[m,h] v1[c]) -- split order fixed
template <bool TRANSPOSED>
__global__ void __launch_bounds__(256) gat_dense_combine_kernel(const float* __restrict__ part, int nsplit, int n, int H, int C,
                                                                const float* __restrict__ v0, const float* __restrict__ v1,
                                                                const float* __restrict__ s0, const float* __restrict__ s1, float* __restrict__ out) {
    const int F = H * C;
    const size_t total4 = (size_t)n * F / 4;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (size_t)gridDim.x * blockDim.x) {
        float4 o = __ldcg(reinterpret_cast<const float4*>(part) + q);
        for (int z = 1; z < nsplit; ++z) {
            const float4 p = __ldcg(reinterpret_cast<const float4*>(part + (size_t)z * n * F) + q);
            o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
        }
        const int m = (int)(q * 4 / F), c = (int)(q * 4 % F), h = c / C;
        const float4 a = __ldg(reinterpret_cast<const float4*>(v0 + c));
        if (!TRANSPOSED) { o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w; }
        else {
            const float4 b = __ldg(reinterpret_cast<const float4*>(v1 + c));
            const float e0 = s0[m * H + h], e1 = s1[m * H + h];
            o.x += e0 * a.x + e1 * b.x; o.y += e0 * a.y + e1 * b.y; o.z += e0 * a.z + e1 * b.z; o.w += e0 * a.w + e1 * b.w;
        }
        reinterpret_cast<float4*>(out)[q] = o;
    }
}

// ------------------------------------------------------------------ bwd-1: dA = G XL^T, fused dz epilogue
// rowdot[i,h] = <g_i, out_i - bias>_h  (= sum_j a_ij dA_ij): warp per row
template <int H>
__global__ void __launch_bounds__(256) gat_rowdot_kernel(const float* __restrict__ g, const float* __restrict__ out, const float* __restrict__ bias,
                                                         int n, int C, float* __restrict__ rowdot) {
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const int F = H * C;
#pragma unroll
    for (int h = 0; h < H; ++h) {
        float s = 0.f;
        for (int c = lane * 4; c < C; c += 128) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(g + (size_t)i * F + h * C + c));
            const float4 o = __ldg(reinterpret_cast<const float4*>(out + (size_t)i * F + h * C + c));
            const float4 b = __ldg(reinterpret_cast<const float4*>(bias + h * C + c));
            s += a.x * (o.x - b.x) + a.y * (o.y - b.y) + a.z * (o.z - b.z) + a.w * (o.w - b.w);
        }
        s = warp_sum(s);
        if (lane == 0) rowdot[i * H + h] = s;
    }
}

// K-major tiles from two row-major [n][ld] matrices: as[k][m] = G[i0+m][cbase+k], bs[k][nn] = XL[j0+nn][cbase+k].
// Warp w owns channels 4w..4w+3 of the k-step, lanes own rows (lane + 32 q): the transposed shared
// stores of a warp then hit 32 consecutive banks (conflict-free); the 64 B a row contributes per
// k-step are fetched as four 16 B pieces by the four warps (same two sectors, L1/L2 hits).
template <int ROWS>
__device__ __forceinline__ void load_kmajor(float4 (&reg)[ROWS / 32], const float* __restrict__ X, int ld, int n, int r0, int cb, int t) {
#pragma unroll
    for (int q = 0; q < ROWS / 32; ++q) {
        const int gr = r0 + (t & 31) + 32 * q;
        reg[q] = gr < n ? __ldg(reinterpret_cast<const float4*>(X + (size_t)gr * ld + cb + (t >> 5) * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
template <int ROWS, int LD>
__device__ __forceinline__ void store_kmajor(float (*__restrict__ s)[LD], const float4 (&reg)[ROWS / 32], int t) {
#pragma unroll
    for (int q = 0; q < ROWS / 32; ++q) {
        const int r = (t & 31) + 32 * q, k = (t >> 5) * 4;
        s[k + 0][r] = reg[q].x; s[k + 1][r] = reg[q].y; s[k + 2][r] = reg[q].z; s[k + 3][r] = reg[q].w;
    }
}

// grid (row tiles of 64 targets, col tiles of 128 sources, H).  Partials:
//   rowpart[(tile_n * n + i) * H + h] = sum_{j in tile} dz_ij     colpart[(tile_m * n + j) * H + h] = sum_{i in tile} dz_ij
__global__ void __launch_bounds__(kThreads) gat_dense_bwd_logits_kernel(const DenseArgs A, const float* __restrict__ g, const float* __restrict__ xl,
                                                                        const float* __restrict__ rowdot, float* __restrict__ rowpart,
                                                                        float* __restrict__ colpart) {
    __shared__ __align__(16) Tiles<BM> T;
    __shared__ float red_row[BM][16 + 1];   // per output row: 16 tx partials
    __shared__ float red_col[BN][8 + 1];    // per output col: 8 ty partials
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int F = A.H * A.C, h = blockIdx.z;
    const int i0 = blockIdx.x * BM, j0 = blockIdx.y * BN;
    float acc[TM][TN];
#pragma unroll
    for (int r = 0; r < TM; ++r)
#pragma unroll
        for (int c = 0; c < TN; ++c) acc[r][c] = 0.f;
    float4 areg[BM / 32], breg[BN / 32];
    const int ksteps = A.C / BK;
    load_kmajor<BM>(areg, g, F, A.n, i0, h * A.C, t);
    load_kmajor<BN>(breg, xl, F, A.n, j0, h * A.C, t);
    store_kmajor<BM, BM>(T.a[0], areg, t);
    store_kmajor<BN, BN>(T.b[0], breg, t);
    __syncthreads();
    for (int ks = 0; ks < ksteps; ++ks) {
        const int cur = ks & 1, nxt = cur ^ 1;
        const bool more = ks + 1 < ksteps;
        if (more) {
            load_kmajor<BM>(areg, g, F, A.n, i0, h * A.C + (ks + 1) * BK, t);
            load_kmajor<BN>(breg, xl, F, A.n, j0, h * A.C + (ks + 1) * BK, t);
        }
        mma_step<BM>(acc, T.a[cur], T.b[cur], ty, tx);
        if (more) {
            store_kmajor<BM, BM>(T.a[nxt], areg, t);
            store_kmajor<BN, BN>(T.b[nxt], breg, t);
        }
        __syncthreads();
    }
    // epilogue: dA -> dz, row / column partial sums
    float csum[TN];
#pragma unroll
    for (int c = 0; c < TN; ++c) csum[c] = 0.f;
#pragma unroll
    for (int r = 0; r < TM; ++r) {
        const int lr = out_row(ty, r), gi = i0 + lr;
        float rsum = 0.f;
        if (gi < A.n) {
            const float adi = A.a_dst[gi * A.H + h], mx = A.rmax[gi * A.H + h], inv = A.rinv[gi * A.H + h], rd = rowdot[gi * A.H + h];
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int gj0 = j0 + half * 64 + tx * 4;
                uint32_t bits = 0;
                if (gj0 < A.n) bits = (A.mask[(size_t)gi * A.words + (gj0 >> 5)] >> (gj0 & 31)) & 0xfu;  // gj0 multiple of 4
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int gj = gj0 + q, c = half * 4 + q;
                    float dz = 0.f;
                    if (gj < A.n && ((bits >> q) & 1u)) {
                        const float z = A.a_src[gj * A.H + h] + adi;
                        const float a = __expf(lrelu(z, A.slope) - mx) * inv;
                        const float de = a * (acc[r][c] - rd);
                        dz = z > 0.f ? de : de * A.slope;
                    }
                    rsum += dz;
                    csum[c] += dz;
                }
            }
        }
        red_row[lr][tx] = rsum;
    }
#pragma unroll
    for (int c = 0; c < TN; ++c) red_col[out_col(tx, c)][ty] = csum[c];
    __syncthreads();
    if (t < BM) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 16; ++q) s += red_row[t][q];
        if (i0 + t < A.n) rowpart[((size_t)blockIdx.y * A.n + i0 + t) * A.H + h] = s;
    }
    {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) s += red_col[t][q];
        if (j0 + t < A.n) colpart[((size_t)blockIdx.x * A.n + j0 + t) * A.H + h] = s;
    }
}

// d_a_dst[i,h] = sum over column tiles, d_a_src[j,h] = sum over row tiles (fixed order)
__global__ void gat_dense_reduce_partials_kernel(const float* __restrict__ rowpart, const float* __restrict__ colpart, int nH, int ntn, int ntm,
                                                 float* __restrict__ d_a_dst, float* __restrict__ d_a_src) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nH) return;
    float s = 0.f;
    for (int q = 0; q < ntn; ++q) s += rowpart[(size_t)q * nH + e];
    d_a_dst[e] = s;
    s = 0.f;
    for (int q = 0; q < ntm; ++q) s += colpart[(size_t)q * nH + e];
    d_a_src[e] = s;
}

}  // namespace
}  // namespace hicgat

using namespace hicgat;

namespace {
constexpr int kMaxSplit = 4;
struct DenseLayout {
    int words, ntm, ntn, nsplit, kper;
    size_t off_rmax, off_rinv, off_rowdot, off_dsrc, off_ddst, off_rowpart, off_colpart, off_split, total;
};
DenseLayout dense_layout(int64_t n, int H, int C = 0) {
    DenseLayout L;
    L.words = (int)((n + 31) / 32);
    L.ntm = (int)((n + BM - 1) / BM);
    L.ntn = (int)((n + BN - 1) / BN);
    const size_t nh = align_up(sizeof(float) * (size_t)n * H, 256);
    L.off_rmax = 0;
    L.off_rinv = L.off_rmax + nh;
    L.off_rowdot = L.off_rinv + nh;
    L.off_dsrc = L.off_rowdot + nh;
    L.off_ddst = L.off_dsrc + nh;
    L.off_rowpart = L.off_ddst + nh;
    L.off_colpart = L.off_rowpart + align_up(sizeof(float) * (size_t)L.ntn * n * H, 256);
    L.off_split = L.off_colpart + align_up(sizeof(float) * (size_t)L.ntm * n * H, 256);
    // split-K of the two SpMM-shaped GEMMs: 64-row tiles are the efficient ones (8x8 per thread), so small
    // maps get their parallelism from splitting the k range instead of from smaller tiles
    L.nsplit = 1;
    L.kper = (int)((n + BK - 1) / BK * BK);
    if (C > 0) {
        const int64_t ctas = (int64_t)L.ntm * H * (C / BN);
        while (L.nsplit < kMaxSplit && ctas * L.nsplit < 2 * 148 && n / (L.nsplit * 2) >= 8 * BK) L.nsplit *= 2;
        L.kper = (int)(((n + L.nsplit - 1) / L.nsplit + BK - 1) / BK * BK);
    }
    L.total = L.off_split + (L.nsplit > 1 ? sizeof(float) * (size_t)L.nsplit * n * H * C : 0);
    return L;
}
}  // namespace

extern "C" size_t hicgat_gat_dense_mask_words(int64_t n) { return n > 0 ? (size_t)((n + 31) / 32) : 0; }

extern "C" int hicgat_gat_dense_build_mask(const int32_t* rowptr, const int32_t* col, int64_t n, uint32_t* mask, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(rowptr && col && mask && n > 0 && n < (1ll << 24), "hicgat_gat_dense_build_mask: bad arguments");
    const int words = (int)((n + 31) / 32);
    HICGAT_CUDA(cudaMemsetAsync(mask, 0, sizeof(uint32_t) * (size_t)n * words, stream));
    mask_from_csr_kernel<<<(unsigned)((n + 7) / 8), 256, 0, stream>>>(rowptr, col, (int)n, words, mask);
    HICGAT_CHECK_LAUNCH("mask_from_csr_kernel");
    return HICGAT_OK;
}

extern "C" size_t hicgat_gat_dense_workspace_bytes(int64_t n, int heads, int channels) {
    if (n <= 0 || !gat_shape_supported(heads, channels)) return 0;
    return dense_layout(n, heads, channels).total;
}

// forward: a_src/a_dst (logit halves) from the caller (gat logit kernel), row stats into the workspace
extern "C" int hicgat_gat_dense_fwd(const int32_t* rowptr, const int32_t* col, const uint32_t* mask, int64_t n, int heads, int channels,
                                    const float* xl, const float* a_src, const float* a_dst, const float* bias, float slope,
                                    float* out, void* workspace, size_t workspace_bytes, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(rowptr && col && mask && xl && a_src && a_dst && bias && out && workspace, "hicgat_gat_dense_fwd: null pointer");
    HICGAT_REQUIRE(n > 0 && n < (1ll << 24) && gat_shape_supported(heads, channels), "hicgat_gat_dense_fwd: unsupported n/heads/channels (%lld,%d,%d)", (long long)n, heads, channels);
    HICGAT_REQUIRE(aligned16(xl) && aligned16(out) && aligned16(bias), "hicgat_gat_dense_fwd: 16-byte alignment required");
    const DenseLayout L = dense_layout(n, heads, channels);
    if (workspace_bytes < L.total) { set_error("hicgat_gat_dense_fwd: workspace %zu < required %zu", workspace_bytes, L.total); return HICGAT_ERR_WORKSPACE; }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* rmax = reinterpret_cast<float*>(ws + L.off_rmax);
    float* rinv = reinterpret_cast<float*>(ws + L.off_rinv);
    const unsigned rgrid = (unsigned)((n + 7) / 8);
    switch (heads) {
        case 1: gat_row_stats_kernel<1><<<rgrid, 256, 0, stream>>>(rowptr, col, a_src, a_dst, slope, (int)n, rmax, rinv); break;
        case 2: gat_row_stats_kernel<2><<<rgrid, 256, 0, stream>>>(rowptr, col, a_src, a_dst, slope, (int)n, rmax, rinv); break;
        default: gat_row_stats_kernel<4><<<rgrid, 256, 0, stream>>>(rowptr, col, a_src, a_dst, slope, (int)n, rmax, rinv); break;
    }
    HICGAT_CHECK_LAUNCH("gat_row_stats_kernel");
    DenseArgs A{(int)n, heads, channels, L.words, mask, a_src, a_dst, rmax, rinv, slope};
    const unsigned ytiles = (unsigned)(heads * (channels / BN));
    float* split = reinterpret_cast<float*>(ws + L.off_split);
    gat_dense_spmm_kernel<false, 64><<<dim3((unsigned)L.ntm, ytiles, (unsigned)L.nsplit), kThreads, 0, stream>>>(A, xl, bias, nullptr, nullptr, nullptr, out, split, L.kper);
    HICGAT_CHECK_LAUNCH("gat_dense_spmm_kernel<fwd>");
    if (L.nsplit > 1) {
        gat_dense_combine_kernel<false><<<148 * 4, 256, 0, stream>>>(split, L.nsplit, (int)n, heads, channels, bias, nullptr, nullptr, nullptr, out);
        HICGAT_CHECK_LAUNCH("gat_dense_combine_kernel<fwd>");
    }
    return HICGAT_OK;
}

// backward: needs the forward's workspace (row stats) untouched, `out` of the forward and g = dL/dout.
// Produces dxl and the logit-half gradients d_a_src / d_a_dst ([n,H], in the workspace and copied out).
extern "C" int hicgat_gat_dense_bwd(const uint32_t* mask, int64_t n, int heads, int channels, const float* xl, const float* a_src,
                                    const float* a_dst, const float* att_l, const float* att_r, const float* bias, float slope,
                                    const float* out, const float* gout, float* dxl, float* d_a_src, float* d_a_dst,
                                    void* workspace, size_t workspace_bytes, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(mask && xl && a_src && a_dst && att_l && att_r && bias && out && gout && dxl && d_a_src && d_a_dst && workspace, "hicgat_gat_dense_bwd: null pointer");
    HICGAT_REQUIRE(n > 0 && n < (1ll << 24) && gat_shape_supported(heads, channels), "hicgat_gat_dense_bwd: unsupported n/heads/channels");
    HICGAT_REQUIRE(aligned16(xl) && aligned16(out) && aligned16(gout) && aligned16(dxl) && aligned16(att_l) && aligned16(att_r) && aligned16(bias), "hicgat_gat_dense_bwd: 16-byte alignment required");
    const DenseLayout L = dense_layout(n, heads, channels);
    if (workspace_bytes < L.total) { set_error("hicgat_gat_dense_bwd: workspace %zu < required %zu", workspace_bytes, L.total); return HICGAT_ERR_WORKSPACE; }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* rmax = reinterpret_cast<float*>(ws + L.off_rmax);
    float* rinv = reinterpret_cast<float*>(ws + L.off_rinv);
    float* rowdot = reinterpret_cast<float*>(ws + L.off_rowdot);
    float* rowpart = reinterpret_cast<float*>(ws + L.off_rowpart);
    float* colpart = reinterpret_cast<float*>(ws + L.off_colpart);
    const unsigned rgrid = (unsigned)((n + 7) / 8);
    switch (heads) {
        case 1: gat_rowdot_kernel<1><<<rgrid, 256, 0, stream>>>(gout, out, bias, (int)n, channels, rowdot); break;
        case 2: gat_rowdot_kernel<2><<<rgrid, 256, 0, stream>>>(gout, out, bias, (int)n, channels, rowdot); break;
        default: gat_rowdot_kernel<4><<<rgrid, 256, 0, stream>>>(gout, out, bias, (int)n, channels, rowdot); break;
    }
    HICGAT_CHECK_LAUNCH("gat_rowdot_kernel");
    DenseArgs A{(int)n, heads, channels, L.words, mask, a_src, a_dst, rmax, rinv, slope};
    dim3 g1((unsigned)L.ntm, (unsigned)L.ntn, (unsigned)heads);
    gat_dense_bwd_logits_kernel<<<g1, kThreads, 0, stream>>>(A, gout, xl, rowdot, rowpart, colpart);
    HICGAT_CHECK_LAUNCH("gat_dense_bwd_logits_kernel");
    const int nH = (int)n * heads;
    gat_dense_reduce_partials_kernel<<<(nH + 255) / 256, 256, 0, stream>>>(rowpart, colpart, nH, L.ntn, L.ntm, d_a_dst, d_a_src);
    HICGAT_CHECK_LAUNCH("gat_dense_reduce_partials_kernel");
    const unsigned ytiles = (unsigned)(heads * (channels / BN));
    float* split = reinterpret_cast<float*>(ws + L.off_split);
    gat_dense_spmm_kernel<true, 64><<<dim3((unsigned)L.ntm, ytiles, (unsigned)L.nsplit), kThreads, 0, stream>>>(A, gout, att_l, att_r, d_a_src, d_a_dst, dxl, split, L.kper);
    HICGAT_CHECK_LAUNCH("gat_dense_spmm_kernel<bwd>");
    if (L.nsplit > 1) {
        gat_dense_combine_kernel<true><<<148 * 4, 256, 0, stream>>>(split, L.nsplit, (int)n, heads, channels, att_l, att_r, d_a_src, d_a_dst, dxl);
        HICGAT_CHECK_LAUNCH("gat_dense_combine_kernel<bwd>");
    }
    return HICGAT_OK;
}
