// Message passing of the two graph-conv layers on the hot path, CSR order, warp per row.
//
//   SAGEConv aggregate : layers.py:75-79   out[i,:] = sum_k w_k x[col_k,:]
//   GATConv            : torch-geometric 1.7.2 GATConv as used at models.py:619 / :1013
//                        (SURVEY.md Appendix A.3): per-edge LeakyReLU logits, segmented softmax
//                        with warp shuffles, vectorised gather-SpMM; backward in the same CSR
//                        order through the transposed-entry permutation (pattern is symmetric).
//
// Nothing is materialised per edge except alpha / dz ([nnz, H] floats); PyG materialises
// [nnz, H, C].  Features are read as float4: lane l owns channels q*128 + 4l .. +3 of each
// 128-wide chunk q (Q = H*C/128 chunks), so one chunk always belongs to a single head.
#include <algorithm>

#include "common.cuh"

namespace hicgat {
namespace {

constexpr int kRowsPerCta = 8;  // 8 warps, one row each

__device__ __forceinline__ float4 ldg_f4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void fma4(float4& acc, float a, const float4& v) {
    acc.x = fmaf(a, v.x, acc.x);
    acc.y = fmaf(a, v.y, acc.y);
    acc.z = fmaf(a, v.z, acc.z);
    acc.w = fmaf(a, v.w, acc.w);
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
    return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
// first k in [lo, hi) with col[k] >= v (col ascending on [lo, hi)), hi if none
__device__ __forceinline__ int lower_bound_i32(const int32_t* __restrict__ col, int lo, int hi, int v) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(col + mid) < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// ------------------------------------------------------------------ weighted CSR SpMM
template <int Q>
__global__ void __launch_bounds__(256) spmm_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                   const float* __restrict__ w, const float* __restrict__ x, int g0, int g1,
                                                   float* __restrict__ out) {
    constexpr int F = Q * 128;
    const int i = g0 + blockIdx.x * kRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= g1) return;
    float4 acc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int rs = rowptr[i], re = rowptr[i + 1];
    for (int base = rs; base < re; base += 32) {
        const int k = base + lane;
        const int myj = k < re ? col[k] : 0;
        const float myw = k < re ? w[k] : 0.f;
        const int cnt = min(32, re - base);
        for (int t = 0; t < cnt; t += 4) {
            int j[4];
            float a[4];
            float4 v[4][Q];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                j[u] = __shfl_sync(0xffffffffu, myj, (t + u) & 31);
                a[u] = __shfl_sync(0xffffffffu, myw, (t + u) & 31);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) v[u][q] = ldg_f4(x + (size_t)j[u] * F + q * 128 + lane * 4);
                }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) fma4(acc[q], a[u], v[u][q]);
                }
        }
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) *reinterpret_cast<float4*>(out + (size_t)(i - g0) * F + q * 128 + lane * 4) = acc[q];
}

// ------------------------------------------------------------------ GAT: logit halves
// a_src[i,h] = <xl[i,h,:], att_l[h,:]>, a_dst[i,h] = <xl[i,h,:], att_r[h,:]>
template <int H, int Q>
__global__ void __launch_bounds__(256) gat_logit_kernel(const float* __restrict__ xl, const float* __restrict__ att_l,
                                                        const float* __restrict__ att_r, int n, float* __restrict__ a_src,
                                                        float* __restrict__ a_dst) {
    constexpr int F = Q * 128, QH = Q / H;
    const int i = blockIdx.x * kRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    float sl[H], sr[H];
#pragma unroll
    for (int h = 0; h < H; ++h) sl[h] = sr[h] = 0.f;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 v = ldg_f4(xl + (size_t)i * F + q * 128 + lane * 4);
        sl[q / QH] += dot4(v, ldg_f4(att_l + q * 128 + lane * 4));
        sr[q / QH] += dot4(v, ldg_f4(att_r + q * 128 + lane * 4));
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float l = warp_sum(sl[h]), r = warp_sum(sr[h]);
        if (lane == 0) {
            a_src[i * H + h] = l;
            a_dst[i * H + h] = r;
        }
    }
}

// ------------------------------------------------------------------ GAT forward
template <int H, int Q, int W>
__global__ void __launch_bounds__(W * 32) gat_fwd_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                      const float* __restrict__ xl, const float* __restrict__ a_src,
                                                      const float* __restrict__ a_dst, const float* __restrict__ bias,
                                                      float slope, int g0, int g1, float* __restrict__ alpha, float* __restrict__ out) {
    constexpr int F = Q * 128, QH = Q / H;
    const int i = g0 + blockIdx.x * W + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= g1) return;
    const int rs = rowptr[i], re = rowptr[i + 1];
    float adst[H], m[H], s[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        adst[h] = a_dst[i * H + h];
        m[h] = -INFINITY;
        s[h] = 0.f;
    }
    // pass 1: row max of leaky_relu(a_src[j] + a_dst[i])
    for (int k = rs + lane; k < re; k += 32) {
        const int j = col[k];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            float z = a_src[j * H + h] + adst[h];
            z = z > 0.f ? z : z * slope;
            m[h] = fmaxf(m[h], z);
        }
    }
#pragma unroll
    for (int h = 0; h < H; ++h) m[h] = warp_max(m[h]);
    // pass 2: p = exp(e - max), row sum; park p in alpha
    for (int k = rs + lane; k < re; k += 32) {
        const int j = col[k];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            float z = a_src[j * H + h] + adst[h];
            z = z > 0.f ? z : z * slope;
            const float p = expf(z - m[h]);
            s[h] += p;
            alpha[(size_t)k * H + h] = p;
        }
    }
    float inv[H];
#pragma unroll
    for (int h = 0; h < H; ++h) inv[h] = 1.0f / (warp_sum(s[h]) + 1e-16f);
    // pass 3: normalise, save alpha, gather-SpMM in CSR order
    float4 acc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int base = rs; base < re; base += 32) {
        const int k = base + lane;
        int myj = 0;
        float mya[H];
#pragma unroll
        for (int h = 0; h < H; ++h) mya[h] = 0.f;
        if (k < re) {
            myj = col[k];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                mya[h] = alpha[(size_t)k * H + h] * inv[h];
                alpha[(size_t)k * H + h] = mya[h];
            }
        }
        const int cnt = min(32, re - base);
        for (int t = 0; t < cnt; t += 4) {
            int j[4];
            float a[4][H];
            float4 v[4][Q];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                j[u] = __shfl_sync(0xffffffffu, myj, (t + u) & 31);
#pragma unroll
                for (int h = 0; h < H; ++h) a[u][h] = __shfl_sync(0xffffffffu, mya[h], (t + u) & 31);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) v[u][q] = ldg_f4(xl + (size_t)j[u] * F + q * 128 + lane * 4);
                }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) fma4(acc[q], a[u][q / QH], v[u][q]);
                }
        }
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 b = ldg_f4(bias + q * 128 + lane * 4);
        float4 o = acc[q];
        o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
        *reinterpret_cast<float4*>(out + (size_t)i * F + q * 128 + lane * 4) = o;
    }
}

// ------------------------------------------------------------------ GAT backward, step 1 (per target row i)
// da_k = <g_i, xl_j>_head ; de_k = a_k (da_k - sum_k' a_k' da_k') ; dz_k = de_k * leaky'(z_k)
// outputs dz [nnz,H] and d_a_dst[i,h] = sum_k dz_k
template <int H, int Q>
__global__ void __launch_bounds__(256) gat_bwd_edge_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                           const float* __restrict__ xl, const float* __restrict__ a_src,
                                                           const float* __restrict__ a_dst, const float* __restrict__ alpha,
                                                           const float* __restrict__ gout, float slope, int n,
                                                           float* __restrict__ dz, float* __restrict__ d_a_dst) {
    constexpr int F = Q * 128, QH = Q / H;
    const int i = blockIdx.x * kRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const int rs = rowptr[i], re = rowptr[i + 1];
    float4 g[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) g[q] = ldg_f4(gout + (size_t)i * F + q * 128 + lane * 4);
    float dotsum[H];
#pragma unroll
    for (int h = 0; h < H; ++h) dotsum[h] = 0.f;
    // pass 1: da_k = <g_i, xl_j>_head for every entry.  Four entries at a time: each lane holds its
    // 16-channel partial of 4 x H dot products, which are reduced across the warp by a
    // transpose-reduce butterfly (4 -> 2 -> 1 values over xor 16 / 8, then xor 4 / 2 / 1): 6 shuffles
    // per head per 4 entries instead of 20, plus one shuffle to hand each sum to the lane that owns
    // the entry.
    for (int base = rs; base < re; base += 32) {
        const int k = base + lane;
        const int myj = k < re ? col[k] : 0;
        const int cnt = min(32, re - base);
        float myda[H];
#pragma unroll
        for (int h = 0; h < H; ++h) myda[h] = 0.f;
        for (int t = 0; t < cnt; t += 4) {
            float4 v[4][Q];
            int j[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) j[u] = __shfl_sync(0xffffffffu, myj, (t + u) & 31);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) v[u][q] = ldg_f4(xl + (size_t)j[u] * F + q * 128 + lane * 4);
                }
            }
            float part[4][H];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
#pragma unroll
                for (int h = 0; h < H; ++h) part[u][h] = 0.f;
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) part[u][q / QH] += dot4(g[q], v[u][q]);
                }
            }
            const bool up16 = (lane & 16) != 0, up8 = (lane & 8) != 0;
            const int e = lane - t;  // entry of this group owned by this lane (valid for 0 <= e < 4)
            const int src = ((e >> 1) & 1) << 4 | (e & 1) << 3;
#pragma unroll
            for (int h = 0; h < H; ++h) {
                // entries {0,1} end up in lanes with bit 4 clear, {2,3} in lanes with bit 4 set
                float w0 = (up16 ? part[2][h] : part[0][h]) + __shfl_xor_sync(0xffffffffu, up16 ? part[0][h] : part[2][h], 16);
                float w1 = (up16 ? part[3][h] : part[1][h]) + __shfl_xor_sync(0xffffffffu, up16 ? part[1][h] : part[3][h], 16);
                float x = (up8 ? w1 : w0) + __shfl_xor_sync(0xffffffffu, up8 ? w0 : w1, 8);
                x += __shfl_xor_sync(0xffffffffu, x, 4);
                x += __shfl_xor_sync(0xffffffffu, x, 2);
                x += __shfl_xor_sync(0xffffffffu, x, 1);
                const float d = __shfl_sync(0xffffffffu, x, src & 31);
                if (e >= 0 && e < 4) myda[h] = d;
            }
        }
        if (k < re) {
#pragma unroll
            for (int h = 0; h < H; ++h) {
                dz[(size_t)k * H + h] = myda[h];
                dotsum[h] += alpha[(size_t)k * H + h] * myda[h];
            }
        }
    }
#pragma unroll
    for (int h = 0; h < H; ++h) dotsum[h] = warp_sum(dotsum[h]);
    // pass 2: softmax + leaky-relu backward
    float adst[H], sdst[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        adst[h] = a_dst[i * H + h];
        sdst[h] = 0.f;
    }
    for (int k = rs + lane; k < re; k += 32) {
        const int j = col[k];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float a = alpha[(size_t)k * H + h];
            const float de = a * (dz[(size_t)k * H + h] - dotsum[h]);
            const float z = a_src[j * H + h] + adst[h];
            const float d = z > 0.f ? de : de * slope;
            dz[(size_t)k * H + h] = d;
            sdst[h] += d;
        }
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float t = warp_sum(sdst[h]);
        if (lane == 0) d_a_dst[i * H + h] = t;
    }
}

// ------------------------------------------------------------------ GAT backward, step 2 (per source row j)
// dxl[j,:] = sum_{i in N(j)} a_ij g_i + d_a_src[j] att_l + d_a_dst[j] att_r ; d_a_src[j,h] = sum_i dz_ij
// entry k' = (j,i) of row j <-> transposed entry perm[k'] = (i,j)
template <int H, int Q>
__global__ void __launch_bounds__(256) gat_bwd_node_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                           const int32_t* __restrict__ perm, const float* __restrict__ alpha,
                                                           const float* __restrict__ dz, const float* __restrict__ gout,
                                                           const float* __restrict__ att_l, const float* __restrict__ att_r,
                                                           const float* __restrict__ d_a_dst, int n, float* __restrict__ d_a_src,
                                                           float* __restrict__ dxl) {
    constexpr int F = Q * 128, QH = Q / H;
    const int jn = blockIdx.x * kRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (jn >= n) return;
    const int rs = rowptr[jn], re = rowptr[jn + 1];
    float4 acc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    float ssrc[H];
#pragma unroll
    for (int h = 0; h < H; ++h) ssrc[h] = 0.f;
    for (int base = rs; base < re; base += 32) {
        const int k = base + lane;
        int myi = 0;
        float mya[H];
#pragma unroll
        for (int h = 0; h < H; ++h) mya[h] = 0.f;
        if (k < re) {
            myi = col[k];
            const int kt = perm[k];
#pragma unroll
            for (int h = 0; h < H; ++h) {
                mya[h] = alpha[(size_t)kt * H + h];
                ssrc[h] += dz[(size_t)kt * H + h];
            }
        }
        const int cnt = min(32, re - base);
        for (int t = 0; t < cnt; t += 4) {
            int ii[4];
            float a[4][H];
            float4 v[4][Q];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                ii[u] = __shfl_sync(0xffffffffu, myi, (t + u) & 31);
#pragma unroll
                for (int h = 0; h < H; ++h) a[u][h] = __shfl_sync(0xffffffffu, mya[h], (t + u) & 31);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) v[u][q] = ldg_f4(gout + (size_t)ii[u] * F + q * 128 + lane * 4);
                }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) fma4(acc[q], a[u][q / QH], v[u][q]);
                }
        }
    }
    float dsrc[H], ddst[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        dsrc[h] = warp_sum(ssrc[h]);
        ddst[h] = d_a_dst[jn * H + h];
        if (lane == 0) d_a_src[jn * H + h] = dsrc[h];
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 al = ldg_f4(att_l + q * 128 + lane * 4), ar = ldg_f4(att_r + q * 128 + lane * 4);
        float4 o = acc[q];
        const float s = dsrc[q / QH], d = ddst[q / QH];
        o.x += s * al.x + d * ar.x;
        o.y += s * al.y + d * ar.y;
        o.z += s * al.z + d * ar.z;
        o.w += s * al.w + d * ar.w;
        *reinterpret_cast<float4*>(dxl + (size_t)jn * F + q * 128 + lane * 4) = o;
    }
}

// ------------------------------------------------------------------ GAT backward, ONE gather pass (default)
// The split backward above gathers 2 KB per edge twice (xl_j per target row, g_i per source row): 2 x 51 GB
// through L1/L2 at 50k loci.  Both can be had from the source side alone:
//   * the softmax row term  sum_k a_ik da_ik = <g_i, out_i - bias>_head  needs no gather at all
//     (gat_bwd_rowdot_kernel, one row-wise pass over g and the saved forward output);
//   * for source row j and its neighbour i (entry k' = (j,i), transposed entry kt = perm[k'] = (i,j)) the
//     gathered g_i serves BOTH the accumulation  dxl_j += a_ij g_i  and the logit gradient
//     da_ij = <g_i, xl_j>_head (xl_j sits in this warp's registers), from which dz_ij follows on the lane that
//     owns the entry.  d a_src[j] = sum_i dz_ij accumulates on the spot; dz_ij is stored at kt so that
//     d a_dst[i] = sum_j dz_ij becomes a contiguous row sum (gat_bwd_dst_kernel, which also adds the
//     d a_dst[i] att_r term to dxl_i).
// Same summation orders as the split kernels except for the row term (a dot product of two rows instead of a
// sum over the row's edges): ~1e-7 relative.
template <int H, int Q>
__global__ void __launch_bounds__(256) gat_bwd_rowdot_kernel(const float* __restrict__ gout, const float* __restrict__ out,
                                                             const float* __restrict__ bias, int n, float* __restrict__ rowdot) {
    constexpr int F = Q * 128, QH = Q / H;
    const int i = blockIdx.x * kRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    float s[H];
#pragma unroll
    for (int h = 0; h < H; ++h) s[h] = 0.f;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 g = ldg_f4(gout + (size_t)i * F + q * 128 + lane * 4);
        float4 o = ldg_f4(out + (size_t)i * F + q * 128 + lane * 4);
        const float4 b = ldg_f4(bias + q * 128 + lane * 4);
        o.x -= b.x; o.y -= b.y; o.z -= b.z; o.w -= b.w;
        s[q / QH] += dot4(g, o);
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float t = warp_sum(s[h]);
        if (lane == 0) rowdot[i * H + h] = t;
    }
}

// Row block [g0, g1) (kRows): only the targets i of the block contribute to source row jn.  The columns of row jn are sorted, so
// they are the contiguous entries ranges[jn] = [lower_bound(g0), lower_bound(g1)) (gat_block_ranges_kernel).  alpha / dz / rowdot /
// gout hold the block's entries / rows only: the host passes them offset back by rowptr[g0] entries / g0 rows, so that entry k and
// row i index them unchanged.  kRows = false is the whole graph, without the range table.
template <int H, int Q, int W, bool kRows>
__global__ void __launch_bounds__(W * 32, 16 / W) gat_bwd_fused_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                               const int32_t* __restrict__ perm, const float* __restrict__ xl,
                                                               const float* __restrict__ a_src, const float* __restrict__ a_dst,
                                                               const float* __restrict__ alpha, const float* __restrict__ rowdot,
                                                               const float* __restrict__ gout, const float* __restrict__ att_l, float slope,
                                                               int n, const int2* __restrict__ ranges, float* __restrict__ dz,
                                                               float* __restrict__ d_a_src, float* __restrict__ dxl) {
    constexpr int F = Q * 128, QH = Q / H;
    const int jn = blockIdx.x * W + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (jn >= n) return;
    int rs, re;
    if constexpr (kRows) {
        const int2 r = ranges[jn];
        rs = r.x;
        re = r.y;
    } else {
        rs = rowptr[jn];
        re = rowptr[jn + 1];
    }
    float4 x[Q], acc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        x[q] = ldg_f4(xl + (size_t)jn * F + q * 128 + lane * 4);
        acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float asrc[H], ssrc[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        asrc[h] = a_src[jn * H + h];
        ssrc[h] = 0.f;
    }
    for (int base = rs; base < re; base += 32) {
        const int k = base + lane;
        int myi = 0, mykt = 0;
        float mya[H], myda[H];
#pragma unroll
        for (int h = 0; h < H; ++h) mya[h] = myda[h] = 0.f;
        if (k < re) {
            myi = col[k];
            mykt = perm[k];
#pragma unroll
            for (int h = 0; h < H; ++h) mya[h] = alpha[(size_t)mykt * H + h];
        }
        const int cnt = min(32, re - base);
        for (int t = 0; t < cnt; t += 4) {
            int ii[4];
            float a[4][H];
            float4 v[4][Q];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                ii[u] = __shfl_sync(0xffffffffu, myi, (t + u) & 31);
#pragma unroll
                for (int h = 0; h < H; ++h) a[u][h] = __shfl_sync(0xffffffffu, mya[h], (t + u) & 31);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) v[u][q] = ldg_f4(gout + (size_t)ii[u] * F + q * 128 + lane * 4);
                }
            float part[4][H];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
#pragma unroll
                for (int h = 0; h < H; ++h) part[u][h] = 0.f;
                if (t + u < cnt) {
#pragma unroll
                    for (int q = 0; q < Q; ++q) {
                        part[u][q / QH] += dot4(x[q], v[u][q]);
                        fma4(acc[q], a[u][q / QH], v[u][q]);
                    }
                }
            }
            // transpose-reduce butterfly of the 4 x H partial dot products (see gat_bwd_edge_kernel)
            const bool up16 = (lane & 16) != 0, up8 = (lane & 8) != 0;
            const int e = lane - t;  // entry of this group owned by this lane (valid for 0 <= e < 4)
            const int src = ((e >> 1) & 1) << 4 | (e & 1) << 3;
#pragma unroll
            for (int h = 0; h < H; ++h) {
                float w0 = (up16 ? part[2][h] : part[0][h]) + __shfl_xor_sync(0xffffffffu, up16 ? part[0][h] : part[2][h], 16);
                float w1 = (up16 ? part[3][h] : part[1][h]) + __shfl_xor_sync(0xffffffffu, up16 ? part[1][h] : part[3][h], 16);
                float y = (up8 ? w1 : w0) + __shfl_xor_sync(0xffffffffu, up8 ? w0 : w1, 8);
                y += __shfl_xor_sync(0xffffffffu, y, 4);
                y += __shfl_xor_sync(0xffffffffu, y, 2);
                y += __shfl_xor_sync(0xffffffffu, y, 1);
                const float d = __shfl_sync(0xffffffffu, y, src & 31);
                if (e >= 0 && e < 4) myda[h] = d;
            }
        }
        if (k < re) {  // softmax + leaky-relu backward on the lane that owns the entry
#pragma unroll
            for (int h = 0; h < H; ++h) {
                const float de = mya[h] * (myda[h] - rowdot[myi * H + h]);
                const float z = asrc[h] + a_dst[myi * H + h];
                const float d = z > 0.f ? de : de * slope;
                dz[(size_t)mykt * H + h] = d;
                ssrc[h] += d;
            }
        }
    }
    float dsrc[H];
#pragma unroll
    for (int h = 0; h < H; ++h) {
        dsrc[h] = warp_sum(ssrc[h]);
        if (lane == 0) d_a_src[jn * H + h] = dsrc[h];
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 al = ldg_f4(att_l + q * 128 + lane * 4);
        float4 o = acc[q];
        const float sc = dsrc[q / QH];
        o.x += sc * al.x; o.y += sc * al.y; o.z += sc * al.z; o.w += sc * al.w;
        *reinterpret_cast<float4*>(dxl + (size_t)jn * F + q * 128 + lane * 4) = o;
    }
}

// ranges[j] = the entries of row j whose column lies in [g0, g1): [lower_bound(g0), lower_bound(g1)) on the sorted columns
__global__ void __launch_bounds__(256) gat_block_ranges_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int n,
                                                               int g0, int g1, int2* __restrict__ ranges) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= n) return;
    const int rs = rowptr[j], re = rowptr[j + 1];
    const int lo = lower_bound_i32(col, rs, re, g0);
    ranges[j] = make_int2(lo, lower_bound_i32(col, lo, re, g1));
}

// d a_dst[i,h] = sum of the row's dz (contiguous), then dxl[i,:] += d a_dst[i,h] att_r; rows i of the block [g0, g1) (dz offset
// back by the host like in gat_bwd_fused_kernel)
template <int H, int Q>
__global__ void __launch_bounds__(256) gat_bwd_dst_kernel(const int32_t* __restrict__ rowptr, const float* __restrict__ dz,
                                                          const float* __restrict__ att_r, int g0, int g1, float* __restrict__ d_a_dst,
                                                          float* __restrict__ dxl) {
    constexpr int F = Q * 128, QH = Q / H;
    const int i = g0 + blockIdx.x * kRowsPerCta + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= g1) return;
    const int rs = rowptr[i], re = rowptr[i + 1];
    float s[H];
#pragma unroll
    for (int h = 0; h < H; ++h) s[h] = 0.f;
    for (int k = rs + lane; k < re; k += 32) {
#pragma unroll
        for (int h = 0; h < H; ++h) s[h] += dz[(size_t)k * H + h];
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        s[h] = warp_sum(s[h]);
        if (lane == 0) d_a_dst[i * H + h] = s[h];
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const float4 ar = ldg_f4(att_r + q * 128 + lane * 4);
        float4* p = reinterpret_cast<float4*>(dxl + (size_t)i * F + q * 128 + lane * 4);
        float4 o = *p;
        const float d = s[q / QH];
        o.x += d * ar.x; o.y += d * ar.y; o.z += d * ar.z; o.w += d * ar.w;
        *p = o;
    }
}

// ------------------------------------------------------------------ GAT backward, step 3 (parameter grads)
// datt_l[c] = sum_j d_a_src[j,h(c)] xl[j,c] ; datt_r[c] = sum_j d_a_dst[j,h(c)] xl[j,c] ; dbias[c] = sum_i g[i,c]
// stage A: kParamCtas CTAs stride over the rows (float4 per thread, two rows in flight) and keep their sums in
// registers; partials are stored TRANSPOSED, part[(k*F + c) * nblk + blk], so that stage B -- one warp per
// output value, lanes striding the nblk partials, fixed order -- reads them coalesced.  Deterministic.
constexpr int kParamRows = 64;   // kept for the workspace formula (upper bound of the partial count)
constexpr int kParamCtas = 148 * 8;  // 4 warps each: ~32 warps per SM keep enough 16-byte loads in flight for a 204 MB stream
__global__ void __launch_bounds__(128) gat_bwd_param_kernel(const float* __restrict__ xl, const float* __restrict__ gout,
                                                            const float* __restrict__ d_a_src, const float* __restrict__ d_a_dst,
                                                            int n, int H, int C, float* __restrict__ part) {
    const int F = H * C, nblk = gridDim.x, blk = blockIdx.x;
    for (int c = threadIdx.x * 4; c < F; c += blockDim.x * 4) {
        const int h = c / C;
        float4 sl = make_float4(0.f, 0.f, 0.f, 0.f), sr = sl, sb = sl;
        int r = blk;
        for (; r + nblk < n; r += 2 * nblk) {
            const float4 x0 = __ldg(reinterpret_cast<const float4*>(xl + (size_t)r * F + c));
            const float4 x1 = __ldg(reinterpret_cast<const float4*>(xl + (size_t)(r + nblk) * F + c));
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gout + (size_t)r * F + c));
            const float4 g1 = __ldg(reinterpret_cast<const float4*>(gout + (size_t)(r + nblk) * F + c));
            const float s0 = d_a_src[r * H + h], t0 = d_a_dst[r * H + h], s1 = d_a_src[(r + nblk) * H + h], t1 = d_a_dst[(r + nblk) * H + h];
            fma4(sl, s0, x0); fma4(sr, t0, x0); sb.x += g0.x; sb.y += g0.y; sb.z += g0.z; sb.w += g0.w;
            fma4(sl, s1, x1); fma4(sr, t1, x1); sb.x += g1.x; sb.y += g1.y; sb.z += g1.z; sb.w += g1.w;
        }
        if (r < n) {
            const float4 x0 = __ldg(reinterpret_cast<const float4*>(xl + (size_t)r * F + c));
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gout + (size_t)r * F + c));
            fma4(sl, d_a_src[r * H + h], x0); fma4(sr, d_a_dst[r * H + h], x0);
            sb.x += g0.x; sb.y += g0.y; sb.z += g0.z; sb.w += g0.w;
        }
        const float vl[4] = {sl.x, sl.y, sl.z, sl.w}, vr[4] = {sr.x, sr.y, sr.z, sr.w}, vb[4] = {sb.x, sb.y, sb.z, sb.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            part[((size_t)(0 * F + c + q)) * nblk + blk] = vl[q];
            part[((size_t)(1 * F + c + q)) * nblk + blk] = vr[q];
            part[((size_t)(2 * F + c + q)) * nblk + blk] = vb[q];
        }
    }
}

// Stage A of a row block [g0, g1): datt_l runs over all n rows (d a_src is a partial sum on every row), datt_r and dbias over the
// block's rows only (gout offset back by g0 rows by the host; d a_dst is read on the block's rows).  Same partial layout.
__global__ void __launch_bounds__(128) gat_bwd_param_rows_kernel(const float* __restrict__ xl, const float* __restrict__ gout,
                                                                 const float* __restrict__ d_a_src, const float* __restrict__ d_a_dst,
                                                                 int n, int g0, int g1, int H, int C, float* __restrict__ part) {
    const int F = H * C, nblk = gridDim.x, blk = blockIdx.x;
    for (int c = threadIdx.x * 4; c < F; c += blockDim.x * 4) {
        const int h = c / C;
        float4 sl = make_float4(0.f, 0.f, 0.f, 0.f), sr = sl, sb = sl;
        for (int r = blk; r < n; r += nblk) fma4(sl, d_a_src[r * H + h], __ldg(reinterpret_cast<const float4*>(xl + (size_t)r * F + c)));
        for (int r = g0 + blk; r < g1; r += nblk) {
            const float4 x0 = __ldg(reinterpret_cast<const float4*>(xl + (size_t)r * F + c));
            const float4 g = __ldg(reinterpret_cast<const float4*>(gout + (size_t)r * F + c));
            fma4(sr, d_a_dst[r * H + h], x0);
            sb.x += g.x; sb.y += g.y; sb.z += g.z; sb.w += g.w;
        }
        const float vl[4] = {sl.x, sl.y, sl.z, sl.w}, vr[4] = {sr.x, sr.y, sr.z, sr.w}, vb[4] = {sb.x, sb.y, sb.z, sb.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            part[((size_t)(0 * F + c + q)) * nblk + blk] = vl[q];
            part[((size_t)(1 * F + c + q)) * nblk + blk] = vr[q];
            part[((size_t)(2 * F + c + q)) * nblk + blk] = vb[q];
        }
    }
}

__global__ void __launch_bounds__(256) gat_bwd_param_reduce_kernel(const float* __restrict__ part, int nblk, int F,
                                                                   float* __restrict__ datt_l, float* __restrict__ datt_r, float* __restrict__ dbias) {
    const int o = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (o >= 3 * F) return;
    float s = 0.f;
    for (int k = lane; k < nblk; k += 32) s += part[(size_t)o * nblk + k];
    s = warp_sum(s);
    if (lane == 0) {
        if (o < F) datt_l[o] = s;
        else if (o < 2 * F) datt_r[o - F] = s;
        else dbias[o - 2 * F] = s;
    }
}

int param_ctas(int64_t n) { return (int)(n < kParamCtas ? n : kParamCtas); }

// warps (= consecutive rows) per CTA of the two gather kernels (gat_fwd / gat_bwd_fused): 8 or 16, see hicgat_gat_set_tuning
int g_gather_warps = 8;
// bytes of L2 set aside for the GATHERED matrix (xl in the forward, gout in the backward): 0 = off
size_t g_l2_persist_bytes = 0;

// Launch of a gather kernel; with g_l2_persist_bytes > 0 the gathered matrix gets a persisting access-policy window (launch
// attribute, nothing is changed on the caller's stream), so that the streamed col / alpha / output traffic does not evict it.
template <typename... KArgs, typename... Args>
void launch_gather(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t stream, const void* gathered, size_t bytes, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    if (g_l2_persist_bytes > 0 && bytes > 0) {
        attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[0].val.accessPolicyWindow.base_ptr = const_cast<void*>(gathered);
        attr[0].val.accessPolicyWindow.num_bytes = bytes;
        attr[0].val.accessPolicyWindow.hitRatio = bytes <= g_l2_persist_bytes ? 1.0f : (float)((double)g_l2_persist_bytes / (double)bytes);
        attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

#define HICGAT_DISPATCH_HQ(H, C, CALL)                              \
    do {                                                            \
        const int q__ = (H) * (C) / 128;                            \
        if ((H) == 1 && q__ == 1) { CALL(1, 1); }                   \
        else if ((H) == 1 && q__ == 2) { CALL(1, 2); }              \
        else if ((H) == 1 && q__ == 4) { CALL(1, 4); }              \
        else if ((H) == 2 && q__ == 2) { CALL(2, 2); }              \
        else if ((H) == 2 && q__ == 4) { CALL(2, 4); }              \
        else if ((H) == 2 && q__ == 8) { CALL(2, 8); }              \
        else if ((H) == 4 && q__ == 4) { CALL(4, 4); }              \
        else if ((H) == 4 && q__ == 8) { CALL(4, 8); }              \
        else { set_error("GAT: unsupported heads=%d channels=%d", (H), (C)); return HICGAT_ERR_INVALID; } \
    } while (0)

}  // namespace
}  // namespace hicgat

using namespace hicgat;

namespace {
int spmm_rows(const char* fn, const int32_t* rowptr, const int32_t* col, const float* w, const float* x, int64_t n, int64_t g0, int64_t g1,
              int64_t f, float* out, cudaStream_t stream) {
    HICGAT_REQUIRE(rowptr && col && w && x && n > 0 && n < (1ll << 31), "%s: bad arguments", fn);
    HICGAT_REQUIRE(0 <= g0 && g0 <= g1 && g1 <= n, "%s: bad row block [%lld, %lld) of n = %lld", fn, (long long)g0, (long long)g1, (long long)n);
    HICGAT_REQUIRE(out || g0 == g1, "%s: null out", fn);
    HICGAT_REQUIRE(aligned16(x) && aligned16(out), "%s: x/out must be 16-byte aligned", fn);
    if (f != 128 && f != 256 && f != 512 && f != 1024) {
        set_error("%s: feature width %lld not in {128,256,512,1024}", fn, (long long)f);
        return HICGAT_ERR_INVALID;
    }
    if (g0 == g1) return HICGAT_OK;
    const unsigned grid = (unsigned)((g1 - g0 + kRowsPerCta - 1) / kRowsPerCta);
    switch (f) {
        case 128: spmm_kernel<1><<<grid, 256, 0, stream>>>(rowptr, col, w, x, (int)g0, (int)g1, out); break;
        case 256: spmm_kernel<2><<<grid, 256, 0, stream>>>(rowptr, col, w, x, (int)g0, (int)g1, out); break;
        case 512: spmm_kernel<4><<<grid, 256, 0, stream>>>(rowptr, col, w, x, (int)g0, (int)g1, out); break;
        default: spmm_kernel<8><<<grid, 256, 0, stream>>>(rowptr, col, w, x, (int)g0, (int)g1, out); break;
    }
    HICGAT_CHECK_LAUNCH("spmm_kernel");
    return HICGAT_OK;
}
}  // namespace

extern "C" int hicgat_spmm_csr_f32(const int32_t* rowptr, const int32_t* col, const float* w, const float* x, int64_t n,
                                   int64_t f, float* out, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(out, "hicgat_spmm_csr_f32: bad arguments");
    return spmm_rows("hicgat_spmm_csr_f32", rowptr, col, w, x, n, 0, n, f, out, static_cast<cudaStream_t>(stream_));
}

extern "C" int hicgat_spmm_csr_rows_f32(const int32_t* rowptr, const int32_t* col, const float* w, const float* x, int64_t n, int64_t g0,
                                        int64_t g1, int64_t f, float* out, hicgat_stream_t stream_) {
    return spmm_rows("hicgat_spmm_csr_rows_f32", rowptr, col, w, x, n, g0, g1, f, out, static_cast<cudaStream_t>(stream_));
}

extern "C" int hicgat_gat_set_tuning(int rows_per_cta, int l2_persist_mb) {
    HICGAT_REQUIRE(rows_per_cta == 8 || rows_per_cta == 16, "hicgat_gat_set_tuning: rows_per_cta must be 8 or 16");
    HICGAT_REQUIRE(l2_persist_mb >= 0, "hicgat_gat_set_tuning: l2_persist_mb must be >= 0");
    size_t bytes = (size_t)l2_persist_mb << 20;
    if (bytes > 0) {  // device-wide carve-out of L2 for persisting lines (current device), capped by what the device allows
        int dev = 0, max_persist = 0, max_window = 0;
        HICGAT_CUDA(cudaGetDevice(&dev));
        HICGAT_CUDA(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev));
        HICGAT_CUDA(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev));
        bytes = std::min(bytes, (size_t)max_persist);
        HICGAT_REQUIRE(bytes > 0 && max_window > 0, "hicgat_gat_set_tuning: the device has no persisting L2 carve-out");
        HICGAT_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes));
    } else if (g_l2_persist_bytes > 0) {
        HICGAT_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0));
        HICGAT_CUDA(cudaCtxResetPersistingL2Cache());
    }
    g_gather_warps = rows_per_cta;
    g_l2_persist_bytes = bytes;
    return HICGAT_OK;
}

namespace {
int gat_fwd_rows(const char* fn, const int32_t* rowptr, const int32_t* col, int64_t n, int64_t g0, int64_t g1, int64_t e0, int heads, int channels,
                 const float* xl, const float* att_l, const float* att_r, const float* bias, float slope, float* a_src, float* a_dst,
                 float* alpha, float* out, cudaStream_t stream) {
    HICGAT_REQUIRE(rowptr && col && xl && att_l && att_r && bias && a_src && a_dst, "%s: null pointer", fn);
    HICGAT_REQUIRE(n > 0 && n < (1ll << 31), "%s: bad n", fn);
    HICGAT_REQUIRE(0 <= g0 && g0 <= g1 && g1 <= n && e0 >= 0, "%s: bad row block [%lld, %lld) of n = %lld", fn, (long long)g0, (long long)g1, (long long)n);
    HICGAT_REQUIRE((alpha && out) || g0 == g1, "%s: null pointer", fn);
    HICGAT_REQUIRE(gat_shape_supported(heads, channels), "%s: unsupported heads=%d channels=%d", fn, heads, channels);
    HICGAT_REQUIRE(aligned16(xl) && aligned16(out) && aligned16(att_l) && aligned16(att_r) && aligned16(bias), "%s: 16-byte alignment required", fn);
    const unsigned grid = (unsigned)((n + kRowsPerCta - 1) / kRowsPerCta);
#define CALL_LOGIT(H, Q) gat_logit_kernel<H, Q><<<grid, 256, 0, stream>>>(xl, att_l, att_r, (int)n, a_src, a_dst)
    HICGAT_DISPATCH_HQ(heads, channels, CALL_LOGIT);
#undef CALL_LOGIT
    HICGAT_CHECK_LAUNCH("gat_logit_kernel");
    if (g0 == g1) return HICGAT_OK;
    const int64_t nb = g1 - g0;
    // the kernel indexes entry k / row i of the whole graph: offset the block's arrays back by e0 entries / g0 rows
    float* const alpha_b = alpha - e0 * heads;
    float* const out_b = out - g0 * heads * channels;
    const size_t gathered_bytes = (size_t)n * heads * channels * sizeof(float);
#define CALL_FWD(H, Q)                                                                                                                  \
    if (g_gather_warps == 16) launch_gather(gat_fwd_kernel<H, Q, 16>, (unsigned)((nb + 15) / 16), 512, stream, xl, gathered_bytes, rowptr, col, xl, a_src, a_dst, bias, slope, (int)g0, (int)g1, alpha_b, out_b); \
    else launch_gather(gat_fwd_kernel<H, Q, 8>, (unsigned)((nb + kRowsPerCta - 1) / kRowsPerCta), 256, stream, xl, gathered_bytes, rowptr, col, xl, a_src, a_dst, bias, slope, (int)g0, (int)g1, alpha_b, out_b)
    HICGAT_DISPATCH_HQ(heads, channels, CALL_FWD);
#undef CALL_FWD
    HICGAT_CHECK_LAUNCH("gat_fwd_kernel");
    return HICGAT_OK;
}
}  // namespace

extern "C" int hicgat_gat_fwd(const int32_t* rowptr, const int32_t* col, int64_t n, int heads, int channels, const float* xl,
                              const float* att_l, const float* att_r, const float* bias, float slope, float* a_src,
                              float* a_dst, float* alpha, float* out, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(alpha && out, "hicgat_gat_fwd: null pointer");
    return gat_fwd_rows("hicgat_gat_fwd", rowptr, col, n, 0, n, 0, heads, channels, xl, att_l, att_r, bias, slope, a_src, a_dst, alpha, out,
                        static_cast<cudaStream_t>(stream_));
}

extern "C" int hicgat_gat_fwd_rows(const int32_t* rowptr, const int32_t* col, int64_t n, int64_t g0, int64_t g1, int64_t e0, int heads, int channels,
                                   const float* xl, const float* att_l, const float* att_r, const float* bias, float slope, float* a_src,
                                   float* a_dst, float* alpha, float* out, hicgat_stream_t stream_) {
    return gat_fwd_rows("hicgat_gat_fwd_rows", rowptr, col, n, g0, g1, e0, heads, channels, xl, att_l, att_r, bias, slope, a_src, a_dst, alpha, out,
                        static_cast<cudaStream_t>(stream_));
}

namespace {
struct BwdLayout {
    size_t off_dz, off_dsrc, off_ddst, off_rowdot, off_part, off_ranges, off_counter, total;
    int nchunks;
};
BwdLayout bwd_layout(int64_t n, int64_t nnz, int H, int C) {
    BwdLayout L;
    const size_t F = (size_t)H * C;
    L.nchunks = (int)((n + kParamRows - 1) / kParamRows);
    L.off_counter = 0;
    L.off_dz = 256;
    L.off_dsrc = L.off_dz + align_up(sizeof(float) * (size_t)nnz * H, 256);
    L.off_ddst = L.off_dsrc + align_up(sizeof(float) * (size_t)n * H, 256);
    L.off_rowdot = L.off_ddst + align_up(sizeof(float) * (size_t)n * H, 256);
    L.off_part = L.off_rowdot + align_up(sizeof(float) * (size_t)n * H, 256);
    L.off_ranges = L.off_part + align_up(sizeof(float) * 3 * F * (size_t)param_ctas(n), 256);
    L.total = L.off_ranges + sizeof(int2) * (size_t)n;  // row-block calls only
    return L;
}
}  // namespace

extern "C" size_t hicgat_gat_bwd_workspace_bytes(int64_t n, int64_t nnz, int heads, int channels) {
    if (n <= 0 || nnz < 0 || !gat_shape_supported(heads, channels)) return 0;
    return bwd_layout(n, nnz, heads, channels).total;
}

extern "C" int hicgat_gat_bwd(const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n, int64_t nnz, int heads,
                              int channels, const float* xl, const float* att_l, const float* att_r, float slope,
                              const float* a_src, const float* a_dst, const float* alpha, const float* gout, float* dxl,
                              float* datt_l, float* datt_r, float* dbias, void* workspace, size_t workspace_bytes,
                              hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(rowptr && col && perm && xl && att_l && att_r && a_src && a_dst && alpha && gout && dxl && datt_l && datt_r && dbias && workspace,
                   "hicgat_gat_bwd: null pointer");
    HICGAT_REQUIRE(n > 0 && n < (1ll << 31) && nnz >= 0 && nnz < (1ll << 31), "hicgat_gat_bwd: bad n/nnz");
    HICGAT_REQUIRE(gat_shape_supported(heads, channels), "hicgat_gat_bwd: unsupported heads=%d channels=%d", heads, channels);
    HICGAT_REQUIRE(aligned16(xl) && aligned16(gout) && aligned16(dxl) && aligned16(att_l) && aligned16(att_r), "hicgat_gat_bwd: 16-byte alignment required");
    const BwdLayout L = bwd_layout(n, nnz, heads, channels);
    if (workspace_bytes < L.total) {
        set_error("hicgat_gat_bwd: workspace %zu < required %zu", workspace_bytes, L.total);
        return HICGAT_ERR_WORKSPACE;
    }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* dz = reinterpret_cast<float*>(ws + L.off_dz);
    float* dsrc = reinterpret_cast<float*>(ws + L.off_dsrc);
    float* ddst = reinterpret_cast<float*>(ws + L.off_ddst);
    float* part = reinterpret_cast<float*>(ws + L.off_part);
    const unsigned grid = (unsigned)((n + kRowsPerCta - 1) / kRowsPerCta);
#define CALL_EDGE(H, Q) gat_bwd_edge_kernel<H, Q><<<grid, 256, 0, stream>>>(rowptr, col, xl, a_src, a_dst, alpha, gout, slope, (int)n, dz, ddst)
    HICGAT_DISPATCH_HQ(heads, channels, CALL_EDGE);
#undef CALL_EDGE
    HICGAT_CHECK_LAUNCH("gat_bwd_edge_kernel");
#define CALL_NODE(H, Q) gat_bwd_node_kernel<H, Q><<<grid, 256, 0, stream>>>(rowptr, col, perm, alpha, dz, gout, att_l, att_r, ddst, (int)n, dsrc, dxl)
    HICGAT_DISPATCH_HQ(heads, channels, CALL_NODE);
#undef CALL_NODE
    HICGAT_CHECK_LAUNCH("gat_bwd_node_kernel");
    const int nblk = param_ctas(n);
    gat_bwd_param_kernel<<<nblk, 128, 0, stream>>>(xl, gout, dsrc, ddst, (int)n, heads, channels, part);
    HICGAT_CHECK_LAUNCH("gat_bwd_param_kernel");
    gat_bwd_param_reduce_kernel<<<(3 * heads * channels + 7) / 8, 256, 0, stream>>>(part, nblk, heads * channels, datt_l, datt_r, dbias);
    HICGAT_CHECK_LAUNCH("gat_bwd_param_reduce_kernel");
    return HICGAT_OK;
}

namespace {
int gat_bwd_fused_rows(const char* fn, const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n, int64_t nnz, int64_t g0,
                       int64_t g1, int64_t e0, int heads, int channels, const float* xl, const float* att_l, const float* att_r, const float* bias,
                       float slope, const float* a_src, const float* a_dst, const float* alpha, const float* out, const float* gout,
                       float* dxl, float* datt_l, float* datt_r, float* dbias, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    HICGAT_REQUIRE(rowptr && col && perm && xl && att_l && att_r && bias && a_src && a_dst && dxl && datt_l && datt_r && dbias && workspace,
                   "%s: null pointer", fn);
    HICGAT_REQUIRE(n > 0 && n < (1ll << 31) && nnz >= 0 && nnz < (1ll << 31), "%s: bad n/nnz", fn);
    HICGAT_REQUIRE(0 <= g0 && g0 <= g1 && g1 <= n && 0 <= e0 && e0 <= nnz, "%s: bad row block [%lld, %lld) of n = %lld", fn, (long long)g0, (long long)g1,
                   (long long)n);
    HICGAT_REQUIRE((alpha && out && gout) || g0 == g1, "%s: null pointer", fn);
    HICGAT_REQUIRE(gat_shape_supported(heads, channels), "%s: unsupported heads=%d channels=%d", fn, heads, channels);
    HICGAT_REQUIRE(aligned16(xl) && aligned16(gout) && aligned16(out) && aligned16(dxl) && aligned16(att_l) && aligned16(att_r) && aligned16(bias),
                   "%s: 16-byte alignment required", fn);
    const BwdLayout L = bwd_layout(n, nnz, heads, channels);
    if (workspace_bytes < L.total) {
        set_error("%s: workspace %zu < required %zu", fn, workspace_bytes, L.total);
        return HICGAT_ERR_WORKSPACE;
    }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* dz = reinterpret_cast<float*>(ws + L.off_dz);
    float* dsrc = reinterpret_cast<float*>(ws + L.off_dsrc);
    float* ddst = reinterpret_cast<float*>(ws + L.off_ddst);
    float* rowdot = reinterpret_cast<float*>(ws + L.off_rowdot);
    float* part = reinterpret_cast<float*>(ws + L.off_part);
    const int64_t nb = g1 - g0, F = (int64_t)heads * channels;
    // the kernels index entry k / row i of the whole graph: the block's arrays are offset back by e0 entries / g0 rows
    const float* const alpha_b = alpha - e0 * heads;
    const float* const gout_b = gout - g0 * F;
    float* const dz_b = dz - e0 * heads;
    float* const rowdot_b = rowdot - g0 * heads;
    const bool whole = g0 == 0 && g1 == n;
    int2* const ranges = reinterpret_cast<int2*>(ws + L.off_ranges);
    const unsigned grid = (unsigned)((n + kRowsPerCta - 1) / kRowsPerCta), grid_b = (unsigned)((nb + kRowsPerCta - 1) / kRowsPerCta);
    if (nb > 0) {  // the block's rows: rowdot [nb, H] from the block's gout / out
#define CALL_ROWDOT(H, Q) gat_bwd_rowdot_kernel<H, Q><<<grid_b, 256, 0, stream>>>(gout, out, bias, (int)nb, rowdot)
        HICGAT_DISPATCH_HQ(heads, channels, CALL_ROWDOT);
#undef CALL_ROWDOT
        HICGAT_CHECK_LAUNCH("gat_bwd_rowdot_kernel");
    }
    if (!whole) {
        gat_block_ranges_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(rowptr, col, (int)n, (int)g0, (int)g1, ranges);
        HICGAT_CHECK_LAUNCH("gat_block_ranges_kernel");
    }
    // every source row j (dxl and d a_src are partial sums over the block's targets when the block is not all rows)
    const size_t gathered_bytes = (size_t)nb * heads * channels * sizeof(float);
#define LAUNCH_FUSED(H, Q, W, R, G, B) launch_gather(gat_bwd_fused_kernel<H, Q, W, R>, G, B, stream, gout, gathered_bytes, rowptr, col, perm, xl, a_src, a_dst, alpha_b, rowdot_b, gout_b, att_l, slope, (int)n, ranges, dz_b, dsrc, dxl)
#define CALL_FUSED(H, Q)                                                                                                                \
    if (g_gather_warps == 16 && whole) LAUNCH_FUSED(H, Q, 16, false, (unsigned)((n + 15) / 16), 512);                                   \
    else if (g_gather_warps == 16) LAUNCH_FUSED(H, Q, 16, true, (unsigned)((n + 15) / 16), 512);                                        \
    else if (whole) LAUNCH_FUSED(H, Q, 8, false, grid, 256);                                                                            \
    else LAUNCH_FUSED(H, Q, 8, true, grid, 256)
    HICGAT_DISPATCH_HQ(heads, channels, CALL_FUSED);
#undef CALL_FUSED
#undef LAUNCH_FUSED
    HICGAT_CHECK_LAUNCH("gat_bwd_fused_kernel");
    if (nb > 0) {
#define CALL_DST(H, Q) gat_bwd_dst_kernel<H, Q><<<grid_b, 256, 0, stream>>>(rowptr, dz_b, att_r, (int)g0, (int)g1, ddst, dxl)
        HICGAT_DISPATCH_HQ(heads, channels, CALL_DST);
#undef CALL_DST
        HICGAT_CHECK_LAUNCH("gat_bwd_dst_kernel");
    }
    const int nblk = param_ctas(n);
    if (g0 == 0 && g1 == n) {
        gat_bwd_param_kernel<<<nblk, 128, 0, stream>>>(xl, gout, dsrc, ddst, (int)n, heads, channels, part);
        HICGAT_CHECK_LAUNCH("gat_bwd_param_kernel");
    } else {
        gat_bwd_param_rows_kernel<<<nblk, 128, 0, stream>>>(xl, gout_b, dsrc, ddst, (int)n, (int)g0, (int)g1, heads, channels, part);
        HICGAT_CHECK_LAUNCH("gat_bwd_param_rows_kernel");
    }
    gat_bwd_param_reduce_kernel<<<(3 * heads * channels + 7) / 8, 256, 0, stream>>>(part, nblk, heads * channels, datt_l, datt_r, dbias);
    HICGAT_CHECK_LAUNCH("gat_bwd_param_reduce_kernel");
    return HICGAT_OK;
}
}  // namespace

extern "C" int hicgat_gat_bwd_fused(const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n, int64_t nnz, int heads,
                                    int channels, const float* xl, const float* att_l, const float* att_r, const float* bias, float slope,
                                    const float* a_src, const float* a_dst, const float* alpha, const float* out, const float* gout,
                                    float* dxl, float* datt_l, float* datt_r, float* dbias, void* workspace, size_t workspace_bytes,
                                    hicgat_stream_t stream_) {
    HICGAT_REQUIRE(alpha && out && gout, "hicgat_gat_bwd_fused: null pointer");
    return gat_bwd_fused_rows("hicgat_gat_bwd_fused", rowptr, col, perm, n, nnz, 0, n, 0, heads, channels, xl, att_l, att_r, bias, slope, a_src, a_dst,
                              alpha, out, gout, dxl, datt_l, datt_r, dbias, workspace, workspace_bytes, static_cast<cudaStream_t>(stream_));
}

extern "C" int hicgat_gat_bwd_fused_rows(const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n, int64_t nnz, int64_t g0,
                                         int64_t g1, int64_t e0, int heads, int channels, const float* xl, const float* att_l, const float* att_r,
                                         const float* bias, float slope, const float* a_src, const float* a_dst, const float* alpha,
                                         const float* out, const float* gout, float* dxl, float* datt_l, float* datt_r, float* dbias,
                                         void* workspace, size_t workspace_bytes, hicgat_stream_t stream_) {
    return gat_bwd_fused_rows("hicgat_gat_bwd_fused_rows", rowptr, col, perm, n, nnz, g0, g1, e0, heads, channels, xl, att_l, att_r, bias, slope, a_src,
                              a_dst, alpha, out, gout, dxl, datt_l, datt_r, dbias, workspace, workspace_bytes, static_cast<cudaStream_t>(stream_));
}

// ------------------------------------------------------------------ pieces shared with the dense-tile path (gat_dense.cu)
extern "C" int hicgat_gat_logits(int64_t n, int heads, int channels, const float* xl, const float* att_l, const float* att_r,
                                 float* a_src, float* a_dst, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(xl && att_l && att_r && a_src && a_dst && n > 0 && n < (1ll << 31), "hicgat_gat_logits: bad arguments");
    HICGAT_REQUIRE(gat_shape_supported(heads, channels), "hicgat_gat_logits: unsupported heads=%d channels=%d", heads, channels);
    HICGAT_REQUIRE(aligned16(xl) && aligned16(att_l) && aligned16(att_r), "hicgat_gat_logits: 16-byte alignment required");
    const unsigned grid = (unsigned)((n + kRowsPerCta - 1) / kRowsPerCta);
#define CALL_LOGIT(H, Q) gat_logit_kernel<H, Q><<<grid, 256, 0, stream>>>(xl, att_l, att_r, (int)n, a_src, a_dst)
    HICGAT_DISPATCH_HQ(heads, channels, CALL_LOGIT);
#undef CALL_LOGIT
    HICGAT_CHECK_LAUNCH("gat_logit_kernel");
    return HICGAT_OK;
}

extern "C" size_t hicgat_gat_param_grads_workspace_bytes(int64_t n, int heads, int channels) {
    if (n <= 0 || !gat_shape_supported(heads, channels)) return 0;
    return 256 + sizeof(float) * 3 * (size_t)heads * channels * (size_t)param_ctas(n);
}

// datt_l[c] = sum_j d_a_src[j,h(c)] xl[j,c] ; datt_r[c] = sum_j d_a_dst[j,h(c)] xl[j,c] ; dbias[c] = sum_i g[i,c]
extern "C" int hicgat_gat_param_grads(int64_t n, int heads, int channels, const float* xl, const float* gout, const float* d_a_src,
                                      const float* d_a_dst, float* datt_l, float* datt_r, float* dbias, void* workspace,
                                      size_t workspace_bytes, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(xl && gout && d_a_src && d_a_dst && datt_l && datt_r && dbias && workspace && n > 0 && n < (1ll << 31), "hicgat_gat_param_grads: bad arguments");
    HICGAT_REQUIRE(gat_shape_supported(heads, channels), "hicgat_gat_param_grads: unsupported heads=%d channels=%d", heads, channels);
    const size_t need = hicgat_gat_param_grads_workspace_bytes(n, heads, channels);
    if (workspace_bytes < need) {
        set_error("hicgat_gat_param_grads: workspace %zu < required %zu", workspace_bytes, need);
        return HICGAT_ERR_WORKSPACE;
    }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* part = reinterpret_cast<float*>(ws + 256);
    const int nblk = param_ctas(n);
    gat_bwd_param_kernel<<<nblk, 128, 0, stream>>>(xl, gout, d_a_src, d_a_dst, (int)n, heads, channels, part);
    HICGAT_CHECK_LAUNCH("gat_bwd_param_kernel");
    gat_bwd_param_reduce_kernel<<<(3 * heads * channels + 7) / 8, 256, 0, stream>>>(part, nblk, heads * channels, datt_l, datt_r, dbias);
    HICGAT_CHECK_LAUNCH("gat_bwd_param_reduce_kernel");
    return HICGAT_OK;
}
