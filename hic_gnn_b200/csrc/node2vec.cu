// node2vec embeddings (node2vec 0.4.3 + gensim 4 skip-gram with negative sampling) on the CSR graph of load_input:
//   * n2v_walk_kernel   : second-order biased random walks, one thread per walk, exact rejection sampling (KnightKing):
//                         O(nnz) memory instead of node2vec 0.4.3's O(sum deg^2) transition tables;
//   * sgns_epoch_kernel : one epoch of skip-gram with negative sampling (word2vec.c / gensim sg=1, hs=0), one warp per
//                         contiguous range of walks, rows spread over the lanes, updates as red.global.add.v4.f32.
// Every random draw is the stateless hash n2v_hash(seed, a, b, c) documented in hicgat.h, so the walks are bit-reproducible
// and a one-warp epoch can be replayed by tests/node2vec_ref.py.
#include "common.cuh"

namespace hicgat {
namespace {

constexpr int SG_WARPS = 8;  // warps per block of the skip-gram kernel

__device__ __forceinline__ uint64_t mix64(uint64_t z) {  // splitmix64 finaliser
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ uint64_t n2v_hash(uint64_t seed, uint64_t a, uint64_t b, uint64_t c) {
    uint64_t h = mix64(seed ^ 0x9E3779B97F4A7C15ull);
    h = mix64(h ^ a);
    h = mix64(h ^ b);
    return mix64(h ^ c);
}

// first k in [beg, end) with cdf[k] > u * cdf[end-1] (clamped to end-1): P(k) proportional to the edge weight
__device__ __forceinline__ int cdf_pick(const float* __restrict__ cdf, int beg, int end, float u) {
    const float x = u * __ldg(cdf + end - 1);
    int lo = beg, hi = end - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(cdf + mid) > x) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

__device__ __forceinline__ bool has_col(const int* __restrict__ col, int beg, int end, int x) {  // sorted row
    while (beg < end) {
        const int mid = (beg + end) >> 1;
        const int c = __ldg(col + mid);
        if (c == x) return true;
        if (c < x) beg = mid + 1;
        else end = mid;
    }
    return false;
}

__global__ void __launch_bounds__(128) n2v_walk_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ cdf,
                                                       const int* __restrict__ starts, int64_t nwalks, int64_t walk_id0, int L, float inv_p,
                                                       float inv_q, uint64_t seed, int* __restrict__ out) {
    const int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (w >= nwalks) return;
    const uint64_t gid = (uint64_t)(walk_id0 + w);
    int* o = out + w * L;
    const float amax = fmaxf(fmaxf(inv_p, 1.f), inv_q);
    int v = __ldg(starts + w), t = -1, s = 1;
    o[0] = v;
    for (; s < L; ++s) {
        const int beg = __ldg(rowptr + v), end = __ldg(rowptr + v + 1);
        if (beg == end) break;
        int x;
        if (t < 0) {
            x = __ldg(col + cdf_pick(cdf, beg, end, (float)(n2v_hash(seed, gid, s, 0) >> 40) * 0x1p-24f));
        } else {
            const int tb = __ldg(rowptr + t), te = __ldg(rowptr + t + 1);
            for (uint64_t a = 0;; ++a) {  // uncapped: a cap would bias the distribution
                const uint64_t h = n2v_hash(seed, gid, s, a);
                x = __ldg(col + cdf_pick(cdf, beg, end, (float)(h >> 40) * 0x1p-24f));
                const float alpha = x == t ? inv_p : (has_col(col, tb, te, x) ? 1.f : inv_q);
                if ((float)(h & 0xFFFFFFull) * 0x1p-24f * amax < alpha) break;
            }
        }
        o[s] = x;
        t = v;
        v = x;
    }
    for (; s < L; ++s) o[s] = -1;
}

// ------------------------------------------------------------------------------------------------ skip-gram
// Rows of syn0 / syn1neg are read at L2 (.cg): other warps add into them during the epoch, and a lane always touches the
// same columns of every row, so a lane's own red.add is visible to its next load of that row (same-thread coherence).
__device__ __forceinline__ float4 ld_row4(const float* p) {
    float4 v;
    asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_add4(float* p, float4 v) {
    asm volatile("red.relaxed.gpu.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ int bisect_left(const uint32_t* __restrict__ cum, int n, uint32_t x) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(cum + mid) < x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// word2vec.c: g = (label - sigma(f)) * alpha, clamped outside [-6, 6]; exact sigma instead of the 1000-entry table
__device__ __forceinline__ float sg_grad(float f, float label, float a) {
    if (f > 6.f) return (label - 1.f) * a;
    if (f < -6.f) return label * a;
    return (label - 1.f / (1.f + expf(-f))) * a;
}

// One (centre, context) pair: targets tg[0..nt) (tg[0] = centre, label 1; then the kept negatives, label 0), processed in
// word2vec.c order, G rows loaded together.  G > 1 only when no target repeats within the pair, so a group's rows are
// the values the serial order would read; with a repeat the caller passes G = 1 and each load follows the previous red.
template <int M, int G>
__device__ __forceinline__ void sg_pair(float* __restrict__ syn0, float* __restrict__ syn1neg, const int* tg, int nt, int o, float a, int lane) {
    constexpr int D = M * 128;
    float4 l1[M], e[M];
    float* r0 = syn0 + (size_t)o * D + lane * 4;
#pragma unroll
    for (int m = 0; m < M; ++m) {
        l1[m] = ld_row4(r0 + m * 128);
        e[m] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int k0 = 0; k0 < nt; k0 += G) {
        float4 row[G][M];
        float f[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
            f[g] = 0.f;
            if (k0 + g < nt) {
                const float* rp = syn1neg + (size_t)tg[k0 + g] * D + lane * 4;
#pragma unroll
                for (int m = 0; m < M; ++m) row[g][m] = ld_row4(rp + m * 128);
            } else {
#pragma unroll
                for (int m = 0; m < M; ++m) row[g][m] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
#pragma unroll
            for (int m = 0; m < M; ++m) {
                f[g] = fmaf(l1[m].x, row[g][m].x, f[g]);
                f[g] = fmaf(l1[m].y, row[g][m].y, f[g]);
                f[g] = fmaf(l1[m].z, row[g][m].z, f[g]);
                f[g] = fmaf(l1[m].w, row[g][m].w, f[g]);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
            for (int g = 0; g < G; ++g) f[g] += __shfl_xor_sync(0xffffffffu, f[g], off);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            if (k0 + g < nt) {
                const float gg = sg_grad(f[g], k0 + g == 0 ? 1.f : 0.f, a);
                float* rp = syn1neg + (size_t)tg[k0 + g] * D + lane * 4;
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    e[m].x = fmaf(gg, row[g][m].x, e[m].x);
                    e[m].y = fmaf(gg, row[g][m].y, e[m].y);
                    e[m].z = fmaf(gg, row[g][m].z, e[m].z);
                    e[m].w = fmaf(gg, row[g][m].w, e[m].w);
                    red_add4(rp + m * 128, make_float4(gg * l1[m].x, gg * l1[m].y, gg * l1[m].z, gg * l1[m].w));
                }
            }
        }
    }
#pragma unroll
    for (int m = 0; m < M; ++m) red_add4(r0 + m * 128, e[m]);
}

template <int M>
struct SgGroup {  // rows loaded together per pair: as many of the 1 + negative targets as registers allow
    static constexpr int G = M <= 2 ? 6 : (M <= 4 ? 3 : (M <= 5 ? 2 : 1));
};

template <int M>
__global__ void __launch_bounds__(SG_WARPS * 32, M <= 6 ? 2 : 1)  // 128 registers up to dim 768
    sgns_epoch_kernel(const int* __restrict__ walks, const int64_t* __restrict__ walk_off, int64_t nwalks, int L,
                      const uint32_t* __restrict__ cum, const uint32_t* __restrict__ keep_thr, int n, int window, int negative,
                      double alpha0, double min_alpha, int epoch, int epochs, uint64_t seed, int64_t num_warps, float* __restrict__ syn0,
                      float* __restrict__ syn1neg) {
    extern __shared__ int sg_smem[];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int* ktok = sg_smem + wib * (2 * L + 32);  // kept tokens of the current walk
    int* kidx = ktok + L;                      // their index in the walk
    int* tg = kidx + L;                        // targets of the current pair
    const int64_t gw = blockIdx.x * (int64_t)SG_WARPS + wib;
    if (gw >= num_warps) return;
    const int64_t w0 = gw * nwalks / num_warps, w1 = (gw + 1) * nwalks / num_warps;
    const double total = (double)epochs * (double)walk_off[nwalks];
    const uint32_t cum_last = __ldg(cum + n - 1);
    const unsigned below = (1u << lane) - 1u;
    for (int64_t w = w0; w < w1; ++w) {
        const int* walk = walks + w * L;
        const int64_t off = walk_off[w];
        int nk = 0;
        for (int base = 0; base < L; base += 32) {  // down-sampling, then compaction of the kept tokens (ballot + prefix)
            const int i = base + lane;
            const int tok = i < L ? __ldg(walk + i) : -1;
            const bool keep = tok >= 0 && (uint32_t)(n2v_hash(seed, (uint64_t)epoch, (uint64_t)(off + i), 0) >> 32) <= __ldg(keep_thr + tok);
            const unsigned b = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int k = nk + __popc(b & below);
                ktok[k] = tok;
                kidx[k] = i;
            }
            nk += __popc(b);
        }
        __syncwarp();
        for (int ci = 0; ci < nk; ++ci) {
            const int c = ktok[ci];
            const int64_t rp = off + kidx[ci];
            const int reach = window - (int)((uint32_t)(n2v_hash(seed, (uint64_t)epoch, (uint64_t)rp, 1ull << 32) >> 32) % (uint32_t)window);
            const float a = (float)fmax(min_alpha, alpha0 - (alpha0 - min_alpha) * ((double)epoch * (double)walk_off[nwalks] + (double)rp) / total);
            const int jlo = max(0, ci - reach), jhi = min(nk - 1, ci + reach);
            int jj = 0;
            for (int j = jlo; j <= jhi; ++j) {
                if (j == ci) continue;
                int t = -1;
                if (lane == 0) {
                    t = c;
                } else if (lane <= negative) {
                    const uint64_t h = n2v_hash(seed, (uint64_t)epoch, (uint64_t)rp, (2ull << 32) | (uint64_t)(jj * negative + lane - 1));
                    t = bisect_left(cum, n, (uint32_t)(h >> 32) % cum_last);
                    if (t == c) t = -1;  // word2vec.c: a negative equal to the centre is skipped
                }
                const unsigned act = __ballot_sync(0xffffffffu, t >= 0);
                if (t >= 0) tg[__popc(act & below)] = t;
                const unsigned same = __match_any_sync(0xffffffffu, t >= 0 ? t : -2 - lane);
                const bool repeat = __any_sync(0xffffffffu, __popc(same) > 1);
                __syncwarp();
                const int o = ktok[j];
                if (repeat) sg_pair<M, 1>(syn0, syn1neg, tg, __popc(act), o, a, lane);
                else sg_pair<M, SgGroup<M>::G>(syn0, syn1neg, tg, __popc(act), o, a, lane);
                __syncwarp();
                ++jj;
            }
        }
        __syncwarp();
    }
}

template <int M>
int launch_sgns(const int* walks, const int64_t* walk_off, int64_t nwalks, int L, const uint32_t* cum, const uint32_t* keep_thr, int n,
                int window, int negative, double alpha, double min_alpha, int epoch, int epochs, uint64_t seed, int64_t num_warps,
                float* syn0, float* syn1neg, cudaStream_t stream) {
    const size_t smem = (size_t)SG_WARPS * (2 * L + 32) * sizeof(int);
    if (num_warps <= 0) {  // fill the GPU (Hogwild)
        int dev = 0, sms = 0, per_sm = 0;
        HICGAT_CUDA(cudaGetDevice(&dev));
        HICGAT_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        HICGAT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgns_epoch_kernel<M>, SG_WARPS * 32, smem));
        num_warps = (int64_t)sms * (per_sm > 0 ? per_sm : 1) * SG_WARPS;
    }
    if (num_warps > nwalks) num_warps = nwalks;
    const unsigned blocks = (unsigned)((num_warps + SG_WARPS - 1) / SG_WARPS);
    sgns_epoch_kernel<M><<<blocks, SG_WARPS * 32, smem, stream>>>(walks, walk_off, nwalks, L, cum, keep_thr, n, window, negative, alpha,
                                                                   min_alpha, epoch, epochs, seed, num_warps, syn0, syn1neg);
    HICGAT_CHECK_LAUNCH("sgns_epoch_kernel");
    return HICGAT_OK;
}

}  // namespace
}  // namespace hicgat

using namespace hicgat;

extern "C" int hicgat_node2vec_walks(const int32_t* rowptr, const int32_t* col, const float* cdf, const int32_t* starts, int64_t num_starts,
                                     int64_t walk_id0, int walk_length, float p, float q, uint64_t seed, int32_t* walks,
                                     hicgat_stream_t stream_) {
    HICGAT_REQUIRE(rowptr && col && cdf && starts && walks, "hicgat_node2vec_walks: null pointer");
    HICGAT_REQUIRE(p > 0.f && q > 0.f && p <= 3.0e38f && q <= 3.0e38f, "hicgat_node2vec_walks: p and q must be finite and > 0 (got %g, %g)", p, q);
    HICGAT_REQUIRE(walk_length >= 1 && walk_length <= HICGAT_N2V_MAX_WALK_LENGTH, "hicgat_node2vec_walks: walk_length must be in [1, %d] (got %d)",
                   HICGAT_N2V_MAX_WALK_LENGTH, walk_length);
    HICGAT_REQUIRE(num_starts >= 0 && walk_id0 >= 0, "hicgat_node2vec_walks: bad num_starts / walk_id0");
    if (num_starts == 0) return HICGAT_OK;
    n2v_walk_kernel<<<(unsigned)((num_starts + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream_)>>>(
        rowptr, col, cdf, starts, num_starts, walk_id0, walk_length, 1.f / p, 1.f / q, seed, walks);
    HICGAT_CHECK_LAUNCH("n2v_walk_kernel");
    return HICGAT_OK;
}

extern "C" int hicgat_sgns_epoch(const int32_t* walks, const int64_t* walk_offsets, int64_t num_walks, int walk_length, const uint32_t* cum_table,
                                 const uint32_t* keep_threshold, int64_t n, int dim, int window, int negative, double alpha, double min_alpha,
                                 int epoch, int epochs, uint64_t seed, int64_t num_warps, float* syn0, float* syn1neg, hicgat_stream_t stream_) {
    HICGAT_REQUIRE(walks && walk_offsets && cum_table && keep_threshold && syn0 && syn1neg, "hicgat_sgns_epoch: null pointer");
    HICGAT_REQUIRE(dim % 128 == 0 && dim >= 128 && dim <= 1024, "hicgat_sgns_epoch: dim must be a multiple of 128 in [128, 1024] (got %d)", dim);
    HICGAT_REQUIRE(walk_length >= 1 && walk_length <= HICGAT_N2V_MAX_WALK_LENGTH, "hicgat_sgns_epoch: walk_length must be in [1, %d] (got %d)",
                   HICGAT_N2V_MAX_WALK_LENGTH, walk_length);
    HICGAT_REQUIRE(window >= 1, "hicgat_sgns_epoch: window must be >= 1 (got %d)", window);
    HICGAT_REQUIRE(negative >= 0 && negative <= 31, "hicgat_sgns_epoch: negative must be in [0, 31] (got %d)", negative);
    HICGAT_REQUIRE(n >= 1 && n < (1ll << 31) && num_walks >= 0, "hicgat_sgns_epoch: bad n / num_walks");
    HICGAT_REQUIRE(epochs >= 1 && epoch >= 0 && epoch < epochs, "hicgat_sgns_epoch: need 0 <= epoch < epochs (got %d, %d)", epoch, epochs);
    HICGAT_REQUIRE(alpha >= 0.0 && min_alpha >= 0.0 && alpha < 1e30 && min_alpha < 1e30, "hicgat_sgns_epoch: alpha and min_alpha must be finite and >= 0");
    HICGAT_REQUIRE(aligned16(syn0) && aligned16(syn1neg), "hicgat_sgns_epoch: syn0 / syn1neg must be 16-byte aligned");
    if (num_walks == 0) return HICGAT_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    switch (dim / 128) {
#define HICGAT_SG_CASE(M) \
    case M: return launch_sgns<M>(walks, walk_offsets, num_walks, walk_length, cum_table, keep_threshold, (int)n, window, negative, alpha, min_alpha, epoch, epochs, seed, num_warps, syn0, syn1neg, stream);
        HICGAT_SG_CASE(1) HICGAT_SG_CASE(2) HICGAT_SG_CASE(3) HICGAT_SG_CASE(4) HICGAT_SG_CASE(5) HICGAT_SG_CASE(6) HICGAT_SG_CASE(7) HICGAT_SG_CASE(8)
#undef HICGAT_SG_CASE
    }
    return HICGAT_ERR_INVALID;
}
