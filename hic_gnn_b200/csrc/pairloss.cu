// Fused pairwise-distance loss (forward + backward in one pass over the target block).
//
// Replaces torch.cdist + MSELoss / L1 / Pearson-moment glue of the reference loops
// (models.py:39, HiC-GNN_main.py:127, HiC_GAT_generalize_directly.py:210-225,
// train_and_test_same_res_GAT_node2vec.py:131-134) without materialising the N x N
// prediction.  HBM-bound: 4 B per ordered pair (one f32 target element), d = 3.
//
// Work decomposition (both kernel variants)
//   CTA  = 8 consumer warps x 128 columns x rb rows; grid = (column strips, row chunks).
//   lane = 4 consecutive columns j, kept as two packed f32x2 pairs so the arithmetic runs on
//          FADD2/FMUL2/FFMA2; x_j and the column-side gradient accumulators live in registers
//          for the whole CTA lifetime, x_i (warp-uniform) is broadcast from shared memory.
//   Because the target is symmetric the column-side sum  g_j = sum_i w_ij (x_j - x_i)  is the
//   complete gradient: no row-side reduction, no atomics.  Row chunks are combined by the last
//   CTA to finish each column strip (fixed summation order => bit-reproducible).
//
// Variant 0 (default, "tma"): every warp keeps a private 3-slot shared-memory ring; lane 0 issues
//   cp.async.bulk.tensor.2d (TMA) boxes of 8 rows x 128 columns (4 KB) that complete on the
//   warp's mbarriers and refills a slot as soon as the warp has consumed it, so no warp ever
//   waits on a global load it issued itself and 2 CTAs x 8 warps x 3 x 4 KB = 192 KB of target
//   are in flight per SM.  TMA zero-fills columns >= n and rows >= r1-r0 (no edge address logic).
// Variant 1 ("ldg"): each lane issues 8 streaming 128-bit ld.global.nc per row group; kept for
//   A/B measurements and as the path used when a tensor map cannot be encoded.  Same triangle modes.
#include <cuda.h>  // CUtensorMap (types only; the encoder is resolved through cudart at run time)

#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "common.cuh"

namespace hicgat {
namespace {

#ifndef HICGAT_PAIR_WARPS
#define HICGAT_PAIR_WARPS 8                // experiments: 4 warps x 4 CTAs per SM
#endif
constexpr int kWarps = HICGAT_PAIR_WARPS; // consumer warps
constexpr int kCtasPerSm = 16 / kWarps;   // 16 resident warps of 128 registers per SM
constexpr int kThreads = kWarps * 32;     // variant 1 block size
constexpr int kCols = 128;                // columns per CTA strip (32 lanes x 4)
constexpr int kU = 8;                     // rows per warp per group / tile
constexpr int kNM = HICGAT_PAIR_NMOM;
constexpr int kCtaSlots = 148 * kCtasPerSm;  // resident CTAs of the TMA kernel (2 per SM)
constexpr int kTileRows = kWarps * kU;    // 64 rows per CTA tile step (8 per warp)
constexpr int kStages = 3;                // TMA slots per warp
constexpr int kSubTileBytes = kU * kCols * 4;               // 4096: one warp's 8 rows x 128 columns
constexpr int kSlotBytes = kSubTileBytes + 256;             // + (x,x,y,y) x8 + (z,z) x8, padded to 128 B
constexpr int kTmaSmem = kWarps * kStages * kSlotBytes + 128;  // 104576 B: two CTAs per SM

// which upper-triangle statistics are accumulated
constexpr uint32_t kMomFull = HICGAT_PAIR_MOMENTS;          // everything (sum t, sum t^2, sum |d-t| too)
constexpr uint32_t kMomLight = HICGAT_PAIR_MOMENTS_D;       // sum d, sum d^2, sum d t, sum (d-t)^2 only

// Debug timeline (scratch builds with -DHICGAT_TRACE only; never in the shipped library): thread 0 of
// every CTA stamps %globaltimer at fixed points of pairloss_tma_kernel into g_trace[cta][8].
#ifdef HICGAT_TRACE
__device__ unsigned long long* g_trace = nullptr;
__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define HICGAT_TR(k)                                                                                         \
    do {                                                                                                     \
        if (threadIdx.x == 0 && g_trace) g_trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)] = gtimer(); \
    } while (0)
#define HICGAT_TRV(k, v)                                                                                     \
    do {                                                                                                     \
        if (threadIdx.x == 0 && g_trace) g_trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)] = (v); \
    } while (0)
#else
#define HICGAT_TR(k) do { } while (0)
#define HICGAT_TRV(k, v) do { } while (0)
#endif

struct Acc {
    f2 gx[2], gy[2], gz[2];          // column-side gradient, 2 column pairs
    f2 see;                          // sum (d-t)^2 over pairs NOT counted in seu
    f2 sd, sdd, st, stt, sdt, seu;   // upper-triangle moments
    float sabs0, sabs1;              // upper-triangle sum |d-t|
};

__device__ __forceinline__ void acc_zero(Acc& a) {
#pragma unroll
    for (int p = 0; p < 2; ++p) a.gx[p] = a.gy[p] = a.gz[p] = 0ull;
    a.see = a.sd = a.sdd = a.st = a.stt = a.sdt = a.seu = 0ull;
    a.sabs0 = a.sabs1 = 0.f;
}

// Second pass of the differentiable Pearson modes (hicgat_pairloss_pearson_grad): the per-pair weight needs the GLOBAL
// moments, so it is a library-internal mode bit that only those entry points set.
constexpr uint32_t kPearson = 64u;
// true when the instantiation produces a gradient (the MSE / L1 bits or the Pearson pass)
__host__ __device__ constexpr bool has_grad(uint32_t mode) { return (mode & (3u | kPearson)) != 0; }

// Coefficients of the Pearson pass, derived on the device from the global moments (see pearson_coef):
// w = (c_mse (d - t) + lamA rho) / d,  rho = t - (beta d + kappa)
struct PearsonCoef {
    f2 lam_a, beta, kappa, cm;
};

template <uint32_t MODE>
__device__ __forceinline__ f2 grad_weight(f2 e, f2 rs, float c_mse, float c_l1, f2 d, f2 t, const PearsonCoef& pc) {
    if constexpr ((MODE & kPearson) != 0) {
        // the residual of the regression of t on d, formed in f32 as t - fma(beta, d, kappa), and the MSE residual are kept
        // apart: folding them into one affine a t + b d + c loses the cancellation of t against beta d + kappa near r = 1
        f2 w = f2_mul(pc.lam_a, f2_sub(t, f2_fma(pc.beta, d, pc.kappa)));
        if constexpr ((MODE & HICGAT_PAIR_GRAD_MSE) != 0) w = f2_fma(pc.cm, e, w);
        return f2_mul(w, rs);
    } else if constexpr ((MODE & 3u) == HICGAT_PAIR_GRAD_MSE) {
        return f2_mul(e, rs);
    } else if constexpr ((MODE & 3u) == HICGAT_PAIR_GRAD_L1) {
        float ea, eb, ra, rb;
        f2_unpack(e, ea, eb);
        f2_unpack(rs, ra, rb);
        return f2_pack(copysignf(ra, ea), copysignf(rb, eb));
    } else if constexpr ((MODE & 3u) == 3u) {
        float ea, eb;
        f2_unpack(e, ea, eb);
        f2 s = f2_pack(copysignf(c_l1, ea), copysignf(c_l1, eb));
        return f2_mul(f2_fma(e, f2_pack(c_mse, c_mse), s), rs);
    } else {
        return 0ull;
    }
}

// d^2 + 1e-30: keeps rsqrt finite on the diagonal / for coincident loci (d = 1e-15, weight * 0 = 0,
// matching ATen's "ratio = 0 where dist == 0") at the cost of nothing: it rides in the first FMA.
#define HICGAT_TINY2 0x0DA242600DA24260ull /* (1e-30f, 1e-30f) */

// Row-side accumulators of ONE row (symmetric / upper-triangle mode): sum over the lane's columns of w * (x_j - x_i).
struct RowAcc {
    f2 x, y, z;
};

// One row x one column pair, no masks.  UPPER: this (row, pair) lies strictly above the diagonal.
// ROWS: upper-triangle mode -- every unordered pair is evaluated once, so the weight also feeds the row-side
// accumulators and the strictly-upper sum of squares is kept apart (it counts twice in the full-matrix loss).
template <uint32_t MODE, bool UPPER, bool ROWS>
__device__ __forceinline__ void pair_fast(Acc& a, RowAcc& ra, int p, f2 xjx, f2 xjy, f2 xjz, f2 xix, f2 xiy,
                                          f2 xiz, f2 t, float c_mse, float c_l1, const PearsonCoef& pc) {
    f2 dx = f2_sub(xjx, xix), dy = f2_sub(xjy, xiy), dz = f2_sub(xjz, xiz);
    f2 d2 = f2_fma(dx, dx, f2_fma(dy, dy, f2_fma(dz, dz, HICGAT_TINY2)));
    float d2a, d2b;
    f2_unpack(d2, d2a, d2b);
    f2 rs = f2_pack(rsqrt_approx(d2a), rsqrt_approx(d2b));
    f2 d = f2_mul(d2, rs);
    f2 e = f2_sub(d, t);
    constexpr bool kMom = UPPER && (MODE & (kMomFull | kMomLight));
    if constexpr ((MODE & kPearson) != 0) {
        // the Pearson pass produces the gradient only (its moments are an input)
    } else if constexpr (kMom || (UPPER && ROWS)) a.seu = f2_fma(e, e, a.seu);
    else a.see = f2_fma(e, e, a.see);
    if constexpr (has_grad(MODE)) {
        f2 w = grad_weight<MODE>(e, rs, c_mse, c_l1, d, t, pc);
        a.gx[p] = f2_fma(w, dx, a.gx[p]);
        a.gy[p] = f2_fma(w, dy, a.gy[p]);
        a.gz[p] = f2_fma(w, dz, a.gz[p]);
        if constexpr (ROWS) {
            ra.x = f2_fma(w, dx, ra.x);
            ra.y = f2_fma(w, dy, ra.y);
            ra.z = f2_fma(w, dz, ra.z);
        }
    }
    if constexpr (kMom) {
        a.sd = f2_add(a.sd, d);
        a.sdd = f2_add(a.sdd, d2);
        a.sdt = f2_fma(d, t, a.sdt);
        if constexpr ((MODE & kMomFull) != 0) {
            float ea, eb;
            f2_unpack(e, ea, eb);
            a.sabs0 += fabsf(ea);
            a.sabs1 += fabsf(eb);
            a.st = f2_add(a.st, t);
            a.stt = f2_fma(t, t, a.stt);
        }
    }
}

// Masked variant for edge strips (columns >= n), partial tiles and diagonal-crossing groups.
// mv: 1 for valid (row, column) -- in upper-triangle mode additionally row <= column; mu: 1 where row < col.
template <uint32_t MODE, bool ROWS>
__device__ __forceinline__ void pair_masked(Acc& a, RowAcc& ra, int p, f2 xjx, f2 xjy, f2 xjz, f2 xix, f2 xiy,
                                            f2 xiz, f2 t, f2 mv, f2 mu, float c_mse, float c_l1, const PearsonCoef& pc) {
    f2 dx = f2_sub(xjx, xix), dy = f2_sub(xjy, xiy), dz = f2_sub(xjz, xiz);
    f2 d2 = f2_fma(dx, dx, f2_fma(dy, dy, f2_fma(dz, dz, HICGAT_TINY2)));
    float d2a, d2b;
    f2_unpack(d2, d2a, d2b);
    f2 rs = f2_pack(rsqrt_approx(d2a), rsqrt_approx(d2b));
    f2 d = f2_mul(d2, rs);
    f2 e = f2_mul(f2_sub(d, t), mv);
    constexpr bool kMom = (MODE & (kMomFull | kMomLight)) != 0;
    if constexpr (has_grad(MODE)) {
        f2 w = f2_mul(grad_weight<MODE>(e, rs, c_mse, c_l1, d, t, pc), mv);
        a.gx[p] = f2_fma(w, dx, a.gx[p]);
        a.gy[p] = f2_fma(w, dy, a.gy[p]);
        a.gz[p] = f2_fma(w, dz, a.gz[p]);
        if constexpr (ROWS) {
            ra.x = f2_fma(w, dx, ra.x);
            ra.y = f2_fma(w, dy, ra.y);
            ra.z = f2_fma(w, dz, ra.z);
        }
    }
    if constexpr ((MODE & kPearson) != 0) {
        // gradient only, as in pair_fast
    } else if constexpr (kMom || ROWS) {
        f2 eu = f2_mul(e, mu);
        f2 el = f2_sub(e, eu);  // the part of e not under the upper mask
        a.see = f2_fma(el, el, a.see);
        a.seu = f2_fma(eu, eu, a.seu);
        if constexpr (kMom) {
            f2 du = f2_mul(d, mu), tu = f2_mul(t, mu);
            a.sd = f2_add(a.sd, du);
            a.sdd = f2_fma(du, du, a.sdd);
            a.sdt = f2_fma(du, tu, a.sdt);
            if constexpr ((MODE & kMomFull) != 0) {
                float ea, eb;
                f2_unpack(eu, ea, eb);
                a.sabs0 += fabsf(ea);
                a.sabs1 += fabsf(eb);
                a.st = f2_add(a.st, tu);
                a.stt = f2_fma(tu, tu, a.stt);
            }
        }
    } else {
        a.see = f2_fma(e, e, a.see);
    }
}

// Row-chunk boundaries (offsets from r0) of the unstaggered [0] and the staggered [1] column strips.
constexpr int kMaxChunks = 128;
struct Schedule {
    int count[2];
    int bounds[2][kMaxChunks + 1];
};

struct Params {
    const float* coords;
    const float* target;  // points at row r0
    int64_t pitch;
    int n, r0, r1, rb, nstrips, nchunks;  // nchunks = grid.y = chunk slots per strip (staggered strips use one more than the others)
    int stagger;                          // 1: strips with odd (strip / 148) use the second boundary table (see chunk_rows)
    Schedule sch;
    float fill;                           // implicit-target kernel: wish distance of every non-edge pair
    float c_mse, c_l1;
    double* moments;
    float* grad;
    double* grad64;        // optional f64 copy of grad (packed all-reduce buffer)
    float* gpart;          // [nchunks][nstrips][384]  per-CTA gradient partials
    double* mpart;         // [nchunks*nstrips][kNM]   per-CTA moment partials
    // upper-triangle ("symmetric") mode: only pairs with row <= column are evaluated; every CTA also emits the ROW-side
    // gradient sums of its rows over its 128 columns: rpart[strip][(row - r0) * 3 + comp], rpitch floats per strip
    int upper;
    int64_t rpitch;
    float* rpart;
    // persistent variant: items = active (chunk, strip) pairs in chunk-major order; item_base[c] = first item of chunk c
    unsigned* work_counter;   // zero before the launch, reset by the combine kernel
    int nitems;
    int item_base[kMaxChunks + 1];
    // static warp partition (variant 4): the strip-major sequence of (strip, row) work is cut into equal runs of seg_len rows,
    // one per warp; the partial of (strip s, warp w) lives in slot (w - first_warp(s)) * nstrips + s
    int64_t seg_len, seg_total;
    int seg_sa, seg_sb, seg_f;   // closed form of the rows per strip, see strip_offset()
    // combine kernel, upper-triangle mode on a short row block: the row-side sums of the rs_count strips that hold this block's loci
    // are cut into rs_groups segments of source strips, one CTA each (see pairloss_combine_kernel); rs_groups <= 1 = one CTA per strip
    int rs_first, rs_count, rs_groups;
    double* rs_scratch;       // [rs_count][rs_groups][384] segment sums
    unsigned* rs_ticket;      // [rs_count] arrival counters, zero between calls
    // Pearson pass: the global f64 moments of the first pass (read on the device only) and whether the Pearson term is
    // weighted by alpha = min(1, 0.1 + 1 / (MSE + 1e-6)) (mse_pearson_grad) or by 1 (pearson)
    const double* pmom;
    int dyn_alpha;
};

// r, beta, kappa, A and alpha from the global moments (f64), rounded once to f32.  Called after griddepcontrol.wait (the
// moments are written by the previous kernels of the stream).  Degenerate moments (v_d v_t <= 0 or not finite: n <= 2,
// coincident loci, a constant target) give a zero Pearson weight: r is NaN there and carries no gradient.
template <uint32_t MODE>
__device__ __forceinline__ PearsonCoef pearson_coef(const double* pm, int n, float c_mse, int dyn_alpha) {
    PearsonCoef pc;
    pc.lam_a = pc.beta = pc.kappa = pc.cm = 0ull;
    if constexpr ((MODE & kPearson) != 0) {
        const double np = 0.5 * (double)n * (double)(n - 1);
        const double sd = pm[2], sdd = pm[3], st = pm[4], stt = pm[5], sdt = pm[6];
        const double vd = sdd - sd * sd / np, vt = stt - st * st / np, c = sdt - sd * st / np;
        const double prod = vd * vt;
        if (prod > 0.0 && prod < INFINITY) {
            const double beta = c / vd;
            const double kappa = st / np - beta * (sd / np);
            double lam = 1.0;
            if (dyn_alpha) {  // the loss value's f32 MSE, as MSELoss returns it
                const double mse = (double)(float)(pm[0] / ((double)n * (double)n));
                lam = fmin(1.0, 0.1 + 1.0 / (mse + 1e-6));
            }
            const float la = (float)(-lam / sqrt(prod)), b = (float)beta, k = (float)kappa;
            pc.lam_a = f2_pack(la, la);
            pc.beta = f2_pack(b, b);
            pc.kappa = f2_pack(k, k);
        }
        pc.cm = f2_pack(c_mse, c_mse);
    }
    return pc;
}

struct ColumnRegs {
    f2 xjx[2], xjy[2], xjz[2], mv[2];
};

__device__ __forceinline__ void load_columns(ColumnRegs& c, const float* __restrict__ coords, int col0, int n) {
    float cj[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int cc = min(col0 + k, n - 1);
#pragma unroll
        for (int q = 0; q < 3; ++q) cj[k][q] = coords[(size_t)cc * 3 + q];
    }
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        c.xjx[p] = f2_pack(cj[2 * p][0], cj[2 * p + 1][0]);
        c.xjy[p] = f2_pack(cj[2 * p][1], cj[2 * p + 1][1]);
        c.xjz[p] = f2_pack(cj[2 * p][2], cj[2 * p + 1][2]);
        c.mv[p] = f2_pack(col0 + 2 * p < n ? 1.f : 0.f, col0 + 2 * p + 1 < n ? 1.f : 0.f);
    }
}

// kU rows of one warp: t[u] = the lane's 4 target values of row (rg + u); xi from shared memory.
struct XiPtr {  // x_i rows behind ordinary shared-memory pointers (variant 1)
    const float4* xy;
    const float2* z;
    __device__ __forceinline__ void load(int u, float4& oxy, float2& oz) const { oxy = xy[u]; oz = z[u]; }
};
struct XiAddr {  // x_i rows behind 32-bit shared-space addresses (TMA variant)
    uint32_t xy, z;
    __device__ __forceinline__ void load(int u, float4& oxy, float2& oz) const;
};

// Transpose-reduce of the 24 row-side sums of one 8-row group (v[3 * u + comp]) across the warp: 24 shuffles instead of
// 24 x 5.  On return lane L holds the warp total of slot  12*b4 + 6*b3 + 3*b2 + (b0 ? 2 : b1)  (b_k = bit k of L);
// lanes with b0 = 1 hold their slot twice (b1 = 0 and b1 = 1).  Fixed order: bit-reproducible.
__device__ __forceinline__ float row_butterfly(const float (&v)[3 * kU], int lane) {
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2, b0 = lane & 1;
    float w12[12], w6[6], w3[3];
#pragma unroll
    for (int k = 0; k < 12; ++k) w12[k] = (b4 ? v[k + 12] : v[k]) + __shfl_xor_sync(0xffffffffu, b4 ? v[k] : v[k + 12], 16);
#pragma unroll
    for (int k = 0; k < 6; ++k) w6[k] = (b3 ? w12[k + 6] : w12[k]) + __shfl_xor_sync(0xffffffffu, b3 ? w12[k] : w12[k + 6], 8);
#pragma unroll
    for (int k = 0; k < 3; ++k) w3[k] = (b2 ? w6[k + 3] : w6[k]) + __shfl_xor_sync(0xffffffffu, b2 ? w6[k] : w6[k + 3], 4);
    const float a = (b1 ? w3[1] : w3[0]) + __shfl_xor_sync(0xffffffffu, b1 ? w3[0] : w3[1], 2);
    const float b = w3[2] + __shfl_xor_sync(0xffffffffu, w3[2], 2);
    return (b0 ? b : a) + __shfl_xor_sync(0xffffffffu, b0 ? a : b, 1);
}
__device__ __forceinline__ int row_butterfly_slot(int lane) {
    return ((lane & 16) ? 12 : 0) + ((lane & 8) ? 6 : 0) + ((lane & 4) ? 3 : 0) + ((lane & 1) ? 2 : ((lane & 2) ? 1 : 0));
}

// ROWS (upper-triangle mode): `rowdst` points at the 3 * kU row-side partials of this group's rows for this strip;
// the group is never strictly below the diagonal (the CTA's row range is clipped at the strip's last column).
template <uint32_t MODE, bool ROWS, typename XI>
__device__ __forceinline__ void process_group(Acc& a, const ColumnRegs& c, const float4 (&t)[kU], const XI xi,
                                              int rows_here, int rg, int col0, int n, bool edge,
                                              int strip_lo, int strip_hi, float c_mse, float c_l1, float* __restrict__ rowdst, int lane,
                                              const PearsonCoef& pc) {
    const bool fast = !edge && rows_here == kU;
    constexpr bool kRowGrad = ROWS && has_grad(MODE);
    float rv[kRowGrad ? 3 * kU : 1];
    if (fast && rg + kU - 1 < strip_lo) {  // strictly above the diagonal
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            float4 xy;
            float2 zz;
            xi.load(u, xy, zz);
            f2 xix = f2_pack(xy.x, xy.y), xiy = f2_pack(xy.z, xy.w), xiz = f2_pack(zz.x, zz.y);
            RowAcc ra = {0ull, 0ull, 0ull};
            pair_fast<MODE, true, ROWS>(a, ra, 0, c.xjx[0], c.xjy[0], c.xjz[0], xix, xiy, xiz, f2_pack(t[u].x, t[u].y), c_mse, c_l1, pc);
            pair_fast<MODE, true, ROWS>(a, ra, 1, c.xjx[1], c.xjy[1], c.xjz[1], xix, xiy, xiz, f2_pack(t[u].z, t[u].w), c_mse, c_l1, pc);
            if constexpr (kRowGrad) {
                rv[3 * u] = f2_hsum(ra.x); rv[3 * u + 1] = f2_hsum(ra.y); rv[3 * u + 2] = f2_hsum(ra.z);
            }
        }
    } else if (!ROWS && fast && rg > strip_hi) {    // strictly below
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            float4 xy;
            float2 zz;
            xi.load(u, xy, zz);
            f2 xix = f2_pack(xy.x, xy.y), xiy = f2_pack(xy.z, xy.w), xiz = f2_pack(zz.x, zz.y);
            RowAcc ra = {0ull, 0ull, 0ull};
            pair_fast<MODE, false, false>(a, ra, 0, c.xjx[0], c.xjy[0], c.xjz[0], xix, xiy, xiz, f2_pack(t[u].x, t[u].y), c_mse, c_l1, pc);
            pair_fast<MODE, false, false>(a, ra, 1, c.xjx[1], c.xjy[1], c.xjz[1], xix, xiy, xiz, f2_pack(t[u].z, t[u].w), c_mse, c_l1, pc);
        }
    } else {
#pragma unroll
        for (int u = 0; u < kU; ++u) {
            RowAcc ra = {0ull, 0ull, 0ull};
            if (u < rows_here) {
                const int r = rg + u;
                float4 xy;
                float2 zz;
                xi.load(u, xy, zz);
                f2 xix = f2_pack(xy.x, xy.y), xiy = f2_pack(xy.z, xy.w), xiz = f2_pack(zz.x, zz.y);
                f2 mu0 = f2_pack((col0 + 0 < n && r < col0 + 0) ? 1.f : 0.f, (col0 + 1 < n && r < col0 + 1) ? 1.f : 0.f);
                f2 mu1 = f2_pack((col0 + 2 < n && r < col0 + 2) ? 1.f : 0.f, (col0 + 3 < n && r < col0 + 3) ? 1.f : 0.f);
                f2 mv0 = c.mv[0], mv1 = c.mv[1];
                if constexpr (ROWS) {  // upper-triangle mode: pairs below the diagonal belong to another tile (as its upper pairs)
                    mv0 = f2_pack((col0 + 0 < n && r <= col0 + 0) ? 1.f : 0.f, (col0 + 1 < n && r <= col0 + 1) ? 1.f : 0.f);
                    mv1 = f2_pack((col0 + 2 < n && r <= col0 + 2) ? 1.f : 0.f, (col0 + 3 < n && r <= col0 + 3) ? 1.f : 0.f);
                }
                pair_masked<MODE, ROWS>(a, ra, 0, c.xjx[0], c.xjy[0], c.xjz[0], xix, xiy, xiz, f2_pack(t[u].x, t[u].y), mv0, mu0, c_mse, c_l1, pc);
                pair_masked<MODE, ROWS>(a, ra, 1, c.xjx[1], c.xjy[1], c.xjz[1], xix, xiy, xiz, f2_pack(t[u].z, t[u].w), mv1, mu1, c_mse, c_l1, pc);
            }
            if constexpr (kRowGrad) {
                rv[3 * u] = f2_hsum(ra.x); rv[3 * u + 1] = f2_hsum(ra.y); rv[3 * u + 2] = f2_hsum(ra.z);
            }
        }
    }
    if constexpr (kRowGrad) {
        // row-side term of locus i: sum_j w_ij (x_i - x_j) = - sum_j w_ij dx_ij ; one coalesced 96-byte store per group
        const float tot = row_butterfly(rv, lane);
        const int slot = row_butterfly_slot(lane);
        if (((lane & 1) == 0 || (lane & 2) == 0) && slot < 3 * rows_here) __stcg(rowdst + slot, -tot);
    }
}

// Row range of (strip, chunk).  The two CTAs that share an SM start together and, with equal
// chunks, would also finish together: both slots then sit in their epilogue / prologue at the same
// time and the SM's share of HBM idles once per wave.  The first wave puts CTAs 148..295 (strips
// 148..295 of chunk 0) into the second slot of every SM, so those strips use a second boundary table
// whose first item is half as long: the two slots stay half a period apart for the rest of the
// kernel.  Chunk lengths need not be equal: the host may shrink the last chunks of every strip so that
// the items dispatched last are short (build_schedule).  Returns the number of chunks of this strip.
__device__ __forceinline__ int strip_parity(const Params& P, int strip) { return (P.stagger && ((strip / 148) & 1)) ? 1 : 0; }
__device__ __forceinline__ int chunk_rows(const Params& P, int strip, int chunk, int& row_begin, int& nrows) {
    const int par = strip_parity(P, strip);
    const int count = P.sch.count[par];
    int start = 0, end = 0;
    if (chunk < count) {
        start = P.sch.bounds[par][chunk];
        end = P.sch.bounds[par][chunk + 1];
    }
    if (P.upper) {  // only rows <= the strip's last column: the rest of the column strip lies below the diagonal
        const int lim = (strip + 1) * kCols - P.r0;
        end = end < lim ? end : lim;
    }
    row_begin = P.r0 + start;
    nrows = end > start ? end - start : 0;
    return count;
}
// number of leading chunks of `strip` that hold rows at all (all of them unless upper-triangle mode clips the strip)
__device__ __forceinline__ int strip_segments(const Params& P, int s);
__device__ __forceinline__ int active_chunks(const Params& P, int strip) {
    if (P.seg_len > 0) return strip_segments(P, strip);  // static warp partition: one partial per warp that touched the strip
    const int par = strip_parity(P, strip);
    int count = P.sch.count[par];
    if (P.upper) {
        const int lim = (strip + 1) * kCols - P.r0;
        while (count > 0 && P.sch.bounds[par][count - 1] >= lim) --count;
    }
    return count;
}

struct CombineSmem {
    float g[kWarps][kCols * 3 + 4];
    double m[kWarps][kNM];
};

// warp-level part of the CTA combine: park this warp's gradients / moments in shared memory
template <uint32_t MODE, bool ROWS = false>
__device__ __forceinline__ void park_warp(const Acc& a, CombineSmem& S, int warp, int lane) {
    if constexpr (has_grad(MODE)) {
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            float x0, x1, y0, y1, z0, z1;
            f2_unpack(a.gx[p], x0, x1);
            f2_unpack(a.gy[p], y0, y1);
            f2_unpack(a.gz[p], z0, z1);
            float* dst = &S.g[warp][(lane * 4 + 2 * p) * 3];
            dst[0] = x0; dst[1] = y0; dst[2] = z0;
            dst[3] = x1; dst[4] = y1; dst[5] = z1;
        }
    }
    constexpr bool kMom = (MODE & (kMomFull | kMomLight)) != 0;
    double m[kNM];
#pragma unroll
    for (int k = 0; k < kNM; ++k) m[k] = 0.0;
    const double seu = (double)f2_hsum(a.seu);
    m[0] = (double)f2_hsum(a.see) + (ROWS ? 2.0 * seu : seu);  // upper-triangle mode: every strictly-upper pair stands for (i,j) and (j,i)
    if constexpr (kMom) {
        m[2] = (double)f2_hsum(a.sd);
        m[3] = (double)f2_hsum(a.sdd);
        m[6] = (double)f2_hsum(a.sdt);
        m[7] = seu;
        if constexpr ((MODE & kMomFull) != 0) {
            m[1] = (double)a.sabs0 + (double)a.sabs1;
            m[4] = (double)f2_hsum(a.st);
            m[5] = (double)f2_hsum(a.stt);
        }
    }
#pragma unroll
    for (int k = 0; k < kNM; ++k) {
        if (k == 0 || kMom) m[k] = warp_sum(m[k]);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kNM; ++k) S.m[warp][k] = m[k];
    }
}

// Programmatic dependent launch: the producer kernels allow pairloss_combine_kernel to be scheduled as soon
// as their last CTA has STARTED; its blocks then sit resident (launch latency, instruction fetch and
// parameter loads done) in griddepcontrol.wait until the producer grid has completed and flushed.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// CTA-level combine.  Called by ALL threads of the block after a __syncthreads() that follows
// park_warp(); nthreads = blockDim.x.  The CTA only STORES its partial (f32 gradient of its 128
// columns, f64 moments) at slot chunk * nstrips + strip and exits: no fence, no ticket, no atomics.
// A streaming CTA slot that sits in a publish round trip (fence + atomic under a saturated memory
// system: ~3 us, measured per CTA with %globaltimer) streams nothing, and row blocks of a few thousand
// rows have only 2-5 items per slot; the cross-CTA sums are done by pairloss_combine_kernel, launched
// right behind on the same stream (the kernel boundary is the release / acquire).
template <uint32_t MODE>
__device__ __forceinline__ void publish_cta(const Params& P, CombineSmem& S, int strip, int chunk, int tid, int nthreads) {
    const int cta = chunk * P.nstrips + strip;
    if constexpr (has_grad(MODE)) {
        float* gp = P.gpart + (size_t)cta * (kCols * 3);
        for (int i = tid; i < kCols * 3; i += nthreads) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += S.g[w][i];
            __stcg(gp + i, s);
        }
    }
    if (tid < kNM) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += S.m[w][tid];
        __stcg(P.mpart + (size_t)cta * kNM + tid, s);
    }
}

// Cross-CTA sums in a FIXED order (bit-reproducible).  Blocks 0 .. nstrips-1: the strip's gradient =
// its row-chunk partials added in chunk order in f64, scaled, rounded once to f32.  Block nstrips: the
// moments = every CTA's f64 partial, thread t taking slots t, t+512, ... (slots of chunks a strip does
// not have are skipped), then lanes, then warps.
constexpr int kCombineThreads = 512;
// `npass` = 2 under programmatic dependent launch: the blocks become resident while the producer's last
// wave is still streaming, and the producer has pushed everything else -- including this kernel's
// instructions -- out of L2 (400 MB+ go through 126 MB).  Pass 0 therefore runs the SAME code on whatever
// the buffers hold, stores nothing, and leaves the instruction cache, the TLB entries and the parameter
// loads warm; pass 1 follows the wait (moment block of a 1 560-partial grid: 8.6 -> 5.4 us after the wait,
// %globaltimer stamps; the gradient blocks did not change).
// Sum of `count` partials src[k * stride] in index order, in f64, B loads per round.  Every load is issued UNCONDITIONALLY (the
// index is clamped, the out-of-range term is replaced by +0.0 afterwards, which leaves the sum unchanged) so that the compiler keeps
// all B in flight before the first add: with a bounds predicate per load it interleaves loads and adds, and the chain of dependent-
// latency rounds -- which is all this kernel consists of on a short row block -- gets several times longer.
template <int B>
__device__ __forceinline__ double ordered_sum(const float* src, size_t stride, int count) {
    double sum = 0.0;
#pragma unroll 1
    for (int c = 0; c < count; c += B) {
        float v[B];
#pragma unroll
        for (int k = 0; k < B; ++k) v[k] = __ldcg(src + (size_t)min(c + k, count - 1) * stride);
#pragma unroll
        for (int k = 0; k < B; ++k) sum += c + k < count ? (double)v[k] : 0.0;
    }
    return sum;
}
// column-side sum of one element of a strip: its per-CTA partials in chunk order
__device__ __forceinline__ double colside_sum(const Params& P, int strip, int tid) {
    return ordered_sum<8>(P.gpart + (size_t)strip * (kCols * 3) + tid, (size_t)P.nstrips * (kCols * 3), active_chunks(P, strip));
}
// row-side sum of one element over the source strips [s_begin, s_end), in strip order
__device__ __forceinline__ double rowside_sum(const Params& P, const float* rsrc, int s_begin, int s_end) {
    return ordered_sum<16>(rsrc + (size_t)s_begin * P.rpitch, (size_t)P.rpitch, s_end - s_begin);
}

// Grid: [1 moment CTA] [rs_count * rs_groups row-side CTAs (only when rs_groups > 1)] [nstrips gradient CTAs].
// Row-side CTAs: a thread sums ONE element over up to nstrips source strips, a chain of dependent-latency rounds (16 loads each).  On
// a short row block (a shard of a sharded run) only a handful of strips hold loci of the block, so that chain -- not bandwidth -- is
// the whole kernel: each such strip is therefore cut into rs_groups segments of source strips, one CTA each; the CTA that arrives
// last at the strip's ticket adds the segment sums in segment order (and the column-side sum) and writes the gradient.  Every sum
// has a fixed order, so the result does not depend on which CTA arrives last: bit-reproducible.
__global__ void __launch_bounds__(kCombineThreads, 2) pairloss_combine_kernel(const Params P, const float scale, const int want_grad, const int npass) {
    pdl_launch_dependents();  // a consumer launched with programmatic serialization (the sharded exchange kernel) may become resident now
    const int tid = threadIdx.x;
    __shared__ double s_m[kCombineThreads / 32][kNM];
    __shared__ int s_last;
    const int G = P.rs_groups > 1 ? P.rs_groups : 0;
    // Block 0 sums the moments: its chain of dependent rounds is as long as a row-side CTA's, so it must not wait for a free slot
    // behind the (more than one wave of) gradient CTAs.  Then the row-side CTAs (longest), then one gradient CTA per strip.
    const int rs_idx = (int)blockIdx.x - 1;                                      // row-side CTA index when 0 <= rs_idx < G * rs_count
    const int bid = blockIdx.x == 0 ? P.nstrips : rs_idx - G * P.rs_count;       // < 0: row-side CTA; [0, nstrips): strip; nstrips: moments
#ifdef HICGAT_TRACE
    unsigned long long* ctr = (g_trace && tid == 0 && (bid == 0 || bid == P.nstrips)) ? g_trace + (size_t)(8190 + (bid == 0 ? 0 : 1)) * 8 : nullptr;
    if (ctr) ctr[0] = gtimer();
#endif
#pragma unroll 1
    for (int pass = 0; pass < npass; ++pass) {
        const bool live = pass == npass - 1;
        if (live) {
            pdl_wait();  // no-op when launched without the programmatic-serialization attribute
            // the persistent kernel's item counter, for the next launch: reset by block 0 (the moment CTA), the one CTA that reaches this
            // live pass in every mode (strip and row-side CTAs may return in the first pass under programmatic dependent launch)
            if (P.work_counter && blockIdx.x == 0 && tid == 0) *P.work_counter = 0u;
#ifdef HICGAT_TRACE
            if (ctr) ctr[1] = gtimer();
#endif
        }
        if (bid < 0) {
            if (!want_grad) return;
            const int bi = rs_idx / G, g = rs_idx - bi * G;
            const int strip = P.rs_first + bi;
            const int locus = strip * kCols + tid / 3;
            if (tid < kCols * 3) {
                double part = 0.0;
                if (locus >= P.r0 && locus < P.r1) {
                    const int len = (P.nstrips - strip + G - 1) / G;
                    const int sb = strip + g * len, se = min(sb + len, P.nstrips);
                    part = rowside_sum(P, P.rpart + (size_t)(locus - P.r0) * 3 + (tid - (tid / 3) * 3), sb, se);
                }
                if (live) P.rs_scratch[((size_t)bi * G + g) * (kCols * 3) + tid] = part;
            }
            if (live) {
                __threadfence();
                __syncthreads();
                if (tid == 0) s_last = atomicAdd(P.rs_ticket + bi, 1u) == (unsigned)(G - 1) ? 1 : 0;
                __syncthreads();
                if (s_last) {
                    __threadfence();
                    if (tid < kCols * 3) {
                        double sum = colside_sum(P, strip, tid);
                        for (int g2 = 0; g2 < G; ++g2) sum += __ldcg(P.rs_scratch + ((size_t)bi * G + g2) * (kCols * 3) + tid);
                        if (locus < P.n) {
                            const double val = sum * (double)scale;
                            if (P.grad) P.grad[(size_t)strip * kCols * 3 + tid] = (float)val;
                            if (P.grad64) P.grad64[(size_t)strip * kCols * 3 + tid] = (double)(float)val;
                        }
                    }
                    if (tid == 0) P.rs_ticket[bi] = 0u;  // for the next call
                }
            }
        } else if (bid < P.nstrips) {
            if (!want_grad) return;
            const int strip = bid;
            if (G && strip >= P.rs_first && strip < P.rs_first + P.rs_count) return;  // written by the strip's row-side CTAs
            // one element of the strip's 384 per thread
            if (tid < kCols * 3) {
                double sum = colside_sum(P, strip, tid);
                const int locus = strip * kCols + tid / 3;
                if (P.upper && locus >= P.r0 && locus < P.r1)  // row-side sums of this locus: one partial per strip at or right of its own
                    sum += rowside_sum(P, P.rpart + (size_t)(locus - P.r0) * 3 + (tid - (tid / 3) * 3), strip, P.nstrips);
                if (live && locus < P.n) {
                    const double val = sum * (double)scale;
                    if (P.grad) P.grad[(size_t)strip * kCols * 3 + tid] = (float)val;
                    if (P.grad64) P.grad64[(size_t)strip * kCols * 3 + tid] = (double)(float)val;
                }
            }
        } else {
            if (!P.moments) {  // Pearson pass: the moments are an input (P.pmom), nothing to sum; stay for the live pass's counter reset
                if (live) return;
                continue;
            }
            double m[kNM];
#pragma unroll
            for (int k = 0; k < kNM; ++k) m[k] = 0.0;
            // every strip has the chunks 0 .. cmin-1; the chunk rows above have holes (strips of the other parity).
            // Upper-triangle mode: a strip has only its leading chunks (rows up to its last column).
            const int cmin = (P.upper || P.seg_len > 0) ? 0 : min(P.sch.count[0], P.stagger ? P.sch.count[1] : P.sch.count[0]);
            const int nfull = P.nstrips * cmin;
#pragma unroll 4
            for (int sl = tid; sl < nfull; sl += kCombineThreads) {
#pragma unroll
                for (int k = 0; k < kNM; ++k) m[k] += __ldcg(P.mpart + (size_t)sl * kNM + k);
            }
            for (int st = tid; st < P.nstrips; st += kCombineThreads) {
                const int cnt = active_chunks(P, st);
                for (int ch = cmin; ch < cnt; ++ch) {
#pragma unroll
                    for (int k = 0; k < kNM; ++k) m[k] += __ldcg(P.mpart + ((size_t)ch * P.nstrips + st) * kNM + k);
                }
            }
#pragma unroll
            for (int k = 0; k < kNM; ++k) m[k] = warp_sum(m[k]);
            __syncthreads();  // s_m of the previous pass has been read
            if ((tid & 31) == 0) {
#pragma unroll
                for (int k = 0; k < kNM; ++k) s_m[tid >> 5][k] = m[k];
            }
            __syncthreads();
            if (live && tid < kNM) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < kCombineThreads / 32; ++w) s += s_m[w][tid];
                P.moments[tid] = s;
            }
        }
    }
#ifdef HICGAT_TRACE
    if (ctr) ctr[2] = gtimer();
#endif
}

// ------------------------------------------------------------------ variant 1 and the implicit target: per-lane target values
// One CTA per (strip, row chunk), the chunk's x_i staged in shared memory; every lane takes its 4 target values of a row group
//   IMPLICIT = false (variant 1): from the target, with streaming 128-bit ld.global.nc loads (8 per group);
//   IMPLICIT = true  (implicit target, SURVEY.md section 8 row f-4): from nowhere -- on a sparse map every non-edge pair has wish
//     distance `fill` (1.0 after cont2dist: zero contacts map to max/max, utils.py:78-80) and the diagonal 0, so the N x N target
//     need not exist.  The loss against that constant background is FP32 / MUFU bound instead of HBM bound;
//     pairloss_csr_fix_kernel then corrects the nnz pairs that do carry a contact.
// ROWS: upper-triangle mode (chunk_rows clips every strip at its last column, so no row below the diagonal strip is loaded).
// Same decomposition, arithmetic and reductions as the TMA kernels.
// x_i is staged in pieces of at most kStageRows rows, so a chunk of any length fits the default 48 KB of shared memory (the
// layout doubles the chunk length of long row blocks to stay within kMaxChunks).  kStageRows is a multiple of kTileRows: every
// warp visits the same row groups in the same order as with the whole chunk staged at once.
constexpr int kStageRows = 1024;
static_assert(kStageRows % kTileRows == 0, "a staging piece must hold whole tiles");
__host__ __device__ constexpr size_t lane_smem_bytes(int rb) {
    return (sizeof(float4) + sizeof(float2)) * (size_t)(rb < kStageRows ? rb : kStageRows);
}
template <uint32_t MODE, bool ROWS, bool IMPLICIT>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) pairloss_lane_kernel(const Params P) {
    pdl_launch_dependents();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int stage_rows = min(P.rb, kStageRows);
    float4* s_xy = reinterpret_cast<float4*>(smem_raw);                                 // [stage_rows] (x,x,y,y)
    float2* s_z = reinterpret_cast<float2*>(smem_raw + sizeof(float4) * stage_rows);    // [stage_rows] (z,z)
    __shared__ CombineSmem S;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x, chunk = blockIdx.y;
    const int n = P.n;
    const int col0 = strip * kCols + lane * 4;
    int row_begin, nrows;
    const int count = chunk_rows(P, strip, chunk, row_begin, nrows);
    if (chunk >= count || nrows <= 0) return;  // unstaggered strips leave the extra chunk slot empty
    const bool edge = (strip + 1) * kCols > n;
    ColumnRegs c;
    load_columns(c, P.coords, col0, n);
    Acc a;
    acc_zero(a);
    const PearsonCoef pc = pearson_coef<MODE>(P.pmom, n, P.c_mse, P.dyn_alpha);
    const bool can_load = col0 + 3 < P.pitch;  // pitch is a multiple of 4 (0 for the implicit target)
    const float* tbase = P.target + (size_t)(row_begin - P.r0) * P.pitch + col0;
    const int strip_lo = strip * kCols, strip_hi = strip_lo + kCols - 1;
    const float f = P.fill;
    for (int p0 = 0; p0 < nrows; p0 += kStageRows) {
        const int prows = min(kStageRows, nrows - p0);
        if (p0 > 0) __syncthreads();  // every warp is done with the previous piece
        for (int r = threadIdx.x; r < prows; r += kThreads) {
            const float* cr = P.coords + (size_t)(row_begin + p0 + r) * 3;
            float x = cr[0], y = cr[1], z = cr[2];
            s_xy[r] = make_float4(x, x, y, y);
            s_z[r] = make_float2(z, z);
        }
        __syncthreads();
        const int ngroups = (prows + kU - 1) / kU;
        for (int g = warp; g < ngroups; g += kWarps) {
            const int rl = p0 + g * kU, rg = row_begin + rl;
            const int rows_here = min(kU, nrows - rl);
            float4 t[kU];
            if constexpr (IMPLICIT) {
#pragma unroll
                for (int u = 0; u < kU; ++u) t[u] = make_float4(f, f, f, f);
                if (rg + kU - 1 >= strip_lo && rg <= strip_hi) {  // the group touches the diagonal: t_ii = 0
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        const int dc = rg + u - col0;
                        if (dc == 0) t[u].x = 0.f;
                        if (dc == 1) t[u].y = 0.f;
                        if (dc == 2) t[u].z = 0.f;
                        if (dc == 3) t[u].w = 0.f;
                    }
                }
            } else {
                if (rows_here == kU && can_load) {
#pragma unroll
                    for (int u = 0; u < kU; ++u) t[u] = ldg_stream_f4(tbase + (size_t)(rl + u) * P.pitch);
                } else {
#pragma unroll
                    for (int u = 0; u < kU; ++u)
                        t[u] = (u < rows_here && can_load) ? ldg_stream_f4(tbase + (size_t)(rl + u) * P.pitch) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            process_group<MODE, ROWS>(a, c, t, XiPtr{s_xy + g * kU, s_z + g * kU}, rows_here, rg, col0, n, edge, strip_lo, strip_hi, P.c_mse, P.c_l1,
                                      ROWS ? P.rpart + (size_t)strip * P.rpitch + (size_t)(rg - P.r0) * 3 : nullptr, lane, pc);
        }
    }
    park_warp<MODE, ROWS>(a, S, warp, lane);
    __syncthreads();
    publish_cta<MODE>(P, S, strip, chunk, threadIdx.x, kThreads);
}

// Correction of the pairs that carry a contact (CSR rows [r0, r1), warp per row, ROW-side sums: by the
// symmetry of the target the row-side contribution of row i equals what the column-side sum of a
// streamed kernel would have put on locus i over all ranks).  For edge (i, j) with wish value t:
//   loss terms   (d - t)^2 - (d - fill)^2            gradient   c * [(d - t) - (d - fill)] / d * (x_i - x_j)
// Moments are corrected for j > i.  Adds into grad rows [r0, r1) and writes per-CTA f64 partials that the
// last CTA adds to `moments` in CTA order.
template <uint32_t MODE>
__global__ void __launch_bounds__(256) pairloss_csr_fix_kernel(const float* __restrict__ coords, const int32_t* __restrict__ rowptr,
                                                               const int32_t* __restrict__ col, const float* __restrict__ tval, float fill, int n,
                                                               int r0, int r1, float c_mse, float c_l1, double* __restrict__ moments,
                                                               float* __restrict__ grad, double* __restrict__ grad64, double* __restrict__ part,
                                                               unsigned* __restrict__ counter, const double* __restrict__ pmom, int dyn_alpha) {
    __shared__ double s_m[8][kNM];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = r0 + blockIdx.x * 8 + warp;
    double m[kNM];
#pragma unroll
    for (int k = 0; k < kNM; ++k) m[k] = 0.0;
    float lam_a = 0.f, cm = 0.f;
    if constexpr ((MODE & kPearson) != 0) {
        float u;
        const PearsonCoef pc = pearson_coef<MODE>(pmom, n, c_mse, dyn_alpha);
        f2_unpack(pc.lam_a, lam_a, u);
        if constexpr ((MODE & HICGAT_PAIR_GRAD_MSE) != 0) cm = c_mse;
    }
    if (i < r1) {
        const float xi = coords[(size_t)i * 3], yi = coords[(size_t)i * 3 + 1], zi = coords[(size_t)i * 3 + 2];
        float gx = 0.f, gy = 0.f, gz = 0.f;
        for (int k = rowptr[i] + lane; k < rowptr[i + 1]; k += 32) {
            const int j = col[k];
            if (j == i) continue;
            const float t = tval[k];
            const float dx = xi - coords[(size_t)j * 3], dy = yi - coords[(size_t)j * 3 + 1], dz = zi - coords[(size_t)j * 3 + 2];
            const float d2 = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, 1e-30f)));
            const float rs = rsqrt_approx(d2);
            const float d = d2 * rs;
            const float et = d - t, ef = d - fill;
            const double dsee = (double)et * et - (double)ef * ef;
            m[0] += dsee;
            float w = 0.f;
            // Pearson pass: [c_mse (d - t) + lamA (t - beta d - kappa)] - [the same at t = fill] = (lamA - c_mse) (t - fill)
            if constexpr ((MODE & kPearson) != 0) w = (lam_a * (t - fill) + cm * (fill - t)) * rs;
            else if constexpr ((MODE & 3u) == HICGAT_PAIR_GRAD_MSE) w = c_mse * (fill - t) * rs;
            else if constexpr ((MODE & 3u) == HICGAT_PAIR_GRAD_L1) w = c_l1 * (copysignf(1.f, et) - copysignf(1.f, ef)) * rs;
            else if constexpr ((MODE & 3u) == 3u) w = (c_mse * (fill - t) + c_l1 * (copysignf(1.f, et) - copysignf(1.f, ef))) * rs;
            gx = fmaf(w, dx, gx); gy = fmaf(w, dy, gy); gz = fmaf(w, dz, gz);
            if constexpr ((MODE & (kMomFull | kMomLight)) != 0) {
                if (j > i) {
                    m[6] += (double)d * ((double)t - (double)fill);
                    m[7] += dsee;
                    if constexpr ((MODE & kMomFull) != 0) {
                        m[1] += (double)fabsf(et) - (double)fabsf(ef);
                        m[4] += (double)t - (double)fill;
                        m[5] += (double)t * t - (double)fill * fill;
                    }
                }
            }
        }
        if constexpr (has_grad(MODE)) {
            gx = warp_sum(gx); gy = warp_sum(gy); gz = warp_sum(gz);
            if (lane == 0) {
                if (grad) { grad[(size_t)i * 3] += gx; grad[(size_t)i * 3 + 1] += gy; grad[(size_t)i * 3 + 2] += gz; }
                if (grad64) {  // packed layout holds f32 values widened: keep that invariant
                    grad64[(size_t)i * 3] = (double)(float)((float)grad64[(size_t)i * 3] + gx);
                    grad64[(size_t)i * 3 + 1] = (double)(float)((float)grad64[(size_t)i * 3 + 1] + gy);
                    grad64[(size_t)i * 3 + 2] = (double)(float)((float)grad64[(size_t)i * 3 + 2] + gz);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < kNM; ++k) m[k] = warp_sum(m[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kNM; ++k) s_m[warp][k] = m[k];
    }
    __syncthreads();
    if (threadIdx.x < kNM) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += s_m[w][threadIdx.x];
        __stcg(part + (size_t)blockIdx.x * kNM + threadIdx.x, s);
    }
    __syncthreads();
    __shared__ unsigned ticket;
    if (threadIdx.x == 0) {
        __threadfence();
        ticket = atomicAdd(counter, 1u);
        __threadfence();
    }
    __syncthreads();
    if (ticket != gridDim.x - 1) return;
    if (threadIdx.x == 0) *counter = 0u;
    // last CTA: add all partials to the moments in CTA order (thread t: CTAs t, t+256, ...; then lanes, warps)
#pragma unroll
    for (int k = 0; k < kNM; ++k) m[k] = 0.0;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += 256) {
#pragma unroll
        for (int k = 0; k < kNM; ++k) m[k] += __ldcg(part + (size_t)b * kNM + k);
    }
#pragma unroll
    for (int k = 0; k < kNM; ++k) m[k] = warp_sum(m[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kNM; ++k) s_m[warp][k] = m[k];
    }
    __syncthreads();
    if (threadIdx.x < kNM && moments) {  // no moments in the Pearson pass
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += s_m[w][threadIdx.x];
        moments[threadIdx.x] += s;
    }
}

// ------------------------------------------------------------------ variant 0: TMA + mbarrier ring
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// explicit shared-space accesses: the ring pointer went through an integer round trip (128-byte
// alignment), so plain C++ dereferences would compile to generic LD/ST with 64-bit address math
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f2(uint32_t addr, float a, float b) {
    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void XiAddr::load(int u, float4& oxy, float2& oz) const {
    oxy = lds_f4(xy + u * 16);
    oz = lds_f2(z + u * 8);
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}

// Every consumer warp runs its OWN ring: lane 0 issues a TMA box of 8 rows x 128 columns (4 KB)
// per stage for the warp's rows of tile t and refills the slot right after the warp has consumed
// it -- no producer warp, no empty barriers, no cross-warp synchronisation in the main loop.
template <uint32_t MODE, bool ROWS>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) pairloss_tma_kernel(const __grid_constant__ CUtensorMap tmap, const Params P) {
    pdl_launch_dependents();
    extern __shared__ unsigned char smem_raw[];
    unsigned char* ring = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
    __shared__ __align__(8) uint64_t full_bar[kWarps][kStages];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strip = blockIdx.x, chunk = blockIdx.y;
    const int n = P.n;
    int row_begin, nrows;
    HICGAT_TR(0);
#ifdef HICGAT_TRACE
    { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); HICGAT_TRV(6, (unsigned long long)smid); HICGAT_TRV(7, 0ull); }
#endif
    const int count = chunk_rows(P, strip, chunk, row_begin, nrows);
    if (chunk >= count || nrows <= 0) return;  // unstaggered strips leave the extra chunk slot empty; upper mode clips strips at the diagonal
    const int ntiles = (nrows + kTileRows - 1) / kTileRows;
    const int col0 = strip * kCols + lane * 4;
    const bool edge = (strip + 1) * kCols > n;
    const int strip_lo = strip * kCols, strip_hi = strip_lo + kCols - 1;
    unsigned char* wring = ring + (size_t)warp * (kStages * kSlotBytes);   // this warp's slots
    const int wrow = warp * kU;                                             // this warp's rows inside a tile

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(&full_bar[warp][s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    }
    pdl_wait();  // everything the previous kernels of this stream wrote (coordinates, a freshly built target) is visible from here on
    __syncwarp();

    // x_i staging: lane k < 24 owns component k%3 of row k/3 and writes it duplicated (v,v)
    const int xi_row = lane / 3, xi_comp = lane - xi_row * 3;
    auto xi_fetch = [&](int t) -> float {
        const int gr = min(row_begin + t * kTileRows + wrow + xi_row, n - 1);
        return lane < 24 ? __ldg(P.coords + (size_t)gr * 3 + xi_comp) : 0.f;
    };
    const uint32_t wring_s = smem_u32(wring);
    const uint32_t xi_off = kSubTileBytes + (xi_comp < 2 ? xi_row * 16 + xi_comp * 8 : kU * 16 + xi_row * 8);
    auto xi_store = [&](int s, float v) {
        if (lane < 24) sts_f2(wring_s + s * kSlotBytes + xi_off, v, v);
    };
    auto issue = [&](int t, int s) {  // lane 0 only
        mbar_arrive_expect_tx(&full_bar[warp][s], (uint32_t)kSubTileBytes);
        tma_load_2d(wring + (size_t)s * kSlotBytes, &tmap, strip * kCols, (row_begin - P.r0) + t * kTileRows + wrow, &full_bar[warp][s]);
    };
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
        if (s < ntiles) {
            if (lane == 0) issue(s, s);
            xi_store(s, xi_fetch(s));
        }
    }
    ColumnRegs c;
    load_columns(c, P.coords, col0, n);
    Acc a;
    acc_zero(a);
    const PearsonCoef pc = pearson_coef<MODE>(P.pmom, n, P.c_mse, P.dyn_alpha);
    __syncwarp();

    for (int t = 0; t < ntiles; ++t) {
        const int s = t % kStages, use = t / kStages;
        const bool refill = t + kStages < ntiles;
        const float xi_next = refill ? xi_fetch(t + kStages) : 0.f;   // in flight during the compute below
        mbar_wait(&full_bar[warp][s], (uint32_t)(use & 1));
#ifdef HICGAT_TRACE
        if (t == 0) HICGAT_TR(1);
#endif
        const uint32_t slot = wring_s + s * kSlotBytes;
        const XiAddr xi{slot + kSubTileBytes, slot + kSubTileBytes + kU * 16};
        const int rows_here = max(0, min(kU, nrows - (t * kTileRows + wrow)));
        float4 tv[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) tv[u] = lds_f4(slot + lane * 16 + u * (kCols * 4));
        const int rg = row_begin + t * kTileRows + wrow;
        process_group<MODE, ROWS>(a, c, tv, xi, rows_here, rg, col0, n, edge, strip_lo, strip_hi, P.c_mse, P.c_l1,
                                  ROWS ? P.rpart + (size_t)strip * P.rpitch + (size_t)(rg - P.r0) * 3 : nullptr, lane, pc);
        __syncwarp();  // every lane is done with slot s
        if (refill) {
            if (lane == 0) issue(t + kStages, s);
            xi_store(s, xi_next);
        }
    }
    HICGAT_TR(2);
    __syncthreads();  // all rings drained: the dynamic shared memory is reused for the combine
    CombineSmem& S = *reinterpret_cast<CombineSmem*>(ring);
    park_warp<MODE, ROWS>(a, S, warp, lane);
    __syncthreads();
    publish_cta<MODE>(P, S, strip, chunk, threadIdx.x, kThreads);
    HICGAT_TR(3);
    HICGAT_TR(5);
}

// ------------------------------------------------------------------ variant 3: persistent CTAs, dynamic item queue
// Same tiles, arithmetic and partial layout as pairloss_tma_kernel, but 2 x 148 CTAs stay resident and pull (chunk, strip) items
// from an atomic counter.  What it buys on small row blocks (a 1/8 shard of the 50k-locus map, the 10k-locus map), where the
// one-CTA-per-item kernel loses 25-40 % to the per-item prologue (~5 us: barrier init, tensor-map fetch, first-tile latency, column
// loads, exit) and to wave quantisation:
//   * a warp that has finished its rows of the current item immediately issues the first TMA boxes of the NEXT item into its ring
//     (the ring and its mbarrier phases simply run on across items), so the next item's data is in flight during the CTA-level combine;
//   * items can be short (128 .. 2048 rows), and the queue balances them dynamically: the slots run dry within one short item.
// Partials are still stored per item (chunk * nstrips + strip) and summed by the combine kernel in a fixed order, so the result does
// not depend on which CTA processed which item: bit-reproducible.
struct PersistSmem {
    float g[kWarps / 2][kCols * 3 + 4];   // two-phase CTA combine: the upper half of the warps parks, the lower half adds
    double m[kWarps][kNM];
    int item[2];
};
constexpr int kPersistSmem = kTmaSmem;     // the ring only: the combine area is static shared memory (it must not alias a ring in use)

__device__ __forceinline__ void decode_item(const Params& P, int item, int& strip, int& chunk, int& row_begin, int& nrows) {
    int lo = 0, hi = P.sch.count[0];  // item_base[lo] <= item < item_base[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (P.item_base[mid] <= item) lo = mid; else hi = mid;
    }
    chunk = lo;
    const int first_strip = P.nstrips - (P.item_base[lo + 1] - P.item_base[lo]);
    strip = first_strip + (item - P.item_base[lo]);
    chunk_rows(P, strip, chunk, row_begin, nrows);
}

template <uint32_t MODE, bool ROWS>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) pairloss_tma_persist_kernel(const __grid_constant__ CUtensorMap tmap, const Params P) {
    pdl_launch_dependents();
    extern __shared__ unsigned char smem_raw[];
    unsigned char* ring = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
    __shared__ __align__(8) uint64_t full_bar[kWarps][kStages];
    __shared__ PersistSmem S;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = P.n;
    unsigned char* wring = ring + (size_t)warp * (kStages * kSlotBytes);
    const uint32_t wring_s = smem_u32(wring);
    const int wrow = warp * kU;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(&full_bar[warp][s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    }
    pdl_wait();
    if (threadIdx.x == 0) {
        S.item[0] = (int)atomicAdd(P.work_counter, 1u);
        S.item[1] = (int)atomicAdd(P.work_counter, 1u);
    }
    __syncthreads();

    const int xi_row = lane / 3, xi_comp = lane - xi_row * 3;
    const uint32_t xi_off = kSubTileBytes + (xi_comp < 2 ? xi_row * 16 + xi_comp * 8 : kU * 16 + xi_row * 8);
    unsigned gt = 0;  // tiles this warp has issued so far: tile g lives in slot g % kStages and is the (g / kStages)-th use of it

    // x_i of tile t of an item: lane k < 24 owns component k % 3 of row k / 3 (stored duplicated (v, v) next to the tile)
    auto xi_fetch = [&](int row_begin, int t) -> float {
        const int gr = min(row_begin + t * kTileRows + wrow + xi_row, n - 1);
        return lane < 24 ? __ldg(P.coords + (size_t)gr * 3 + xi_comp) : 0.f;
    };
    // issue tile t of an item (row_begin, strip) as this warp's ring entry number g; v = xi_fetch(row_begin, t), fetched earlier
    auto issue = [&](int strip, int row_begin, int t, unsigned g, float v) {
        const int s = (int)(g % kStages);
        if (lane == 0) {
            mbar_arrive_expect_tx(&full_bar[warp][s], (uint32_t)kSubTileBytes);
            tma_load_2d(wring + (size_t)s * kSlotBytes, &tmap, strip * kCols, (row_begin - P.r0) + t * kTileRows + wrow, &full_bar[warp][s]);
        }
        if (lane < 24) sts_f2(wring_s + s * kSlotBytes + xi_off, v, v);
    };

    int cur = S.item[0], nxt = S.item[1];
    int strip = 0, chunk = 0, row_begin = 0, nrows = 0;
    if (cur < P.nitems) {
        decode_item(P, cur, strip, chunk, row_begin, nrows);
        const int nt = (nrows + kTileRows - 1) / kTileRows;
        for (int t = 0; t < kStages && t < nt; ++t) issue(strip, row_begin, t, gt + t, xi_fetch(row_begin, t));
    }
    __syncwarp();
    for (int it = 0; cur < P.nitems; ++it) {
        const int ntiles = (nrows + kTileRows - 1) / kTileRows;
        const int col0 = strip * kCols + lane * 4;
        const bool edge = (strip + 1) * kCols > n;
        const int strip_lo = strip * kCols, strip_hi = strip_lo + kCols - 1;
        ColumnRegs c;
        load_columns(c, P.coords, col0, n);
        Acc a;
        acc_zero(a);
        const PearsonCoef pc = pearson_coef<MODE>(P.pmom, n, P.c_mse, P.dyn_alpha);
        for (int t = 0; t < ntiles; ++t) {
            const unsigned g = gt + t;
            const int s = (int)(g % kStages);
            const bool refill = t + kStages < ntiles;
            const float xi_next = refill ? xi_fetch(row_begin, t + kStages) : 0.f;   // in flight during the compute below
            mbar_wait(&full_bar[warp][s], (g / kStages) & 1u);
            const uint32_t slot = wring_s + s * kSlotBytes;
            const XiAddr xi{slot + kSubTileBytes, slot + kSubTileBytes + kU * 16};
            const int rows_here = max(0, min(kU, nrows - (t * kTileRows + wrow)));
            float4 tv[kU];
#pragma unroll
            for (int u = 0; u < kU; ++u) tv[u] = lds_f4(slot + lane * 16 + u * (kCols * 4));
            const int rg = row_begin + t * kTileRows + wrow;
            process_group<MODE, ROWS>(a, c, tv, xi, rows_here, rg, col0, n, edge, strip_lo, strip_hi, P.c_mse, P.c_l1,
                                      ROWS ? P.rpart + (size_t)strip * P.rpitch + (size_t)(rg - P.r0) * 3 : nullptr, lane, pc);
            __syncwarp();  // every lane is done with slot s
            if (refill) issue(strip, row_begin, t + kStages, g + kStages, xi_next);
        }
        gt += (unsigned)ntiles;
        // this warp's ring is empty: start the NEXT item's first tiles before the CTA-level combine
        int nstrip = 0, nchunk = 0, nrow_begin = 0, nnrows = 0;
        if (nxt < P.nitems) {
            decode_item(P, nxt, nstrip, nchunk, nrow_begin, nnrows);
            const int nt = (nnrows + kTileRows - 1) / kTileRows;
            for (int t = 0; t < kStages && t < nt; ++t) issue(nstrip, nrow_begin, t, gt + t, xi_fetch(nrow_begin, t));
        }
        // ---- CTA combine in two phases (half the shared memory): warps 4..7 park, warps 0..3 add their own on top
        constexpr bool kMom = (MODE & (kMomFull | kMomLight)) != 0;
        {
            double m[kNM];
#pragma unroll
            for (int k = 0; k < kNM; ++k) m[k] = 0.0;
            const double seu = (double)f2_hsum(a.seu);
            m[0] = (double)f2_hsum(a.see) + (ROWS ? 2.0 * seu : seu);
            if constexpr (kMom) {
                m[2] = (double)f2_hsum(a.sd); m[3] = (double)f2_hsum(a.sdd); m[6] = (double)f2_hsum(a.sdt); m[7] = seu;
                if constexpr ((MODE & kMomFull) != 0) {
                    m[1] = (double)a.sabs0 + (double)a.sabs1; m[4] = (double)f2_hsum(a.st); m[5] = (double)f2_hsum(a.stt);
                }
            }
#pragma unroll
            for (int k = 0; k < kNM; ++k)
                if (k == 0 || kMom) m[k] = warp_sum(m[k]);
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < kNM; ++k) S.m[warp][k] = m[k];
            }
        }
        float gv[2][6];
        if constexpr (has_grad(MODE)) {
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                f2_unpack(a.gx[p], gv[p][0], gv[p][3]);
                f2_unpack(a.gy[p], gv[p][1], gv[p][4]);
                f2_unpack(a.gz[p], gv[p][2], gv[p][5]);
            }
            if (warp >= kWarps / 2) {
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    float* dst = &S.g[warp - kWarps / 2][(lane * 4 + 2 * p) * 3];
#pragma unroll
                    for (int q = 0; q < 6; ++q) dst[q] = gv[p][q];
                }
            }
        }
        __syncthreads();
        if constexpr (has_grad(MODE)) {
            if (warp < kWarps / 2) {
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    float* dst = &S.g[warp][(lane * 4 + 2 * p) * 3];
#pragma unroll
                    for (int q = 0; q < 6; ++q) dst[q] += gv[p][q];   // fixed order: (w + 4) + w
                }
            }
        }
        __syncthreads();
        {
            const int cta = chunk * P.nstrips + strip;
            if constexpr (has_grad(MODE)) {
                float* gp = P.gpart + (size_t)cta * (kCols * 3);
                for (int i = threadIdx.x; i < kCols * 3; i += kThreads) {
                    float sum = 0.f;
#pragma unroll
                    for (int w = 0; w < kWarps / 2; ++w) sum += S.g[w][i];
                    __stcg(gp + i, sum);
                }
            }
            if (threadIdx.x < kNM) {
                double sum = 0.0;
#pragma unroll
                for (int w = 0; w < kWarps; ++w) sum += S.m[w][threadIdx.x];
                __stcg(P.mpart + (size_t)cta * kNM + threadIdx.x, sum);
            }
            if (threadIdx.x == 0) S.item[it & 1] = (int)atomicAdd(P.work_counter, 1u);  // the item after next
        }
        __syncthreads();
        cur = nxt;
        nxt = S.item[it & 1];
        strip = nstrip; chunk = nchunk; row_begin = nrow_begin; nrows = nnrows;
    }
}

// ------------------------------------------------------------------ variant 4: static warp partition
// For SMALL row blocks (a 1/8 shard of the 50k-locus map, the 10k-locus map) the item kernels lose 25-40 % to per-item overhead and to
// the last, partly filled wave.  Here nothing is dispatched at all: the work of the block, written as the strip-major sequence of
// (strip, row) units -- strip s contributes rows_s = clamp(128 (s + 1) - r0, 0, nrows) units in upper-triangle mode, nrows otherwise --
// is cut into 2 368 equal runs, one per resident warp (2 CTAs x 8 warps x 148 SMs).  A warp streams its run through its own TMA ring in
// 8-row tiles, publishes one partial per strip it touches (1-3) straight from its registers, and exits: no CTA-level synchronisation,
// no queue, no tail beyond one tile.  rows_s is piecewise linear in s, so strip offsets and their inverse are closed forms (no tables).
// Partials are indexed by (strip, segment) and summed by the combine kernel in segment (= row) order: bit-reproducible.
__device__ __forceinline__ int64_t strip_rows_of(const Params& P, int s) {
    if (!P.upper) return P.r1 - P.r0;
    const int64_t v = (int64_t)(s + 1) * kCols - P.r0;
    const int64_t nrows = P.r1 - P.r0;
    return v < 0 ? 0 : (v > nrows ? nrows : v);
}
// number of (strip, row) units before strip s
__device__ __forceinline__ int64_t strip_offset(const Params& P, int s) {
    const int64_t nrows = P.r1 - P.r0;
    if (!P.upper) return (int64_t)s * nrows;
    if (s <= P.seg_sa) return 0;
    const int64_t m = (s < P.seg_sb ? s : P.seg_sb) - P.seg_sa;       // strips in the growing part
    int64_t off = m * P.seg_f + 64 * m * (m - 1);
    if (s > P.seg_sb) off += (int64_t)(s - P.seg_sb) * nrows;
    return off;
}
__device__ __forceinline__ int strip_of_unit(const Params& P, int64_t p) {
    const int64_t nrows = P.r1 - P.r0;
    if (!P.upper) return (int)(p / nrows);
    const int64_t off_b = strip_offset(P, P.seg_sb);
    if (p >= off_b) return P.seg_sb + (int)((p - off_b) / nrows);
    // largest m with m f + 64 m (m - 1) <= p
    const double b = (double)P.seg_f - 64.0;
    int64_t m = (int64_t)((-b + sqrt(b * b + 256.0 * (double)p)) / 128.0);
    if (m < 0) m = 0;
    while (m > 0 && m * P.seg_f + 64 * m * (m - 1) > p) --m;
    while ((m + 1) * P.seg_f + 64 * (m + 1) * m <= p) ++m;
    return P.seg_sa + (int)m;
}
__device__ __forceinline__ int strip_segments(const Params& P, int s) {  // warps that touch strip s
    const int64_t rows = strip_rows_of(P, s);
    if (rows <= 0) return 0;
    const int64_t off = strip_offset(P, s);
    return (int)((off + rows - 1) / P.seg_len - off / P.seg_len) + 1;
}

template <uint32_t MODE, bool ROWS>
__global__ void __launch_bounds__(kThreads, kCtasPerSm) pairloss_tma_warp_kernel(const __grid_constant__ CUtensorMap tmap, const Params P) {
    pdl_launch_dependents();
    extern __shared__ unsigned char smem_raw[];
    unsigned char* ring = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
    __shared__ __align__(8) uint64_t full_bar[kWarps][kStages];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = P.n;
    unsigned char* wring = ring + (size_t)warp * (kStages * kSlotBytes);
    const uint32_t wring_s = smem_u32(wring);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(&full_bar[warp][s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    }
    pdl_wait();
    __syncwarp();
    const int64_t gw = (int64_t)blockIdx.x * kWarps + warp;
    int64_t p = gw * P.seg_len;
    const int64_t pend = p + P.seg_len < P.seg_total ? p + P.seg_len : P.seg_total;
    const int xi_row = lane / 3, xi_comp = lane - xi_row * 3;
    const uint32_t xi_off = kSubTileBytes + (xi_comp < 2 ? xi_row * 16 + xi_comp * 8 : kU * 16 + xi_row * 8);
    unsigned gt = 0;
    while (p < pend) {
        const int strip = strip_of_unit(P, p);
        const int64_t soff = strip_offset(P, strip);
        const int row_lo = (int)(p - soff);                                  // local rows (offsets from r0) of this strip
        int64_t take = strip_rows_of(P, strip) - row_lo;
        if (take > pend - p) take = pend - p;
        const int nrows = (int)take;
        const int row_begin = P.r0 + row_lo;
        const int ntiles = (nrows + kU - 1) / kU;
        const int col0 = strip * kCols + lane * 4;
        const bool edge = (strip + 1) * kCols > n;
        const int strip_lo = strip * kCols, strip_hi = strip_lo + kCols - 1;
        auto xi_fetch = [&](int t) -> float {
            const int gr = min(row_begin + t * kU + xi_row, n - 1);
            return lane < 24 ? __ldg(P.coords + (size_t)gr * 3 + xi_comp) : 0.f;
        };
        auto issue = [&](int t, unsigned g, float v) {
            const int s = (int)(g % kStages);
            if (lane == 0) {
                mbar_arrive_expect_tx(&full_bar[warp][s], (uint32_t)kSubTileBytes);
                tma_load_2d(wring + (size_t)s * kSlotBytes, &tmap, strip * kCols, row_lo + t * kU, &full_bar[warp][s]);
            }
            if (lane < 24) sts_f2(wring_s + s * kSlotBytes + xi_off, v, v);
        };
        for (int t = 0; t < kStages && t < ntiles; ++t) issue(t, gt + t, xi_fetch(t));
        ColumnRegs c;
        load_columns(c, P.coords, col0, n);
        Acc a;
        acc_zero(a);
        const PearsonCoef pc = pearson_coef<MODE>(P.pmom, n, P.c_mse, P.dyn_alpha);
        __syncwarp();
        for (int t = 0; t < ntiles; ++t) {
            const unsigned g = gt + t;
            const int s = (int)(g % kStages);
            const bool refill = t + kStages < ntiles;
            const float xi_next = refill ? xi_fetch(t + kStages) : 0.f;
            mbar_wait(&full_bar[warp][s], (g / kStages) & 1u);
            const uint32_t slot = wring_s + s * kSlotBytes;
            const XiAddr xi{slot + kSubTileBytes, slot + kSubTileBytes + kU * 16};
            const int rows_here = min(kU, nrows - t * kU);
            float4 tv[kU];
#pragma unroll
            for (int u = 0; u < kU; ++u) tv[u] = lds_f4(slot + lane * 16 + u * (kCols * 4));
            const int rg = row_begin + t * kU;
            process_group<MODE, ROWS>(a, c, tv, xi, rows_here, rg, col0, n, edge, strip_lo, strip_hi, P.c_mse, P.c_l1,
                                      ROWS ? P.rpart + (size_t)strip * P.rpitch + (size_t)(rg - P.r0) * 3 : nullptr, lane, pc);
            __syncwarp();
            if (refill) issue(t + kStages, g + kStages, xi_next);
        }
        gt += (unsigned)ntiles;
        // ---- publish this warp's partial of the strip: slot (segment index, strip)
        const int seg = (int)(gw - soff / P.seg_len);
        const size_t slot_id = (size_t)seg * P.nstrips + strip;
        if constexpr (has_grad(MODE)) {
            float* gp = P.gpart + slot_id * (kCols * 3) + lane * 12;
            float x0, x1, y0, y1, z0, z1, x2, x3, y2, y3, z2, z3;
            f2_unpack(a.gx[0], x0, x1); f2_unpack(a.gy[0], y0, y1); f2_unpack(a.gz[0], z0, z1);
            f2_unpack(a.gx[1], x2, x3); f2_unpack(a.gy[1], y2, y3); f2_unpack(a.gz[1], z2, z3);
            __stcg(reinterpret_cast<float4*>(gp), make_float4(x0, y0, z0, x1));
            __stcg(reinterpret_cast<float4*>(gp) + 1, make_float4(y1, z1, x2, y2));
            __stcg(reinterpret_cast<float4*>(gp) + 2, make_float4(z2, x3, y3, z3));
        }
        {
            constexpr bool kMom = (MODE & (kMomFull | kMomLight)) != 0;
            double m[kNM];
#pragma unroll
            for (int k = 0; k < kNM; ++k) m[k] = 0.0;
            const double seu = (double)f2_hsum(a.seu);
            m[0] = (double)f2_hsum(a.see) + (ROWS ? 2.0 * seu : seu);
            if constexpr (kMom) {
                m[2] = (double)f2_hsum(a.sd); m[3] = (double)f2_hsum(a.sdd); m[6] = (double)f2_hsum(a.sdt); m[7] = seu;
                if constexpr ((MODE & kMomFull) != 0) {
                    m[1] = (double)a.sabs0 + (double)a.sabs1; m[4] = (double)f2_hsum(a.st); m[5] = (double)f2_hsum(a.stt);
                }
            }
#pragma unroll
            for (int k = 0; k < kNM; ++k)
                if (k == 0 || kMom) m[k] = warp_sum(m[k]);
            if (lane < kNM) {
                double v = 0.0;
#pragma unroll
                for (int k = 0; k < kNM; ++k) v = lane == k ? m[k] : v;
                __stcg(P.mpart + slot_id * kNM + lane, v);
            }
        }
        p += take;
    }
}

// ------------------------------------------------------------------ materialising variant
__global__ void pairdist_fwd_kernel(const float* __restrict__ coords, int n, float* __restrict__ dist, int64_t pitch) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int i0 = blockIdx.y * 16;
    if (j >= n) return;
    const float xj = coords[j * 3], yj = coords[j * 3 + 1], zj = coords[j * 3 + 2];
    for (int i = i0; i < min(i0 + 16, n); ++i) {
        const float dx = xj - __ldg(coords + i * 3), dy = yj - __ldg(coords + i * 3 + 1), dz = zj - __ldg(coords + i * 3 + 2);
        dist[(size_t)i * pitch + j] = sqrtf(dx * dx + dy * dy + dz * dz);
    }
}

// grad_coords[i] = sum_j (G[i,j] + G[j,i]) (x_i - x_j)/d_ij ; one warp per locus i
__global__ void pairdist_bwd_kernel(const float* __restrict__ coords, int n, const float* __restrict__ G, int64_t pitch, float* __restrict__ gc) {
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    const float xi = coords[i * 3], yi = coords[i * 3 + 1], zi = coords[i * 3 + 2];
    float gx = 0.f, gy = 0.f, gz = 0.f;
    for (int j = lane; j < n; j += 32) {
        const float dx = xi - coords[j * 3], dy = yi - coords[j * 3 + 1], dz = zi - coords[j * 3 + 2];
        const float d2 = dx * dx + dy * dy + dz * dz;
        if (d2 > 0.f) {
            const float w = (G[(size_t)i * pitch + j] + G[(size_t)j * pitch + i]) * rsqrtf(d2);
            gx += w * dx; gy += w * dy; gz += w * dz;
        }
    }
    gx = warp_sum(gx); gy = warp_sum(gy); gz = warp_sum(gz);
    if (lane == 0) { gc[i * 3] = gx; gc[i * 3 + 1] = gy; gc[i * 3 + 2] = gz; }
}

// ------------------------------------------------------------------ host side
int g_rows_per_cta = 0;
int g_stagger = 1;
int g_variant = 0;  // 0 = TMA ring (default), 1 = per-lane streaming loads
const bool g_pdl = []() { const char* e = getenv("HICGAT_NO_PDL"); return !(e && e[0] == '1'); }();  // A/B: plain launch of the combine kernel

int pick_rows_per_cta(int64_t nrows, int nstrips, int variant) {
    if (g_rows_per_cta > 0) return variant == 0 ? (g_rows_per_cta + kTileRows - 1) / kTileRows * kTileRows : g_rows_per_cta;
    if (nrows <= 0) return kTileRows;  // empty row block: nothing is launched
    if (variant == 0) {
        // One CTA per (column strip, row chunk) item, 2 resident CTAs per SM.  Long chunks keep the
        // per-CTA prologue / combine and the partial buffers small; what matters then is the wave
        // quantisation ceil(items / 296) / (items / 296).  Among chunk lengths of 1024..4096 rows
        // (shorter only when the block would otherwise give fewer than two items per CTA slot)
        // pick the one with the smallest makespan estimate, preferring longer chunks on ties.
        int64_t nch_lo = (nrows + 4095) / 4096, nch_hi = nrows / 1024;
        int64_t nch_items = (2 * kCtaSlots + nstrips - 1) / nstrips;
        if (nch_items > (nrows + kTileRows - 1) / kTileRows) nch_items = (nrows + kTileRows - 1) / kTileRows;
        if (nch_hi < nch_items) nch_hi = nch_items;
        if (nch_lo < 1) nch_lo = 1;
        if (nch_hi < nch_lo) nch_hi = nch_lo;
        int best_rb = kTileRows;
        double best = 1e30;
        for (int64_t nch = nch_lo; nch <= nch_hi; ++nch) {
            const int64_t rb = ((nrows + nch - 1) / nch + kTileRows - 1) / kTileRows * kTileRows;
            const int64_t chunks = (nrows + rb - 1) / rb;
            const double items = (double)nstrips * (double)chunks;
            const double cost = ceil(items / kCtaSlots) * ((double)rb + 96.0);  // rows per CTA slot + per-CTA overhead
            if (cost < best * 0.999) {
                best = cost;
                best_rb = (int)rb;
            }
        }
        return best_rb;
    }
    // largest chunk that still gives >= ~6 CTAs per SM (148 SMs); bounds the partial buffers
    const int64_t want = 148 * 6;
    int rb = 1024;
    while (rb > 64 && (int64_t)nstrips * ((nrows + rb - 1) / rb) < want) rb >>= 1;
    return rb;
}

struct Layout {
    int nstrips, rb, nchunks, stagger;
    Schedule sch;
    size_t nslots;           // partial slots in gpart / mpart = nstrips * nchunks
    size_t off_gpart, off_mpart, off_rpart, off_counter, total;
    int64_t rpitch;          // upper-triangle mode: floats per strip in rpart (0 otherwise)
    int persistent;          // variant 3: item queue
    int nitems;
    int item_base[kMaxChunks + 1];
    int64_t seg_len, seg_total;  // variant 4: static warp partition (seg_len = 0 otherwise)
    int seg_sa, seg_sb, seg_f, seg_warps;
    int rs_first, rs_count, rs_groups;       // combine kernel: segmented row-side sums (upper-triangle mode, short row blocks)
    size_t off_rs_ticket, off_rs_scratch;
};

int g_rs_groups_max = 4;  // hicgat_pairloss_set_combine: 1 = one combine CTA per strip (no segments)
int g_rs_min_strips = 96; // shortest segment worth a CTA of its own (measured on 1/8 .. 1/2 blocks of a 390-strip map: chains of
                          // 390 / 338 strips gain 10 % / 3 % of the whole loss evaluation from 4 / 3 segments, a 138-strip chain loses 2 %)

// Upper-triangle mode: how many CTAs share the row-side sums of one strip of this block's loci (see pairloss_combine_kernel), and
// the workspace behind it.  At most one wave of row-side CTAs (2 per SM) and g_rs_groups_max segments of at least g_rs_min_strips strips.
void add_rowside_layout(Layout& L, int64_t r0, int64_t r1, bool sym) {
    L.rs_first = 0;
    L.rs_count = 0;
    L.rs_groups = 1;
    L.off_rs_ticket = L.off_rs_scratch = L.total;
    if (!sym || r1 <= r0) return;
    L.rs_first = (int)(r0 / kCols);
    L.rs_count = (int)((r1 - 1) / kCols) - L.rs_first + 1;
    int g = std::min((2 * 148) / L.rs_count, g_rs_groups_max);
    const int longest = L.nstrips - L.rs_first;
    while (g > 1 && (longest + g - 1) / g < g_rs_min_strips) --g;
    L.rs_groups = std::max(g, 1);
    if (L.rs_groups > 1) {
        L.off_rs_ticket = align_up(L.total, 256);
        L.off_rs_scratch = L.off_rs_ticket + align_up(sizeof(unsigned) * (size_t)L.rs_count, 256);
        L.total = L.off_rs_scratch + sizeof(double) * (size_t)L.rs_count * L.rs_groups * kCols * 3;
    }
}

int g_tail_depth = -1;    // -1 = library default; >= 0: hicgat_pairloss_set_schedule
int g_tail_min_rows = 256;

// Chunk lengths of one strip: `bulk` chunks of (about) rb rows followed by a tail of `depth` chunks that
// halve each time (rb/2, rb/4, ... >= tail_min).  The hardware dispatches CTAs in (chunk, strip) order, so
// the tail items are the ones that run last: the slots run dry within one SHORT item of each other
// instead of one full-length item (measured on row blocks of 5-10k rows: the last 20-25 % of the kernel
// ran with < 40 % of the CTA slots busy).  The staggered table starts with half a chunk and gets the
// other half back right before the tail.  `unit` = rounding of the chunk lengths.
void build_schedule(int64_t nrows, int rb, int depth, int tail_min, bool stagger, int unit, Schedule& S) {
    auto round_up = [&](int64_t v) { return (int)((v + unit - 1) / unit * unit); };
    int tail[16];
    int ntail = 0;
    int64_t tail_rows = 0;
    for (int i = 1; i <= depth && ntail < 16; ++i) {
        int t = round_up(rb >> i);
        if (t < tail_min) t = round_up(tail_min);
        if (t >= rb) break;                             // chunks are already at the minimum
        if (tail_rows + t + rb / 2 > nrows) break;      // keep at least half a bulk chunk
        tail[ntail++] = t;
        tail_rows += t;
        if (t == round_up(tail_min)) break;             // no point in repeating the minimum
    }
    const int64_t bulk_rows = nrows - tail_rows;
    int nbulk = (int)((bulk_rows + rb - 1) / rb);
    if (nbulk < 1) nbulk = 1;
    const int blen = round_up((bulk_rows + nbulk - 1) / nbulk);
    for (int par = 0; par < 2; ++par) {
        int* b = S.bounds[par];
        int c = 0;
        int64_t pos = 0;
        b[0] = 0;
        auto push = [&](int64_t len, int64_t limit) {
            if (len <= 0 || pos >= limit || c >= kMaxChunks) return;
            pos = pos + len < limit ? pos + len : limit;
            b[++c] = (int)pos;
        };
        const int half = (par == 1 && stagger) ? round_up(blen / 2) : 0;
        if (half) push(half, bulk_rows);
        for (int k = 0; k < nbulk; ++k) push(blen, bulk_rows);
        if (pos < bulk_rows) push(bulk_rows - pos, bulk_rows);
        for (int k = 0; k < ntail; ++k) push(tail[k], nrows);
        if (pos < nrows) {  // out of table entries (never with rb >= nrows / 100): the last chunk takes the rest
            if (c < kMaxChunks) ++c;
            b[c] = (int)nrows;
        }
        S.count[par] = c > 0 ? c : 1;
        if (c == 0) b[1] = (int)nrows;
    }
    if (!stagger) {
        S.count[1] = S.count[0];
        for (int k = 0; k <= kMaxChunks; ++k) S.bounds[1][k] = S.bounds[0][k];
    }
}

// Upper-triangle mode: the work of a column strip grows with its index (strip s holds rows <= 128 s + 127 only), so the
// rectangular wave-quantisation estimate of pick_rows_per_cta does not apply.  The grid is dispatched chunk-major /
// strip-minor onto 296 CTA slots; this replays that greedy assignment with cost(item) = rows + 160 (per-CTA prologue and
// combine, in row units) and returns the makespan.  Host side, a few ms at 50k loci: cached per shape by make_layout.
double simulate_upper(int64_t r0, int nstrips, const Schedule& S, int stagger) {
    std::vector<double> heap(kCtaSlots, 0.0);  // min-heap of slot finish times
    auto cmp = [](double a, double b) { return a > b; };
    const int nchunks = S.count[0] > S.count[1] ? S.count[0] : S.count[1];
    double makespan = 0.0;
    for (int chunk = 0; chunk < nchunks; ++chunk) {
        for (int strip = 0; strip < nstrips; ++strip) {
            const int par = (stagger && ((strip / 148) & 1)) ? 1 : 0;
            if (chunk >= S.count[par]) continue;
            const int64_t start = S.bounds[par][chunk];
            int64_t end = S.bounds[par][chunk + 1];
            const int64_t lim = (int64_t)(strip + 1) * kCols - r0;
            if (end > lim) end = lim;
            if (end <= start) continue;  // exits at once
            std::pop_heap(heap.begin(), heap.end(), cmp);
            const double t = heap.back() + (double)(end - start) + 160.0;  // measured: ~5 us of CTA prologue + combine per item = 160 rows
            heap.back() = t;
            std::push_heap(heap.begin(), heap.end(), cmp);
            if (t > makespan) makespan = t;
        }
    }
    return makespan;
}

Layout make_layout_uncached(int64_t n, int64_t r0, int64_t r1, int variant, bool sym) {
    Layout L;
    L.nstrips = (int)((n + kCols - 1) / kCols);
    const int64_t nrows = r1 - r0;
    L.persistent = variant == 3 ? 1 : 0;
    L.seg_len = L.seg_total = 0;
    L.seg_sa = L.seg_sb = L.seg_f = L.seg_warps = 0;
    if (variant == 4 && nrows > 0) {
        // static warp partition: closed form of rows per strip (see strip_offset) and the run length per warp
        L.seg_sa = sym ? (int)(r0 / kCols) : 0;
        L.seg_f = sym ? (int)(kCols - (r0 % kCols)) : 0;
        L.seg_sb = sym ? L.seg_sa + (int)((std::max<int64_t>(nrows - L.seg_f, 0) + kCols - 1) / kCols) : 0;
        int64_t total = 0;
        for (int st = 0; st < L.nstrips; ++st) {
            int64_t v = sym ? std::min<int64_t>(std::max<int64_t>((int64_t)(st + 1) * kCols - r0, 0), nrows) : nrows;
            total += v;
        }
        L.seg_total = total;
        const int64_t slots = (int64_t)kCtaSlots * kWarps;
        int64_t len = (total + slots - 1) / slots;
        len = std::max<int64_t>((len + kU - 1) / kU * kU, kU);
        L.seg_len = len;
        L.seg_warps = (int)((total + len - 1) / len);
        L.rb = kTileRows; L.stagger = 0; L.persistent = 0; L.nitems = 0;
        memset(&L.sch, 0, sizeof(L.sch));
        memset(L.item_base, 0, sizeof(L.item_base));
        L.sch.count[0] = L.sch.count[1] = 1;
        L.sch.bounds[0][1] = L.sch.bounds[1][1] = (int)nrows;
        L.nchunks = (int)((nrows + len - 1) / len) + 1;  // segments a strip can be cut into
        L.nslots = (size_t)L.nstrips * L.nchunks;
        L.off_mpart = 0;
        L.off_gpart = L.off_mpart + align_up(sizeof(double) * kNM * L.nslots, 256);
        L.off_rpart = align_up(L.off_gpart + sizeof(float) * (size_t)kCols * 3 * L.nslots, 256);
        L.rpitch = sym ? (int64_t)align_up((size_t)nrows * 3, 32) : 0;
        L.off_counter = align_up(L.off_rpart + sizeof(float) * (size_t)L.rpitch * L.nstrips, 256);
        L.total = L.off_counter + 256;
        add_rowside_layout(L, r0, r1, sym);
        return L;
    }
    if (variant == 3 || variant == 4) variant = 0;  // same tiles / partial layout as the TMA kernel
    const int unit = variant == 0 ? kTileRows : 8;
    int depth = 0, tail_min = g_tail_min_rows;
    memset(&L.sch, 0, sizeof(L.sch));
    memset(L.item_base, 0, sizeof(L.item_base));
    L.nitems = 0;
    if (L.persistent && nrows > 0) {
        // items are cheap (the next item's tiles are in flight during the combine) and balanced dynamically: aim at ~12 items per
        // CTA slot, 128 .. 2048 rows each; no stagger, no tail
        double work = 0.0;  // strip-rows of this block
        for (int s = 0; s < L.nstrips; ++s) {
            const int64_t lim = sym ? std::min<int64_t>(nrows, (int64_t)(s + 1) * kCols - r0) : nrows;
            if (lim > 0) work += (double)lim;
        }
        int64_t rb = (int64_t)(work / kCtaSlots / 12.0);
        rb = (rb + kTileRows - 1) / kTileRows * kTileRows;
        if (g_rows_per_cta > 0) rb = (g_rows_per_cta + kTileRows - 1) / kTileRows * kTileRows;
        rb = std::max<int64_t>(2 * kTileRows, std::min<int64_t>(rb, 2048));
        while ((nrows + rb - 1) / rb > kMaxChunks - 20) rb += kTileRows;
        L.rb = (int)rb;
        L.stagger = 0;
    } else if (sym && g_rows_per_cta == 0 && g_tail_depth < 0 && nrows > 0) {
        // equal chunks, no explicit tail (the triangle tapers by itself): pick the chunk length by simulation
        static const int cand0[] = {256, 384, 512, 640, 768, 1024, 1280, 1536, 2048, 3072, 4096};
        static const int cand1[] = {256, 384, 512, 768, 1024};  // per-lane kernels: a chunk is at most one x_i staging piece (kStageRows)
        const int* cand = variant == 0 ? cand0 : cand1;
        const int ncand = variant == 0 ? 11 : 5;
        double best = 1e300;
        int best_rb = cand[ncand - 1], best_stagger = 0, best_depth = 0;
        for (int k = 0; k < ncand; ++k) {
            const int rb = cand[k];
            if ((nrows + rb - 1) / rb > kMaxChunks - 20) continue;
            const int uniform_chunks = (int)((nrows + rb - 1) / rb);
            const int stagger = (variant == 0 && g_stagger && L.nstrips > 148 && uniform_chunks >= 2) ? 1 : 0;
            for (int d = 0; d <= (variant == 0 ? 3 : 0); ++d) {  // optionally a halving tail of d chunks (down to 128 rows) behind the bulk
                Schedule S;
                memset(&S, 0, sizeof(S));
                build_schedule(nrows, rb, d, 128, stagger != 0, unit, S);
                const double m = simulate_upper(r0, L.nstrips, S, stagger);
                if (m < best * 0.995) {
                    best = m;
                    best_rb = rb;
                    best_stagger = stagger;
                    best_depth = d;
                }
            }
        }
        depth = best_depth;
        tail_min = 128;
        L.rb = best_rb;
        while ((nrows + L.rb - 1) / L.rb > kMaxChunks - 20) L.rb *= 2;
        L.stagger = best_stagger;
    } else {
        L.rb = pick_rows_per_cta(nrows, L.nstrips, variant);
        while ((nrows + L.rb - 1) / L.rb > kMaxChunks - 20) L.rb *= 2;  // boundary table size
        const int uniform_chunks = (int)((nrows + L.rb - 1) / L.rb);
        // stagger (chunk_rows): only where a second CTA slot per SM is filled in the first wave
        L.stagger = (variant == 0 && g_stagger && L.nstrips > 148 && uniform_chunks >= 2) ? 1 : 0;
        // Default tail: maps of up to 148 strips (no stagger, 1-3 items per CTA slot) end with three halving chunks
        // down to 128 rows behind bulk chunks of at most 1024 rows (10k loci: 91.5 -> 85.3 us, measured with
        // scripts/bench_pairloss_variants.py); staggered grids keep equal chunks (a tail measured +-1 % there).
        if (variant == 0) {
            if (g_tail_depth >= 0) {
                depth = g_tail_depth;
            } else if (!L.stagger && nrows >= 2048 && g_rows_per_cta == 0) {
                depth = 3;
                tail_min = 128;
                if (L.rb > 1024) L.rb = 1024;
            }
        }
    }
    build_schedule(nrows > 0 ? nrows : 1, L.rb, depth, tail_min, L.stagger != 0, unit, L.sch);
    L.nchunks = L.sch.count[0] > L.sch.count[1] ? L.sch.count[0] : L.sch.count[1];
    // the per-lane-load and implicit-target kernels stage x_i of the longest chunk in shared memory, kStageRows rows at a time
    int longest = 0;
    for (int par = 0; par < 2; ++par)
        for (int k = 0; k < L.sch.count[par]; ++k) longest = std::max(longest, L.sch.bounds[par][k + 1] - L.sch.bounds[par][k]);
    L.rb = longest;
    L.nslots = (size_t)L.nstrips * L.nchunks;
    L.off_mpart = 0;
    L.off_gpart = L.off_mpart + align_up(sizeof(double) * kNM * L.nslots, 256);
    L.off_rpart = align_up(L.off_gpart + sizeof(float) * (size_t)kCols * 3 * L.nslots, 256);
    L.rpitch = sym ? (int64_t)align_up((size_t)(nrows > 0 ? nrows : 1) * 3, 32) : 0;
    L.off_counter = align_up(L.off_rpart + sizeof(float) * (size_t)L.rpitch * L.nstrips, 256);
    L.total = L.off_counter + 256;
    add_rowside_layout(L, r0, r1, sym);
    if (L.persistent) {
        for (int c = 0; c < L.sch.count[0]; ++c) {
            int first = 0;
            if (sym) first = (int)std::max<int64_t>(0, (r0 + L.sch.bounds[0][c]) / kCols);  // strips left of it lie below the diagonal
            if (first > L.nstrips) first = L.nstrips;
            L.item_base[c + 1] = L.item_base[c] + (L.nstrips - first);
        }
        L.nitems = L.item_base[L.sch.count[0]];
    }
    return L;
}

// make_layout runs on the host for every call of the loss; the upper-triangle schedule search costs milliseconds, so
// layouts are memoised per (shape, variant, mode, tuning).  Thread-safe.
Layout make_layout(int64_t n, int64_t r0, int64_t r1, int variant, bool sym = false) {
    struct Key {
        int64_t n, r0, r1;
        int variant, sym, rows, stagger, depth, tail_min, rs_max, rs_min;
        bool operator<(const Key& o) const {
            return std::tie(n, r0, r1, variant, sym, rows, stagger, depth, tail_min, rs_max, rs_min) <
                   std::tie(o.n, o.r0, o.r1, o.variant, o.sym, o.rows, o.stagger, o.depth, o.tail_min, o.rs_max, o.rs_min);
        }
    };
    static std::mutex mu;
    static std::map<Key, Layout> cache;
    const Key key{n, r0, r1, variant, sym ? 1 : 0, g_rows_per_cta, g_stagger, g_tail_depth, g_tail_min_rows, g_rs_groups_max, g_rs_min_strips};
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    if (cache.size() > 4096) cache.clear();  // the host-buffer path walks many row blocks: bound the memo
    const Layout L = make_layout_uncached(n, r0, r1, variant, sym);
    cache.emplace(key, L);
    return L;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// 2-D map over this rank's target rows: dim0 = n valid columns (pitch only enters the stride, so
// padding columns are never read and columns >= n are zero-filled), dim1 = r1 - r0 rows.
bool make_target_map(CUtensorMap* map, const float* target, int64_t pitch, int64_t n, int64_t nrows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)n, (cuuint64_t)nrows};
    const cuuint64_t gstride[1] = {(cuuint64_t)pitch * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)kCols, (cuuint32_t)kU};
    const cuuint32_t estride[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(target), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <uint32_t MODE>
cudaError_t launch_combine(const Params& P, cudaStream_t stream) {
    // the Pearson pass carries its coefficients in the per-pair weight: no scale
    const float scale = (MODE & kPearson) ? 1.f : ((MODE & 3u) == HICGAT_PAIR_GRAD_MSE) ? P.c_mse : ((MODE & 3u) == HICGAT_PAIR_GRAD_L1) ? P.c_l1 : 1.f;
    const int want_grad = has_grad(MODE) ? 1 : 0;
    if (g_pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(P.nstrips + 1 + (P.rs_groups > 1 ? P.rs_groups * P.rs_count : 0));
        cfg.blockDim = dim3(kCombineThreads);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, pairloss_combine_kernel, P, scale, want_grad, 2);
    }
    pairloss_combine_kernel<<<P.nstrips + 1 + (P.rs_groups > 1 ? P.rs_groups * P.rs_count : 0), kCombineThreads, 0, stream>>>(P, scale, want_grad, 1);
    return cudaGetLastError();
}

template <uint32_t MODE, bool ROWS>
cudaError_t launch_tma(const CUtensorMap& map, const Params& P, dim3 grid, cudaStream_t stream) {
    // opt in to > 48 KB dynamic shared memory: a per-DEVICE function attribute, set once per (instantiation, device)
    static std::atomic<uint64_t> attr_set{0};
    int dev = 0;
    cudaGetDevice(&dev);
    const uint64_t bit = 1ull << (dev & 63);
    if (dev >= 64 || !(attr_set.load(std::memory_order_relaxed) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(pairloss_tma_kernel<MODE, ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTmaSmem);
        if (e != cudaSuccess) return e;
        attr_set.fetch_or(bit, std::memory_order_relaxed);
    }
    // programmatic stream serialization: the CTAs may become resident (barrier init, tensor-map prefetch, schedule lookup)
    // while the previous kernel of the stream drains; griddepcontrol.wait precedes the first global read
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kTmaSmem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, pairloss_tma_kernel<MODE, ROWS>, map, P);
}

template <uint32_t MODE, bool ROWS>
cudaError_t launch_persist(const CUtensorMap& map, const Params& P, cudaStream_t stream) {
    static std::atomic<uint64_t> attr_set{0};
    int dev = 0;
    cudaGetDevice(&dev);
    const uint64_t bit = 1ull << (dev & 63);
    if (dev >= 64 || !(attr_set.load(std::memory_order_relaxed) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(pairloss_tma_persist_kernel<MODE, ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPersistSmem);
        if (e != cudaSuccess) return e;
        attr_set.fetch_or(bit, std::memory_order_relaxed);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)std::min(P.nitems, kCtaSlots));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kPersistSmem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, pairloss_tma_persist_kernel<MODE, ROWS>, map, P);
}

template <uint32_t MODE, bool ROWS>
cudaError_t launch_warp(const CUtensorMap& map, const Params& P, int nwarps, cudaStream_t stream) {
    static std::atomic<uint64_t> attr_set{0};
    int dev = 0;
    cudaGetDevice(&dev);
    const uint64_t bit = 1ull << (dev & 63);
    if (dev >= 64 || !(attr_set.load(std::memory_order_relaxed) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(pairloss_tma_warp_kernel<MODE, ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTmaSmem);
        if (e != cudaSuccess) return e;
        attr_set.fetch_or(bit, std::memory_order_relaxed);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((nwarps + kWarps - 1) / kWarps));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kTmaSmem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, pairloss_tma_warp_kernel<MODE, ROWS>, map, P);
}

template <uint32_t MODE>
cudaError_t launch_mode(int variant, const CUtensorMap& map, const Params& P, dim3 grid, cudaStream_t stream) {
    cudaError_t e;
    if (variant == 4) {
        const int nwarps = (int)((P.seg_total + P.seg_len - 1) / P.seg_len);
        e = P.upper ? launch_warp<MODE, true>(map, P, nwarps, stream) : launch_warp<MODE, false>(map, P, nwarps, stream);
    } else if (variant == 3) {
        e = P.upper ? launch_persist<MODE, true>(map, P, stream) : launch_persist<MODE, false>(map, P, stream);
    } else if (variant == 0) {
        e = P.upper ? launch_tma<MODE, true>(map, P, grid, stream) : launch_tma<MODE, false>(map, P, grid, stream);
    } else {
        const size_t smem = lane_smem_bytes(P.rb);
        if (P.upper) pairloss_lane_kernel<MODE, true, false><<<grid, kThreads, smem, stream>>>(P);
        else pairloss_lane_kernel<MODE, false, false><<<grid, kThreads, smem, stream>>>(P);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return e;
    return launch_combine<MODE>(P, stream);
}

}  // namespace
}  // namespace hicgat

using namespace hicgat;

#ifdef HICGAT_TRACE
extern "C" __attribute__((visibility("default"))) int hicgat_debug_set_trace(unsigned long long* buf) {
    return cudaMemcpyToSymbol(g_trace, &buf, sizeof(buf)) == cudaSuccess ? 0 : -1;
}
#endif

extern "C" int hicgat_pairloss_set_combine(int rowside_groups_max, int rowside_min_strips) {
    if (rowside_groups_max < 1 || rowside_groups_max > 16 || rowside_min_strips < 1) {
        set_error("hicgat_pairloss_set_combine: rowside_groups_max must be in [1,16], rowside_min_strips >= 1");
        return HICGAT_ERR_INVALID;
    }
    g_rs_groups_max = rowside_groups_max;
    g_rs_min_strips = rowside_min_strips;
    return HICGAT_OK;
}

extern "C" int hicgat_pairloss_set_tuning(int rows_per_cta, int variant) {
    if (rows_per_cta != 0 && (rows_per_cta < 8 || rows_per_cta > 4096 || (rows_per_cta % 8) != 0)) {
        set_error("hicgat_pairloss_set_tuning: rows_per_cta must be 0 or a multiple of 8 in [8,4096]");
        return HICGAT_ERR_INVALID;
    }
    if (variant < 0 || variant > 4) {
        set_error("hicgat_pairloss_set_tuning: variant must be 0 (TMA ring), 1 (per-lane loads), 2 (TMA ring, unstaggered chunks), 3 (persistent TMA ring) or 4 (static warp partition)");
        return HICGAT_ERR_INVALID;
    }
    g_rows_per_cta = rows_per_cta;
    g_variant = variant == 2 ? 0 : variant;
    g_stagger = variant == 2 ? 0 : 1;
    return HICGAT_OK;
}

extern "C" int hicgat_pairloss_set_schedule(int tail_depth, int tail_min_rows) {
    if (tail_depth < -1 || tail_depth > 8 || tail_min_rows < 64 || tail_min_rows > 4096) {
        set_error("hicgat_pairloss_set_schedule: tail_depth must be -1 (default) or 0..8, tail_min_rows 64..4096");
        return HICGAT_ERR_INVALID;
    }
    g_tail_depth = tail_depth;
    g_tail_min_rows = tail_min_rows;
    return HICGAT_OK;
}

extern "C" int hicgat_pairloss_describe_schedule_mode(int64_t n, int64_t r0, int64_t r1, uint32_t mode, int32_t* out, int32_t capacity);
extern "C" int hicgat_pairloss_describe_schedule(int64_t n, int64_t r0, int64_t r1, int32_t* out, int32_t capacity) {
    return hicgat_pairloss_describe_schedule_mode(n, r0, r1, 0u, out, capacity);
}

extern "C" int hicgat_pairloss_describe_schedule_mode(int64_t n, int64_t r0, int64_t r1, uint32_t mode, int32_t* out, int32_t capacity) {
    if (n <= 0 || r0 < 0 || r1 < r0 || r1 > n || !out || capacity < 4) {
        set_error("hicgat_pairloss_describe_schedule: bad arguments");
        return HICGAT_ERR_INVALID;
    }
    const Layout L = make_layout(n, r0, r1, g_variant, (mode & HICGAT_PAIR_SYMMETRIC) != 0);
    const int need = 4 + (L.sch.count[0] + 1) + (L.sch.count[1] + 1);
    if (capacity < need) {
        set_error("hicgat_pairloss_describe_schedule: capacity %d < %d", (int)capacity, need);
        return HICGAT_ERR_WORKSPACE;
    }
    int k = 0;
    out[k++] = L.nstrips;
    out[k++] = L.stagger;
    out[k++] = L.sch.count[0];
    out[k++] = L.sch.count[1];
    for (int par = 0; par < 2; ++par)
        for (int c = 0; c <= L.sch.count[par]; ++c) out[k++] = L.sch.bounds[par][c];
    return k;
}

extern "C" double hicgat_pairloss_estimate_cost(int64_t n, int64_t r0, int64_t r1, uint32_t mode) {
    if (n <= 0 || r0 < 0 || r1 < r0 || r1 > n) return -1.0;
    if (r1 == r0) return 0.0;
    const bool sym = (mode & HICGAT_PAIR_SYMMETRIC) != 0;
    const Layout L = make_layout(n, r0, r1, g_variant, sym);
    if (sym) return simulate_upper(r0, L.nstrips, L.sch, L.stagger);
    // full-matrix mode: every strip has every chunk
    Schedule S = L.sch;
    return simulate_upper(-(int64_t)n * 2, L.nstrips, S, L.stagger);  // a diagonal far to the left clips nothing
}

extern "C" size_t hicgat_pairloss_workspace_bytes(int64_t n, int64_t r0, int64_t r1) {
    if (n <= 0 || r0 < 0 || r1 < r0 || r1 > n) return 0;
    // for the CURRENT tuning (re-query after set_tuning); covers either variant
    const size_t a = make_layout(n, r0, r1, 0).total, b = make_layout(n, r0, r1, 1).total, c = make_layout(n, r0, r1, 3).total, d = make_layout(n, r0, r1, 4).total;
    return std::max(std::max(a, d), std::max(b, c));
}

extern "C" size_t hicgat_pairloss_workspace_bytes_mode(int64_t n, int64_t r0, int64_t r1, uint32_t mode) {
    if (n <= 0 || r0 < 0 || r1 < r0 || r1 > n) return 0;
    const bool sym = (mode & HICGAT_PAIR_SYMMETRIC) != 0;
    const size_t a = make_layout(n, r0, r1, 0, sym).total, b = make_layout(n, r0, r1, 1, sym).total, c = make_layout(n, r0, r1, 3, sym).total,
                 d = make_layout(n, r0, r1, 4, sym).total;
    return std::max(std::max(a, d), std::max(b, c));
}

static int pairloss_impl(const float* coords, const float* target, int64_t pitch, int64_t n,
                         int64_t r0, int64_t r1, uint32_t mode, float c_mse, float c_l1,
                         double* moments, float* grad, double* grad64, void* workspace, size_t workspace_bytes,
                         hicgat_stream_t stream_, const double* pmom = nullptr, int dyn_alpha = 0) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(n > 0 && n < (1ll << 30) && r0 >= 0 && r1 >= r0 && r1 <= n, "hicgat_pairloss_fwd_bwd: bad n/r0/r1 (%lld,%lld,%lld)", (long long)n, (long long)r0, (long long)r1);
    // an empty row block (r0 == r1, a trailing rank of a sharded run) has no target rows to point at
    HICGAT_REQUIRE(coords && (target || r0 == r1) && (moments || pmom) && workspace, "hicgat_pairloss_fwd_bwd: null pointer");
    HICGAT_REQUIRE(pitch >= n && (pitch % 4) == 0, "hicgat_pairloss_fwd_bwd: pitch %lld must be >= n and a multiple of 4", (long long)pitch);
    HICGAT_REQUIRE(aligned16(target), "hicgat_pairloss_fwd_bwd: target must be 16-byte aligned");  // NULL passes
    HICGAT_REQUIRE((mode & ~63u) == 0, "hicgat_pairloss_fwd_bwd: unknown mode bits 0x%x", mode);
    const bool ws_clean = (mode & HICGAT_PAIR_WS_CLEAN) != 0;  // the persistent variant keeps ONE item counter in the workspace (left at zero by every call)
    mode &= ~HICGAT_PAIR_WS_CLEAN;
    const bool sym = (mode & HICGAT_PAIR_SYMMETRIC) != 0;
    mode &= ~HICGAT_PAIR_SYMMETRIC;
    if (mode & HICGAT_PAIR_MOMENTS) mode &= ~HICGAT_PAIR_MOMENTS_D;          // full moments include the light set
    if ((mode & HICGAT_PAIR_MOMENTS_D) && (mode & HICGAT_PAIR_GRAD_L1)) {     // the L1 value needs sum |d-t|: full set
        mode = (mode & ~HICGAT_PAIR_MOMENTS_D) | HICGAT_PAIR_MOMENTS;
    }
    if (pmom) mode |= kPearson;  // second pass of the differentiable Pearson modes (hicgat_pairloss_pearson_grad)
    HICGAT_REQUIRE(!has_grad(mode) || grad || grad64, "hicgat_pairloss_fwd_bwd: grad is NULL but a gradient mode is set");
    int variant = g_variant;
    CUtensorMap map;
    // a target no tensor map can be encoded for goes through the per-lane-load kernel (same sums, either triangle mode)
    if (variant != 1 && r1 > r0 && !make_target_map(&map, target, pitch, n, r1 - r0)) variant = 1;
    const Layout L = make_layout(n, r0, r1, variant, sym);
    if (workspace_bytes < L.total) {
        set_error("hicgat_pairloss_fwd_bwd: workspace %zu < required %zu", workspace_bytes, L.total);
        return HICGAT_ERR_WORKSPACE;
    }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    if (r1 == r0) {  // empty row block: contributes nothing
        if (moments) HICGAT_CUDA(cudaMemsetAsync(moments, 0, sizeof(double) * kNM, stream));
        if (grad) HICGAT_CUDA(cudaMemsetAsync(grad, 0, sizeof(float) * 3 * (size_t)n, stream));
        if (grad64) HICGAT_CUDA(cudaMemsetAsync(grad64, 0, sizeof(double) * 3 * (size_t)n, stream));
        return HICGAT_OK;
    }
    // the combine kernel writes no gradient in a mode without one: the packed buffer is all-reduced whole, so it gets zeros
    if (grad64 && !has_grad(mode)) HICGAT_CUDA(cudaMemsetAsync(grad64, 0, sizeof(double) * 3 * (size_t)n, stream));
    Params P;
    P.coords = coords; P.target = target; P.pitch = pitch;
    P.n = (int)n; P.r0 = (int)r0; P.r1 = (int)r1; P.rb = L.rb; P.nstrips = L.nstrips; P.nchunks = L.nchunks; P.stagger = L.stagger; P.sch = L.sch;
    P.fill = 0.f;
    P.c_mse = c_mse; P.c_l1 = c_l1; P.moments = moments; P.grad = grad; P.grad64 = grad64;
    P.pmom = pmom; P.dyn_alpha = dyn_alpha;
    P.mpart = reinterpret_cast<double*>(ws + L.off_mpart);
    P.gpart = reinterpret_cast<float*>(ws + L.off_gpart);
    P.upper = sym ? 1 : 0; P.rpitch = L.rpitch; P.rpart = reinterpret_cast<float*>(ws + L.off_rpart);
    P.work_counter = nullptr; P.nitems = 0;
    P.seg_len = L.seg_len; P.seg_total = L.seg_total; P.seg_sa = L.seg_sa; P.seg_sb = L.seg_sb; P.seg_f = L.seg_f;
    if (L.persistent) {
        P.work_counter = reinterpret_cast<unsigned*>(ws + L.off_counter);
        P.nitems = L.nitems;
        memcpy(P.item_base, L.item_base, sizeof(P.item_base));
        if (!ws_clean) HICGAT_CUDA(cudaMemsetAsync(P.work_counter, 0, sizeof(unsigned), stream));
    }
    P.rs_first = L.rs_first; P.rs_count = L.rs_count; P.rs_groups = L.rs_groups;
    P.rs_ticket = reinterpret_cast<unsigned*>(ws + L.off_rs_ticket);
    P.rs_scratch = reinterpret_cast<double*>(ws + L.off_rs_scratch);
    // the tickets return to zero at the end of every call; a workspace of unknown content is cleared first
    if (L.rs_groups > 1 && !ws_clean) HICGAT_CUDA(cudaMemsetAsync(P.rs_ticket, 0, sizeof(unsigned) * (size_t)L.rs_count, stream));
    dim3 grid(L.nstrips, L.nchunks);
    cudaError_t err = cudaSuccess;
    switch (mode) {
#define HICGAT_CASE(M) case M: err = launch_mode<M>(variant, map, P, grid, stream); break;
        HICGAT_CASE(0u) HICGAT_CASE(1u) HICGAT_CASE(2u) HICGAT_CASE(3u) HICGAT_CASE(4u)
        HICGAT_CASE(5u) HICGAT_CASE(6u) HICGAT_CASE(7u) HICGAT_CASE(8u) HICGAT_CASE(9u)
        HICGAT_CASE(64u) HICGAT_CASE(65u)
#undef HICGAT_CASE
        default:
            set_error("hicgat_pairloss_fwd_bwd: unsupported mode 0x%x", mode);
            return HICGAT_ERR_INVALID;
    }
    if (err != cudaSuccess) {
        set_error("pairloss kernel launch failed: %s", cudaGetErrorString(err));
        return HICGAT_ERR_CUDA;
    }
    count_launch(2);
    return HICGAT_OK;
}

extern "C" int hicgat_pairloss_fwd_bwd(const float* coords, const float* target, int64_t pitch, int64_t n,
                                       int64_t r0, int64_t r1, uint32_t mode, float c_mse, float c_l1,
                                       double* moments, float* grad, void* workspace, size_t workspace_bytes,
                                       hicgat_stream_t stream) {
    return pairloss_impl(coords, target, pitch, n, r0, r1, mode, c_mse, c_l1, moments, grad, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int hicgat_pairloss_fwd_bwd_packed(const float* coords, const float* target, int64_t pitch, int64_t n,
                                              int64_t r0, int64_t r1, uint32_t mode, float c_mse, float c_l1,
                                              double* packed, void* workspace, size_t workspace_bytes,
                                              hicgat_stream_t stream) {
    if (!packed) {
        set_error("hicgat_pairloss_fwd_bwd_packed: null pointer");
        return HICGAT_ERR_INVALID;
    }
    return pairloss_impl(coords, target, pitch, n, r0, r1, mode, c_mse, c_l1, packed, nullptr, packed + HICGAT_PAIR_NMOM, workspace, workspace_bytes, stream);
}

// ------------------------------------------------------------------ implicit (sparse) target entry points
namespace {
struct SparseLayout {
    Layout dense;
    size_t off_counter, off_part, total;
    int fix_ctas;
};
SparseLayout sparse_layout(int64_t n, int64_t r0, int64_t r1, bool sym = false) {
    SparseLayout L;
    L.dense = make_layout(n, r0, r1, 1, sym);  // the per-lane kernel's chunks and partial slots
    L.fix_ctas = (int)((r1 - r0 + 7) / 8);
    if (L.fix_ctas < 1) L.fix_ctas = 1;
    L.off_counter = align_up(L.dense.total, 256);
    L.off_part = L.off_counter + 256;
    L.total = L.off_part + sizeof(double) * kNM * (size_t)L.fix_ctas;
    return L;
}

template <uint32_t MODE>
cudaError_t launch_sparse(const Params& P, dim3 grid, const int32_t* rowptr, const int32_t* col, const float* tval, int fix_ctas, double* part,
                          unsigned* counter, cudaStream_t stream) {
    const size_t smem = lane_smem_bytes(P.rb);
    if (P.upper) pairloss_lane_kernel<MODE, true, true><<<grid, kThreads, smem, stream>>>(P);
    else pairloss_lane_kernel<MODE, false, true><<<grid, kThreads, smem, stream>>>(P);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    e = launch_combine<MODE>(P, stream);
    if (e != cudaSuccess) return e;
    pairloss_csr_fix_kernel<MODE><<<fix_ctas, 256, 0, stream>>>(P.coords, rowptr, col, tval, P.fill, P.n, P.r0, P.r1, P.c_mse, P.c_l1, P.moments, P.grad,
                                                                 P.grad64, part, counter, P.pmom, P.dyn_alpha);
    return cudaGetLastError();
}
}  // namespace

extern "C" size_t hicgat_pairloss_sparse_workspace_bytes(int64_t n, int64_t r0, int64_t r1) {
    if (n <= 0 || r0 < 0 || r1 < r0 || r1 > n) return 0;
    return std::max(sparse_layout(n, r0, r1, true).total, sparse_layout(n, r0, r1, false).total);  // with or without HICGAT_PAIR_SYMMETRIC
}

static int pairloss_sparse_impl(const float* coords, const int32_t* rowptr, const int32_t* col, const float* tval, float fill, int64_t n,
                                int64_t r0, int64_t r1, uint32_t mode, float c_mse, float c_l1, double* moments, float* grad, double* grad64,
                                void* workspace, size_t workspace_bytes, hicgat_stream_t stream_, const double* pmom = nullptr,
                                int dyn_alpha = 0) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(n > 0 && n < (1ll << 30) && r0 >= 0 && r1 >= r0 && r1 <= n, "hicgat_pairloss_sparse_fwd_bwd: bad n/r0/r1 (%lld,%lld,%lld)", (long long)n, (long long)r0, (long long)r1);
    HICGAT_REQUIRE(coords && rowptr && (col || r0 == r1) && (tval || r0 == r1) && (moments || pmom) && workspace, "hicgat_pairloss_sparse_fwd_bwd: null pointer");
    HICGAT_REQUIRE((mode & ~63u) == 0, "hicgat_pairloss_sparse_fwd_bwd: unknown mode bits 0x%x", mode);
    const bool ws_clean = (mode & HICGAT_PAIR_WS_CLEAN) != 0;
    const bool sym = (mode & HICGAT_PAIR_SYMMETRIC) != 0;
    mode &= ~(HICGAT_PAIR_WS_CLEAN | HICGAT_PAIR_SYMMETRIC);
    if (mode & HICGAT_PAIR_MOMENTS) mode &= ~HICGAT_PAIR_MOMENTS_D;
    if ((mode & HICGAT_PAIR_MOMENTS_D) && (mode & HICGAT_PAIR_GRAD_L1)) mode = (mode & ~HICGAT_PAIR_MOMENTS_D) | HICGAT_PAIR_MOMENTS;
    if (pmom) mode |= kPearson;
    HICGAT_REQUIRE(!has_grad(mode) || grad || grad64, "hicgat_pairloss_sparse_fwd_bwd: grad is NULL but a gradient mode is set");
    const SparseLayout L = sparse_layout(n, r0, r1, sym);
    if (workspace_bytes < L.total) {
        set_error("hicgat_pairloss_sparse_fwd_bwd: workspace %zu < required %zu", workspace_bytes, L.total);
        return HICGAT_ERR_WORKSPACE;
    }
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    if (!ws_clean) {
        HICGAT_CUDA(cudaMemsetAsync(ws + L.off_counter, 0, sizeof(unsigned), stream));  // ticket of pairloss_csr_fix_kernel
    }
    if (r1 == r0) {
        if (moments) HICGAT_CUDA(cudaMemsetAsync(moments, 0, sizeof(double) * kNM, stream));
        if (grad) HICGAT_CUDA(cudaMemsetAsync(grad, 0, sizeof(float) * 3 * (size_t)n, stream));
        if (grad64) HICGAT_CUDA(cudaMemsetAsync(grad64, 0, sizeof(double) * 3 * (size_t)n, stream));
        return HICGAT_OK;
    }
    Params P;
    P.coords = coords; P.target = nullptr; P.pitch = 0;
    P.n = (int)n; P.r0 = (int)r0; P.r1 = (int)r1; P.rb = L.dense.rb; P.nstrips = L.dense.nstrips; P.nchunks = L.dense.nchunks; P.stagger = L.dense.stagger; P.sch = L.dense.sch;
    P.fill = fill;
    P.c_mse = c_mse; P.c_l1 = c_l1; P.moments = moments; P.grad = grad; P.grad64 = grad64;
    P.pmom = pmom; P.dyn_alpha = dyn_alpha;
    P.mpart = reinterpret_cast<double*>(ws + L.dense.off_mpart);
    P.gpart = reinterpret_cast<float*>(ws + L.dense.off_gpart);
    P.upper = sym ? 1 : 0; P.rpitch = L.dense.rpitch; P.rpart = reinterpret_cast<float*>(ws + L.dense.off_rpart);
    P.work_counter = nullptr; P.nitems = 0;
    P.seg_len = 0; P.seg_total = 0; P.seg_sa = P.seg_sb = P.seg_f = 0;
    P.rs_first = L.dense.rs_first; P.rs_count = L.dense.rs_count; P.rs_groups = L.dense.rs_groups;
    P.rs_ticket = reinterpret_cast<unsigned*>(ws + L.dense.off_rs_ticket);
    P.rs_scratch = reinterpret_cast<double*>(ws + L.dense.off_rs_scratch);
    if (L.dense.rs_groups > 1 && !ws_clean) HICGAT_CUDA(cudaMemsetAsync(P.rs_ticket, 0, sizeof(unsigned) * (size_t)L.dense.rs_count, stream));
    dim3 grid(L.dense.nstrips, L.dense.nchunks);
    double* part = reinterpret_cast<double*>(ws + L.off_part);
    unsigned* counter = reinterpret_cast<unsigned*>(ws + L.off_counter);
    cudaError_t err = cudaSuccess;
    switch (mode) {
#define HICGAT_CASE(M) case M: err = launch_sparse<M>(P, grid, rowptr, col, tval, L.fix_ctas, part, counter, stream); break;
        HICGAT_CASE(0u) HICGAT_CASE(1u) HICGAT_CASE(2u) HICGAT_CASE(3u) HICGAT_CASE(4u)
        HICGAT_CASE(5u) HICGAT_CASE(6u) HICGAT_CASE(7u) HICGAT_CASE(8u) HICGAT_CASE(9u)
        HICGAT_CASE(64u) HICGAT_CASE(65u)
#undef HICGAT_CASE
        default:
            set_error("hicgat_pairloss_sparse_fwd_bwd: unsupported mode 0x%x", mode);
            return HICGAT_ERR_INVALID;
    }
    if (err != cudaSuccess) {
        set_error("sparse pairloss kernel launch failed: %s", cudaGetErrorString(err));
        return HICGAT_ERR_CUDA;
    }
    count_launch(3);
    return HICGAT_OK;
}

extern "C" int hicgat_pairloss_sparse_fwd_bwd(const float* coords, const int32_t* rowptr, const int32_t* col, const float* tval, float fill,
                                              int64_t n, int64_t r0, int64_t r1, uint32_t mode, float c_mse, float c_l1, double* moments,
                                              float* grad, void* workspace, size_t workspace_bytes, hicgat_stream_t stream) {
    return pairloss_sparse_impl(coords, rowptr, col, tval, fill, n, r0, r1, mode, c_mse, c_l1, moments, grad, nullptr, workspace, workspace_bytes, stream);
}

// ------------------------------------------------------------------ differentiable Pearson: second pass
namespace {
constexpr uint32_t kPearsonModeBits = HICGAT_PAIR_SYMMETRIC | HICGAT_PAIR_WS_CLEAN | HICGAT_PAIR_GRAD_MSE;
int check_pearson_args(const char* what, uint32_t mode, const double* moments, const float* grad) {
    if (!moments || !grad) {
        set_error("%s: null moments / grad", what);
        return HICGAT_ERR_INVALID;
    }
    if ((mode & ~kPearsonModeBits) != 0) {
        set_error("%s: mode 0x%x: only HICGAT_PAIR_SYMMETRIC | HICGAT_PAIR_WS_CLEAN | HICGAT_PAIR_GRAD_MSE are accepted", what, mode);
        return HICGAT_ERR_INVALID;
    }
    return HICGAT_OK;
}
}  // namespace

extern "C" int hicgat_pairloss_pearson_grad(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1,
                                            uint32_t mode, const double* moments, float c_mse, int dyn_alpha, float* grad, void* workspace,
                                            size_t workspace_bytes, hicgat_stream_t stream) {
    const int rc = check_pearson_args("hicgat_pairloss_pearson_grad", mode, moments, grad);
    if (rc != HICGAT_OK) return rc;
    return pairloss_impl(coords, target, pitch, n, r0, r1, mode, c_mse, 0.f, nullptr, grad, nullptr, workspace, workspace_bytes, stream, moments,
                         dyn_alpha ? 1 : 0);
}

extern "C" int hicgat_pairloss_sparse_pearson_grad(const float* coords, const int32_t* rowptr, const int32_t* col, const float* tval, float fill,
                                                   int64_t n, int64_t r0, int64_t r1, uint32_t mode, const double* moments, float c_mse,
                                                   int dyn_alpha, float* grad, void* workspace, size_t workspace_bytes, hicgat_stream_t stream) {
    const int rc = check_pearson_args("hicgat_pairloss_sparse_pearson_grad", mode, moments, grad);
    if (rc != HICGAT_OK) return rc;
    return pairloss_sparse_impl(coords, rowptr, col, tval, fill, n, r0, r1, mode, c_mse, 0.f, nullptr, grad, nullptr, workspace, workspace_bytes,
                                stream, moments, dyn_alpha ? 1 : 0);
}

extern "C" int hicgat_pairdist_fwd(const float* coords, int64_t n, float* dist, int64_t pitch, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(coords && dist && n > 0 && pitch >= n && n < (1ll << 30), "hicgat_pairdist_fwd: bad arguments");
    dim3 grid((unsigned)((n + 255) / 256), (unsigned)((n + 15) / 16));
    pairdist_fwd_kernel<<<grid, 256, 0, stream>>>(coords, (int)n, dist, pitch);
    HICGAT_CHECK_LAUNCH("pairdist_fwd_kernel");
    return HICGAT_OK;
}

extern "C" int hicgat_pairdist_bwd(const float* coords, int64_t n, const float* grad_dist, int64_t pitch,
                                   float* grad_coords, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(coords && grad_dist && grad_coords && n > 0 && pitch >= n && n < (1ll << 30), "hicgat_pairdist_bwd: bad arguments");
    pairdist_bwd_kernel<<<(unsigned)((n + 7) / 8), 256, 0, stream>>>(coords, (int)n, grad_dist, pitch, grad_coords);
    HICGAT_CHECK_LAUNCH("pairdist_bwd_kernel");
    return HICGAT_OK;
}
