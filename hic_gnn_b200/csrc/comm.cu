// One-shot all-reduce of the row-sharded loss partials over NVLink peer memory.
//
// The reference has no multi-device code; this is the exchange step of the row-sharded
// pairwise loss (SURVEY.md section 8e).  Every rank's fused loss kernel leaves its partial
// [8 x f64 moments | 3n x f32 gradient contribution] in a SYMMETRIC buffer (the same allocation
// mapped into every rank's address space over NVLink / NVSwitch).  One kernel per rank then
//   1. signals "my partial for epoch e is complete" into every peer's signal pad
//      (release at system scope) and waits until all peers have signalled epoch e;
//   2. reads all `world` partials straight from peer memory (ld.relaxed.sys, 128-bit) and adds
//      them in rank order 0..world-1 (gradient: f32 partials accumulated in f64, rounded once),
//      so every rank computes bit-identical sums;
//   3. writes moments (f64, + an optional constant vector) and the gradient as f32 [n,3].
// There is no trailing barrier: the caller alternates between two packed buffers (epoch parity),
// and a rank can only reach epoch e+1's barrier after finishing epoch e's reads, so a buffer is
// never rewritten (epoch e+2's loss kernel) while a peer still reads it.
// Signal slots hold monotonically increasing epochs, so they are never reset.
#include "common.cuh"

namespace hicgat {
namespace {

constexpr int kMaxWorld = 16;

struct PeerTable {
    const unsigned char* buf[kMaxWorld];  // peer r's partial for this epoch parity: [8 x f64 moments | 3n x f32 gradient]
    uint32_t* pad[kMaxWorld];             // peer r's signal pad (uint32 slots)
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_relaxed_sys_f32x4(const void* p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_relaxed_sys_f32(const void* p) {
    float v;
    asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const void* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(256) allreduce_partials_kernel(const PeerTable T, int rank, int world, int slot_base, uint32_t epoch,
                                                                 int64_t nfloat, const double* __restrict__ moment_const,
                                                                 double* __restrict__ out_moments, float* __restrict__ out_grad) {
    // ---- 1. cross-GPU barrier on this epoch (block 0 signals; every block polls its own pad)
    if (blockIdx.x == 0 && threadIdx.x < world) {
        __threadfence_system();  // the loss kernel's writes (previous launch on this stream) -> visible to peers
        st_release_sys(T.pad[threadIdx.x] + slot_base + rank, epoch);
    }
    if (threadIdx.x < world) {
        const uint32_t* mine = T.pad[rank] + slot_base + threadIdx.x;
        // epochs only grow; the signed distance handles the 2^32 wrap
        while ((int32_t)(ld_acquire_sys(mine) - epoch) < 0) { __nanosleep(20); }
    }
    __syncthreads();

    // ---- 2. moments: f64, rank order
    if (blockIdx.x == 0 && threadIdx.x < HICGAT_PAIR_NMOM) {
        double s = 0.0;
        for (int r = 0; r < world; ++r) s += ld_relaxed_sys_f64(T.buf[r] + 8 * threadIdx.x);
        out_moments[threadIdx.x] = s + (moment_const ? moment_const[threadIdx.x] : 0.0);
    }
    // ---- 3. gradient: f32 partials, accumulated in f64 in rank order, rounded once
    const int64_t quads = nfloat >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < quads; i += (int64_t)gridDim.x * blockDim.x) {
        double sx = 0.0, sy = 0.0, sz = 0.0, sw = 0.0;
        for (int r = 0; r < world; ++r) {
            const float4 v = ld_relaxed_sys_f32x4(T.buf[r] + 64 + 16 * i);
            sx += (double)v.x; sy += (double)v.y; sz += (double)v.z; sw += (double)v.w;
        }
        reinterpret_cast<float4*>(out_grad)[i] = make_float4((float)sx, (float)sy, (float)sz, (float)sw);
    }
    if (blockIdx.x == 0 && threadIdx.x < (nfloat & 3)) {
        const int64_t e = (quads << 2) + threadIdx.x;
        double s = 0.0;
        for (int r = 0; r < world; ++r) s += (double)ld_relaxed_sys_f32(T.buf[r] + 64 + 4 * e);
        out_grad[e] = (float)s;
    }
}


// ------------------------------------------------------------------ two-shot variant (default)
// The one-shot kernel above moves world x (64 + 12n) bytes INTO every rank (4.8 MB at 50k loci on 8 GPUs) and takes
// its epoch from the host, so it cannot be captured in a CUDA graph.  Two-shot: after the first barrier rank r reduces
// only slice r of the gradient (1/world of it, read from all peers in rank order, f64 accumulation, rounded once) and
// stores the result into EVERY rank's result buffer; a second barrier tells everybody that all slices have landed.
// Per rank 2 x 12n bytes cross NVLink instead of world x 12n, every element is reduced exactly once (bit-identical on all
// ranks by construction), and -- because a rank leaves the kernel only after all peers have finished READING its partial --
// neither the partial nor the result buffer needs double buffering.  The epoch lives in device memory (`state[0]`, bumped
// by the last block to leave), so every launch has identical arguments: graph-capturable.  Launched with programmatic
// stream serialization: the blocks are resident (and have their parameters) when the producer grid completes.
struct PeerTable2 {
    const unsigned char* part[kMaxWorld];  // peer r's partial: [8 x f64 moments | 3n x f32 gradient, padded to 16 B]
    unsigned char* res[kMaxWorld];         // peer r's result buffer: 3n x f32 gradient, padded to 16 B
    uint32_t* pad[kMaxWorld];              // peer r's signal pad
};

__device__ __forceinline__ void st_relaxed_sys_f32x4(void* p, float4 v) {
    asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_gpu_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ ulonglong2 ld_relaxed_sys_u64x2(const void* p) {
    ulonglong2 v;
    asm volatile("ld.relaxed.sys.global.v2.u64 {%0,%1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_u64x2(void* p, ulonglong2 v) {
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(v.x), "l"(v.y) : "memory");
}

// The two barriers of a two-shot kernel (every block of the grid calls both, in order).  Entry: wait for the producer grid (programmatic
// stream serialization), take this launch's epoch from `state`, and barrier A -- every rank's source is complete.
__device__ __forceinline__ uint32_t twoshot_enter(const PeerTable2& T, int rank, int world, int slot_base, const uint32_t* state) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next kernel may set itself up behind this one
    asm volatile("griddepcontrol.wait;" ::: "memory");  // the producer of the local source has completed and flushed
    const uint32_t epoch = ld_relaxed_gpu_u32(state) + 1u;
    uint32_t* const sig_a = T.pad[rank] + slot_base;             // "source of epoch e is complete", one slot per source rank
    if (blockIdx.x == 0 && threadIdx.x < world) {
        __threadfence_system();
        st_release_sys(T.pad[threadIdx.x] + slot_base + rank, epoch);
    }
    if (threadIdx.x < world) {
        while ((int32_t)(ld_acquire_sys(sig_a + threadIdx.x) - epoch) < 0) { __nanosleep(20); }
    }
    __syncthreads();
    return epoch;
}

// Barrier B -- the last block of this rank to finish its stores signals every peer, all wait for every peer's signal -- then the last
// block to leave publishes the epoch and clears the tickets (every block has read state[0] by now).
__device__ __forceinline__ void twoshot_leave(const PeerTable2& T, int rank, int world, int slot_base, uint32_t* state, uint32_t epoch) {
    __shared__ unsigned s_ticket;
    uint32_t* const sig_b = T.pad[rank] + slot_base + kMaxWorld; // "my reduced slice of epoch e has landed everywhere"
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        s_ticket = atomicAdd(state + 1, 1u);
        __threadfence_system();
    }
    __syncthreads();
    if (s_ticket == gridDim.x - 1 && threadIdx.x < world) st_release_sys(T.pad[threadIdx.x] + slot_base + kMaxWorld + rank, epoch);
    if (threadIdx.x < world) {
        while ((int32_t)(ld_acquire_sys(sig_b + threadIdx.x) - epoch) < 0) { __nanosleep(20); }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t2 = atomicAdd(state + 2, 1u);
        if (t2 == gridDim.x - 1) {
            state[1] = 0u;
            state[2] = 0u;
            __threadfence();
            state[0] = epoch;
        }
    }
}

template <int WORLD>  // 0 = run-time world
__global__ void __launch_bounds__(256) allreduce_twoshot_kernel(const PeerTable2 T, int rank, int world_rt, int slot_base, uint32_t* __restrict__ state,
                                                                int64_t total_quads, int64_t slice_quads, const double* __restrict__ moment_const,
                                                                double* __restrict__ out_moments) {
    const int world = WORLD ? WORLD : world_rt;
    const uint32_t epoch = twoshot_enter(T, rank, world, slot_base, state);
    // ---- moments: 8 doubles per rank, every rank sums all of them in rank order
    if (blockIdx.x == 0 && threadIdx.x < HICGAT_PAIR_NMOM) {
        double s = 0.0;
        for (int r = 0; r < world; ++r) s += ld_relaxed_sys_f64(T.part[r] + 8 * threadIdx.x);
        out_moments[threadIdx.x] = s + (moment_const ? moment_const[threadIdx.x] : 0.0);
    }
    // ---- my slice: all `world` loads of an element in flight together, summed in rank order, stored to every rank
    const int64_t base = (int64_t)rank * slice_quads;
    int64_t cnt = total_quads - base;
    cnt = cnt < 0 ? 0 : (cnt > slice_quads ? slice_quads : cnt);
    constexpr int kUnroll = WORLD ? WORLD : kMaxWorld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = 16 * (base + i);
        float4 v[kUnroll];
#pragma unroll
        for (int r = 0; r < kUnroll; ++r) v[r] = r < world ? ld_relaxed_sys_f32x4(T.part[r] + 64 + off) : make_float4(0.f, 0.f, 0.f, 0.f);
        double sx = 0.0, sy = 0.0, sz = 0.0, sw = 0.0;
#pragma unroll
        for (int r = 0; r < kUnroll; ++r) {
            if (r < world) { sx += (double)v[r].x; sy += (double)v[r].y; sz += (double)v[r].z; sw += (double)v[r].w; }
        }
        const float4 o = make_float4((float)sx, (float)sy, (float)sz, (float)sw);
#pragma unroll
        for (int r = 0; r < kUnroll; ++r) {
            if (r < world) st_relaxed_sys_f32x4(T.res[r] + off, o);
        }
    }
    twoshot_leave(T, rank, world, slot_base, state, epoch);
}

// u64 sums: slice `rank` of the 16-byte pairs (and, on the last rank's slice owner, an odd trailing element), every load of an element in
// flight together, stored into every rank's result.  Integer adds: the result does not depend on the order.
__global__ void __launch_bounds__(256) allreduce_u64_twoshot_kernel(const PeerTable2 T, int rank, int world, int slot_base, uint32_t* __restrict__ state,
                                                                    int64_t count, int64_t slice_pairs) {
    const uint32_t epoch = twoshot_enter(T, rank, world, slot_base, state);
    const int64_t pairs = count >> 1;
    const int64_t base = (int64_t)rank * slice_pairs;
    int64_t cnt = pairs - base;
    cnt = cnt < 0 ? 0 : (cnt > slice_pairs ? slice_pairs : cnt);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t off = 16 * (base + i);
        ulonglong2 v[kMaxWorld];
#pragma unroll
        for (int r = 0; r < kMaxWorld; ++r) v[r] = r < world ? ld_relaxed_sys_u64x2(T.part[r] + off) : make_ulonglong2(0ull, 0ull);
        ulonglong2 o = make_ulonglong2(0ull, 0ull);
#pragma unroll
        for (int r = 0; r < kMaxWorld; ++r) { o.x += v[r].x; o.y += v[r].y; }
#pragma unroll
        for (int r = 0; r < kMaxWorld; ++r) {
            if (r < world) st_relaxed_sys_u64x2(T.res[r] + off, o);
        }
    }
    if ((count & 1) && rank == world - 1 && blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t off = 8 * (count - 1);
        unsigned long long o = 0ull;
        for (int r = 0; r < world; ++r) {
            unsigned long long v;
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(T.part[r] + off) : "memory");
            o += v;
        }
        for (int r = 0; r < world; ++r) asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(T.res[r] + off), "l"(o) : "memory");
    }
    twoshot_leave(T, rank, world, slot_base, state, epoch);
}

}  // namespace
}  // namespace hicgat

using namespace hicgat;

extern "C" int hicgat_allreduce_partials_p2p(const uint64_t* peer_bufs_host, const uint64_t* signal_pads_host, int rank, int world,
                                             int64_t n, int64_t buf_offset_bytes, int slot_base, uint32_t epoch,
                                             const double* moment_const, double* out_moments, float* out_grad,
                                             hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(peer_bufs_host && signal_pads_host && out_moments && out_grad, "hicgat_allreduce_partials_p2p: null pointer");
    HICGAT_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "hicgat_allreduce_partials_p2p: bad rank/world (%d/%d)", rank, world);
    HICGAT_REQUIRE(n > 0 && n < (1ll << 30) && buf_offset_bytes >= 0 && (buf_offset_bytes % 16) == 0 && slot_base >= 0, "hicgat_allreduce_partials_p2p: bad n/offset");
    HICGAT_REQUIRE(aligned16(out_grad), "hicgat_allreduce_partials_p2p: out_grad must be 16-byte aligned");
    PeerTable T;
    for (int r = 0; r < world; ++r) {
        HICGAT_REQUIRE(peer_bufs_host[r] && signal_pads_host[r], "hicgat_allreduce_partials_p2p: null peer pointer for rank %d", r);
        HICGAT_REQUIRE((peer_bufs_host[r] % 16) == 0, "hicgat_allreduce_partials_p2p: peer buffer %d not 16-byte aligned", r);
        T.buf[r] = reinterpret_cast<const unsigned char*>(peer_bufs_host[r] + (uint64_t)buf_offset_bytes);
        T.pad[r] = reinterpret_cast<uint32_t*>(signal_pads_host[r]);
    }
    const int64_t nfloat = 3 * n;
    int grid = (int)((nfloat / 4 + 255) / 256);
    if (grid > 148) grid = 148;  // all blocks co-resident: every block polls the barrier
    if (grid < 1) grid = 1;
    allreduce_partials_kernel<<<grid, 256, 0, stream>>>(T, rank, world, slot_base, epoch, nfloat, moment_const, out_moments, out_grad);
    HICGAT_CHECK_LAUNCH("allreduce_partials_kernel");
    return HICGAT_OK;
}

extern "C" int hicgat_allreduce_partials_twoshot(const uint64_t* peer_partials_host, const uint64_t* peer_results_host, const uint64_t* signal_pads_host,
                                                 int rank, int world, int64_t n, int slot_base, uint32_t* state, const double* moment_const,
                                                 double* out_moments, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(peer_partials_host && peer_results_host && signal_pads_host && out_moments && state, "hicgat_allreduce_partials_twoshot: null pointer");
    HICGAT_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "hicgat_allreduce_partials_twoshot: bad rank/world (%d/%d)", rank, world);
    HICGAT_REQUIRE(n > 0 && n < (1ll << 30) && slot_base >= 0, "hicgat_allreduce_partials_twoshot: bad n/slot_base");
    PeerTable2 T;
    for (int r = 0; r < world; ++r) {
        HICGAT_REQUIRE(peer_partials_host[r] && peer_results_host[r] && signal_pads_host[r], "hicgat_allreduce_partials_twoshot: null peer pointer for rank %d", r);
        HICGAT_REQUIRE((peer_partials_host[r] % 16) == 0 && (peer_results_host[r] % 16) == 0, "hicgat_allreduce_partials_twoshot: peer buffer %d not 16-byte aligned", r);
        T.part[r] = reinterpret_cast<const unsigned char*>(peer_partials_host[r]);
        T.res[r] = reinterpret_cast<unsigned char*>(peer_results_host[r]);
        T.pad[r] = reinterpret_cast<uint32_t*>(signal_pads_host[r]);
    }
    const int64_t total_quads = (3 * n + 3) / 4;  // buffers are padded to 16 bytes; the padding floats stay zero
    const int64_t slice_quads = (total_quads + world - 1) / world;
    int grid = (int)((slice_quads + 255) / 256);
    if (grid > 64) grid = 64;  // all blocks are co-resident (every block takes part in the barriers)
    if (grid < 1) grid = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(256);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e;
    switch (world) {
        case 2: e = cudaLaunchKernelEx(&cfg, allreduce_twoshot_kernel<2>, T, rank, world, slot_base, state, total_quads, slice_quads, moment_const, out_moments); break;
        case 4: e = cudaLaunchKernelEx(&cfg, allreduce_twoshot_kernel<4>, T, rank, world, slot_base, state, total_quads, slice_quads, moment_const, out_moments); break;
        case 8: e = cudaLaunchKernelEx(&cfg, allreduce_twoshot_kernel<8>, T, rank, world, slot_base, state, total_quads, slice_quads, moment_const, out_moments); break;
        default: e = cudaLaunchKernelEx(&cfg, allreduce_twoshot_kernel<0>, T, rank, world, slot_base, state, total_quads, slice_quads, moment_const, out_moments); break;
    }
    if (e != cudaSuccess) {
        set_error("allreduce_twoshot_kernel: launch failed: %s", cudaGetErrorString(e));
        return HICGAT_ERR_CUDA;
    }
    count_launch();
    return HICGAT_OK;
}

extern "C" int hicgat_allreduce_u64_twoshot(const uint64_t* peer_src_host, const uint64_t* peer_dst_host, const uint64_t* signal_pads_host, int rank,
                                            int world, int64_t count, int slot_base, uint32_t* state, hicgat_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    HICGAT_REQUIRE(peer_src_host && peer_dst_host && signal_pads_host && state, "hicgat_allreduce_u64_twoshot: null pointer");
    HICGAT_REQUIRE(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "hicgat_allreduce_u64_twoshot: bad rank/world (%d/%d)", rank, world);
    HICGAT_REQUIRE(count > 0 && slot_base >= 0, "hicgat_allreduce_u64_twoshot: bad count/slot_base");
    PeerTable2 T;
    for (int r = 0; r < world; ++r) {
        HICGAT_REQUIRE(peer_src_host[r] && peer_dst_host[r] && signal_pads_host[r], "hicgat_allreduce_u64_twoshot: null peer pointer for rank %d", r);
        HICGAT_REQUIRE((peer_src_host[r] % 16) == 0 && (peer_dst_host[r] % 16) == 0, "hicgat_allreduce_u64_twoshot: peer buffer %d not 16-byte aligned", r);
        T.part[r] = reinterpret_cast<const unsigned char*>(peer_src_host[r]);
        T.res[r] = reinterpret_cast<unsigned char*>(peer_dst_host[r]);
        T.pad[r] = reinterpret_cast<uint32_t*>(signal_pads_host[r]);
    }
    const int64_t slice_pairs = (count / 2 + world - 1) / world;
    int grid = (int)((slice_pairs + 255) / 256);
    if (grid > 64) grid = 64;  // all blocks are co-resident (every block takes part in the barriers)
    if (grid < 1) grid = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(256);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, allreduce_u64_twoshot_kernel, T, rank, world, slot_base, state, count, slice_pairs);
    if (e != cudaSuccess) {
        set_error("allreduce_u64_twoshot_kernel: launch failed: %s", cudaGetErrorString(e));
        return HICGAT_ERR_CUDA;
    }
    count_launch();
    return HICGAT_OK;
}
