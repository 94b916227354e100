// Shared device helpers of the tensor-core MLP stage kernels (mlp_tc.cu, mlp_pipe.cu): tcgen05 / TMEM / mbarrier /
// bulk-copy PTX wrappers, the 128-byte-swizzled operand tile layouts, the 3xTF32 split and the BatchNorm record.
#pragma once
#include "common.cuh"

// ---- argument blocks of the stage kernels (shared by the phase-serial kernels in mlp_tc.cu and the warp-specialised
// pipelines in mlp_pipe.cu)
struct LinFwdArgs {
    const float *X; int64_t N; int K;
    const float *in_bn; int in_act; float in_slope;
    const float *W; const float *bias; int M;
    float *Y;
    int stats;
    float *part;
    int num_tiles;
    int x_direct = 0;      // pipelined kernels: read X with plain (bounds-checked) global loads instead of bulk slabs (K % 4 != 0 or unaligned)
};
struct LinBwdArgs {
    const float *G; const float *Gseg; const int32_t *row2seg; const float *Yo; int64_t N; int M;
    const float *bn; const float *sums; int g_masked;
    const float *W; int K;
    const float *X; const float *in_bn; int in_act; float in_slope;
    float *GX;
    float *part;
    int num_tiles;
    int x_direct = 0;      // as in LinFwdArgs (only without a data gradient: the epilogue's mask pass reads the staged X slab)
};

// BatchNorm finalisation parameters of a forward stage (training-mode nn.BatchNorm1d semantics)
struct BnFinalArgs {
    const float *gamma; const float *beta; float eps; float momentum;
    float *bn_out; float *run_mean; float *run_var; long long *nbt;
};

namespace {

constexpr int TC_THREADS = 128;          // 4 warps <-> the 128 TMEM lanes
#ifndef TC_SPLIT_ACC
#define TC_SPLIT_ACC 1                   // accumulators per logical GEMM (1, 2; see lin_fwd_kernel)
#endif
constexpr uint32_t PANEL128 = 128u * 128u;   // bytes of one 128-row panel (32 floats per row)

__device__ __forceinline__ uint32_t s_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ bool aligned16_dev(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_alloc(uint32_t smem_dst, uint32_t cols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_dealloc(uint32_t taddr, uint32_t cols) {    // the same warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], tf32 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// this warp's 32 lanes x 32 consecutive columns -> 32 registers per thread (thread = lane = accumulator row)
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// v = sum of NB column blocks (32 columns each, `stride` columns apart): the hi/lo halves and split accumulators of one
// logical accumulator block, added smallest-index first with round-to-nearest fp32 adds
template <int NB>
__device__ __forceinline__ void tc_ld_sum(uint32_t taddr, uint32_t stride, float (&v)[32]) {
    tc_ld32(taddr, v);
    tc_wait_ld();
#pragma unroll
    for (int b = 1; b < NB; ++b) {
        float u[32];
        tc_ld32(taddr + b * stride, u);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += u[i];
    }
}

// shared-memory matrix descriptor, 128-byte swizzle (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout SWIZZLE_128B=2 [61,64))
constexpr uint32_t LAYOUT_SW128 = 2, LAYOUT_SW128_32B = 1;
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = LAYOUT_SW128) {
    uint64_t d = static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;
    d |= static_cast<uint64_t>(layout) << 61;
    return d;
}
// MN-major operand (the contraction index runs over tile ROWS): 32-bit types must use the 128B-swizzle with 32-byte
// base (cute::UMMA::LayoutType::SWIZZLE_128B_BASE32B; atoms of 32 floats x 4 rows, Swizzle<2,5,2> on byte addresses).
// LBO = stride between 32-float blocks of the MN index (a panel), SBO = stride between groups of 4 rows (512 B).
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr, uint32_t panel_bytes) {
    return make_desc(saddr, panel_bytes, 512u, LAYOUT_SW128_32B);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=f32 [4,6), a=b=tf32 [7,10)/[10,13), a/b major (1 = MN)
// [15]/[16], N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(a_mn) << 15) | (static_cast<uint32_t>(b_mn) << 16) |
           (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// byte offset of 16-byte chunk `chunk` (4 floats) of row `row` in a swizzled tile whose panels hold `panel_rows` rows
__device__ __forceinline__ uint32_t tile_off(int row, int chunk, int panel_rows) {
    return static_cast<uint32_t>(chunk >> 3) * static_cast<uint32_t>(panel_rows * 128) + static_cast<uint32_t>(row) * 128u +
           static_cast<uint32_t>(((chunk & 7) ^ (row & 7)) << 4);
}
// the same tile shape in the MN-major swizzle: 32-byte unit index XOR (row & 3)
__device__ __forceinline__ uint32_t tile_off_mn(int row, int chunk, int panel_rows) {
    return static_cast<uint32_t>(chunk >> 3) * static_cast<uint32_t>(panel_rows * 128) + static_cast<uint32_t>(row) * 128u +
           static_cast<uint32_t>(((chunk & 7) ^ ((row & 3) << 1)) << 4);
}
__device__ __forceinline__ void sts128(uint32_t a, const float4 &v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds128s(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
// x = hi + lo (+ O(2^-22 |x|)), both exactly representable in tf32 (round-to-nearest split)
__device__ __forceinline__ void split_tf32(float x, float &hi, float &lo) {
    uint32_t h, l;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));
    hi = __uint_as_float(h);
    const float r = x - hi;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"(r));
    lo = __uint_as_float(l);
}
// hi part to hi_base + off + off_hi, lo part to lo_base + off + off_lo
__device__ __forceinline__ void store_split(uint32_t hi_base, uint32_t lo_base, uint32_t off, const float4 &v, uint32_t off_hi,
                                            uint32_t off_lo) {
    float4 h, l;
    split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
    sts128(hi_base + off + off_hi, h);
    sts128(lo_base + off + off_lo, l);
}
// the same split value into two differently swizzled tiles (K-major copy + MN-major copy)
__device__ __forceinline__ void store_split2(uint32_t hi_a, uint32_t lo_a, uint32_t off_a, uint32_t hi_b, uint32_t lo_b,
                                             uint32_t off_b, const float4 &v) {
    float4 h, l;
    split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
    sts128(hi_a + off_a, h); sts128(lo_a + off_a, l);
    sts128(hi_b + off_b, h); sts128(lo_b + off_b, l);
}
// 4 consecutive floats of a row-major (rows x ncols, leading dimension ncols) matrix, zero beyond ncols
__device__ __forceinline__ float4 load_chunk(const float *__restrict__ base, int64_t row, int ncols, int c, bool vec) {
    float4 v = zero4();
    const int c0 = 4 * c;
    if (c0 >= ncols) return v;
    const float *p = base + row * ncols + c0;
    if (vec) return __ldg(reinterpret_cast<const float4 *>(p));
    v.x = __ldg(p);
    if (c0 + 1 < ncols) v.y = __ldg(p + 1);
    if (c0 + 2 < ncols) v.z = __ldg(p + 2);
    if (c0 + 3 < ncols) v.w = __ldg(p + 3);
    return v;
}
__device__ __forceinline__ void store_chunk(float *__restrict__ base, int64_t row, int ncols, int c, const float4 &v, bool vec) {
    const int c0 = 4 * c;
    if (c0 >= ncols) return;
    float *p = base + row * ncols + c0;
    if (vec) { *reinterpret_cast<float4 *>(p) = v; return; }
    p[0] = v.x;
    if (c0 + 1 < ncols) p[1] = v.y;
    if (c0 + 2 < ncols) p[2] = v.z;
    if (c0 + 3 < ncols) p[3] = v.w;
}
// per-channel vector (length n) -> the 4 channels of chunk c, zero beyond n
__device__ __forceinline__ float4 load_vec4(const float *__restrict__ v, int n, int c) {
    float4 r = zero4();
    if (v == nullptr) return r;
    const int c0 = 4 * c;
    if (c0 < n) r.x = __ldg(v + c0);
    if (c0 + 1 < n) r.y = __ldg(v + c0 + 1);
    if (c0 + 2 < n) r.z = __ldg(v + c0 + 2);
    if (c0 + 3 < n) r.w = __ldg(v + c0 + 3);
    return r;
}

__device__ __forceinline__ float act_f(float x, int act, float slope) {
    if (act == DN4GL_ACT_RELU) return fmaxf(x, 0.f);
    if (act == DN4GL_ACT_LEAKY_RELU) return x > 0.f ? x : slope * x;
    return x;
}
__device__ __forceinline__ float dact_f(float x, int act, float slope) {   // derivative at the pre-activation x
    if (act == DN4GL_ACT_RELU) return x > 0.f ? 1.f : 0.f;
    if (act == DN4GL_ACT_LEAKY_RELU) return x > 0.f ? 1.f : slope;
    return 1.f;
}

// BatchNorm record of one normalisation over C channels: rec[0:C) mean, [C:2C) rstd, [2C:3C) k = gamma*rstd, [3C:4C) beta
struct Bn4 {
    float4 mean, rstd, k, beta;
};
__device__ __forceinline__ Bn4 load_bn4(const float *rec, int C, int c) {
    Bn4 b;
    b.mean = load_vec4(rec, C, c);
    b.rstd = load_vec4(rec == nullptr ? nullptr : rec + C, C, c);
    b.k = load_vec4(rec == nullptr ? nullptr : rec + 2 * C, C, c);
    b.beta = load_vec4(rec == nullptr ? nullptr : rec + 3 * C, C, c);
    return b;
}
__device__ __forceinline__ float4 bn_apply(const float4 &x, const Bn4 &b) {
    return make_float4(fmaf(x.x - b.mean.x, b.k.x, b.beta.x), fmaf(x.y - b.mean.y, b.k.y, b.beta.y),
                       fmaf(x.z - b.mean.z, b.k.z, b.beta.z), fmaf(x.w - b.mean.w, b.k.w, b.beta.w));
}

// sum over the lanes of a warp that hold the same chunk (lanes l, l + CH, l + 2CH, ...), fixed butterfly
template <int CH>
__device__ __forceinline__ void chunk_allreduce(float4 &v) {
#pragma unroll
    for (int o = CH; o < 32; o <<= 1) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, o); v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
        v.z += __shfl_xor_sync(0xffffffffu, v.z, o); v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// raw-tile ring: a row tile of a row-major matrix is one contiguous slab, so ONE bulk asynchronous copy (TMA engine,
// cp.async.bulk ... mbarrier::complete_tx) per matrix brings it into shared memory, RING tiles ahead of its use; the
// global-load latency that bounded the first version of these kernels (profiles/r1c: long_scoreboard) is hidden.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void *src_gmem, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src_gmem), "r"(bytes), "r"(bar)
                 : "memory");
}
// chunk c (16 bytes) of row r of a raw slab with `ncols` floats per row (ncols % 4 == 0), zero beyond ncols
__device__ __forceinline__ float4 raw_chunk(uint32_t slab, int r, int ncols, int c) {
    if (4 * c >= ncols) return zero4();
    return lds128s(slab + static_cast<uint32_t>(r * ncols * 4 + c * 16));
}

// ---- grid rendezvous (kernels whose CTAs are all resident: launched COOPERATIVELY, launch_coop below).  The merges of
// per-CTA partials used to be done by the last CTA to finish (one ticket level in the forward stage, two in the backward
// stage) or by a follow-up kernel: 4.1 us / 7.4 us between the last CTA leaving its tile loop and the end of the stage
// kernels (profiles/r2z_pipe_timeline.txt), a fifth of the backward stage.  Now every CTA arrives once its partials are
// written, and the merge is SPREAD over the CTAs -- each takes a few output entries, the lanes / threads over the
// partials: one round of loads per entry instead of serial merge levels.
//   grid_arrive: the CTA's earlier global stores are published (bar.sync, then a gpu-scope fence by thread 0 -- the
//                cooperative-groups pattern) and the CTA is counted; merging CTAs wait until all G have arrived and take
//                a ticket saying so (issued before the merge, read after it: its round trip hides behind the loads).
//   grid_depart: the merging CTA holding the last ticket -- every other merger is past its wait by then -- puts both
//                counters back to zero for the next launch.
// The wait is bounded: a grid that never completes (a launch that was not cooperative after all) traps instead of
// hanging the device.
__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int grid_arrive(int *arrive, int *passed, int G, bool wait) {
    int ticket = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(arrive, 1);
        if (wait) {
            unsigned spins = 0;
            while (ld_acquire_gpu(arrive) < G)
                if (++spins > (1u << 25)) __trap();
            ticket = atomicAdd(passed, 1);
        }
    }
    __syncthreads();
    return ticket;      // meaningful in thread 0 of a merging CTA
}
__device__ __forceinline__ void grid_depart(int *arrive, int *passed, int ticket, int mergers) {
    if (threadIdx.x == 0 && ticket == mergers - 1) {
        *passed = 0;
        *arrive = 0;
    }
}
__device__ __forceinline__ double warp_sum_f64(double v) {      // fixed butterfly
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// cooperative launch: the driver places the grid only when ALL its CTAs fit on the device at once (and refuses a grid
// that never could), which is what the grid rendezvous relies on.  Captured into CUDA graphs like any other launch.
template <typename... P, typename... A>
static inline cudaError_t launch_coop(void (*kernel)(P...), int grid, int block, size_t smem, cudaStream_t stream, A &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(static_cast<unsigned>(block));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<P>(args)...);
}

}  // namespace
