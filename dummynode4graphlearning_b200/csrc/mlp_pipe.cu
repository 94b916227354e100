// libdn4gl.so -- the tensor-core MLP stages as WARP-SPECIALISED PIPELINES (round 2).
//
// mlp_tc.cu runs the phases of a row tile one after the other behind __syncthreads (load -> convert -> MMA -> read the
// accumulators -> store): at the sizes of the reference's configurations (1e5 rows, 8 tiles per SM) every phase is
// latency-bound and the kernel reaches a fifth of the HBM rate (profiles/r1d, r2a).  Here the same arithmetic is split
// over dedicated warps of ONE persistent CTA per SM that hand tiles to each other through mbarriers:
//
//   producer warp  (1 lane)   cp.async.bulk of the raw row slabs (TMA engine) into a RING of slots
//   converter warps           raw slab -> BatchNorm/activation prologue -> hi/lo tf32 split -> swizzled operand tiles
//   MMA warp       (1 lane)   tcgen05.mma.kind::tf32 into DOUBLE-BUFFERED tensor-memory accumulators, tcgen05.commit
//   epilogue warps (4)        tcgen05.ld -> bias / statistics / masks -> coalesced 128-bit global stores
//
// so that the load of tile t+2, the conversion of tile t+1, the MMAs of tile t+1 and the epilogue of tile t overlap.
// The few-CTA reduction kernels that used to follow every stage (bn_finalize, lin_bwd_reduce) are gone: the grid is
// launched cooperatively, every CTA publishes its partials and is counted (tc_common.cuh: grid_arrive), and the merge is
// spread over the CTAs -- each takes a few output entries and adds the partials in a fixed order, so the result does
// not depend on which CTA arrives last.
//
// Accuracy of the fp32 emulation (3xTF32, x = hi + lo): the tensor core truncates after every accumulation, a BIASED
// error that grows with the number of MMAs added into one accumulator at full magnitude (DESIGN.md section 4 K6).  Two
// measures: (1) all A_lo MMAs are issued FIRST (their sum is 2^-11 of the result, truncation at that magnitude is
// harmless) and only then the A_hi MMAs; (2) the A_hi k-steps are spread over NACC accumulators that the epilogue
// adds in round-to-nearest fp32.  The double-buffered accumulators hide the extra tensor-memory reads.
#include <type_traits>
#include "common.cuh"
#include "tc_common.cuh"

namespace {

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
template <int COUNT>
__device__ __forceinline__ void named_bar_sync(int id) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(COUNT) : "memory");
}
__device__ __forceinline__ void tc_ld32_nowait(uint32_t taddr, float (&v)[32]) {
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
// v = sum of NB column blocks (32 columns each, `stride` columns apart), blocks added in index order with round-to-nearest
// fp32 adds; at most two blocks are live in registers (tensor-memory loads have a ~12-cycle latency: nothing to hide)
template <int NB>
__device__ __forceinline__ void tc_ld_sum2(uint32_t taddr, uint32_t stride, float (&v)[32]) {
    tc_ld32_nowait(taddr, v);
#pragma unroll
    for (int b = 1; b < NB; ++b) {
        float u[32];
        tc_ld32_nowait(taddr + b * stride, u);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += u[i];
    }
    if (NB == 1) tc_wait_ld();
}

// ---- optional per-role wait accounting (debug build -DDN4GL_PIPE_TL, tools/pipe_timeline.py): cycles every role spends
// blocked in its mbarrier waits vs. its whole tile loop, per CTA.  g_pipe_tl[cta][role][0] = loop cycles, [1..3] = cycles
// in the role's 1st / 2nd / 3rd kind of wait.  The role that waits least is the pipeline's bottleneck.
#ifdef DN4GL_PIPE_TL
__device__ long long g_pipe_tl[148 * 4 * 4];
__device__ unsigned long long g_pipe_span[148 * 4];      // per CTA %globaltimer: entry, set-up done, roles done, exit
__device__ __forceinline__ unsigned long long gtime_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TL_SPAN(k) do { if (threadIdx.x == 0 && blockIdx.x < 148) g_pipe_span[blockIdx.x * 4 + (k)] = gtime_ns(); } while (0)
#define TL_DECL long long tl_t0 = clock64(), tl_w[3] = {0, 0, 0}
#define TL_WAIT(k, stmt) do { const long long c0__ = clock64(); stmt; tl_w[k] += clock64() - c0__; } while (0)
#define TL_DONE(role) do { if (blockIdx.x < 148) { long long *p__ = g_pipe_tl + (blockIdx.x * 4 + (role)) * 4; \
    p__[0] = clock64() - tl_t0; p__[1] = tl_w[0]; p__[2] = tl_w[1]; p__[3] = tl_w[2]; } } while (0)
#else
#define TL_SPAN(k) do { } while (0)
#define TL_DECL do { } while (0)
#define TL_WAIT(k, stmt) stmt
#define TL_DONE(role) do { } while (0)
#endif

__device__ __forceinline__ int lds32f_i(uint32_t a) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float lds32f(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
// shared -> global bulk asynchronous store (TMA engine), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, uint32_t src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *src_gmem, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// v = 8 chunks of 4 floats; afterwards register chunk p holds the original chunk p ^ (lane & 7): three conditional-swap
// stages (static register indices only), 96 selects
__device__ __forceinline__ void lane_rotate_chunks(float (&v)[32], int lane) {
#pragma unroll
    for (int bit = 0; bit < 3; ++bit) {
        const bool sw = (lane >> bit) & 1;
#pragma unroll
        for (int p = 0; p < 8; ++p) {
            if (p & (1 << bit)) continue;
            const int q = p | (1 << bit);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float x = v[4 * p + i], y = v[4 * q + i];
                v[4 * p + i] = sw ? y : x;
                v[4 * q + i] = sw ? x : y;
            }
        }
    }
}

// x = hi + lo for the 3xTF32 emulation, in 3 instructions per element: hi = x rounded to nearest at tf32 precision
// (integer add of half an ulp + mask; finite inputs), lo = x - hi (exact in fp32).  lo is stored as it is: the tensor core
// reads the upper 19 bits of a tf32 operand, i.e. truncates lo -- an error below 2^-21 |x| whose sign follows lo, which is
// symmetric around zero because hi is rounded to nearest (no bias).  (cvt.rna.tf32.f32 has no SASS instruction on sm_100:
// ptxas expands each one into 4, the split cost 9 instructions per element and bounded the converter warps.)
__device__ __forceinline__ void split_fast(float x, float &hi, float &lo) {
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
    lo = x - hi;
}
__device__ __forceinline__ void store_split_fast(uint32_t hi_addr, uint32_t lo_delta, const float4 &v) {
    float4 h, l;
    split_fast(v.x, h.x, l.x); split_fast(v.y, h.y, l.y); split_fast(v.z, h.z, l.z); split_fast(v.w, h.w, l.w);
    sts128(hi_addr, h);
    sts128(hi_addr + lo_delta, l);
}

template <int ACT>
__device__ __forceinline__ float act_t(float x, float slope) {
    if (ACT == DN4GL_ACT_RELU) return fmaxf(x, 0.f);
    if (ACT == DN4GL_ACT_LEAKY_RELU) return x > 0.f ? x : slope * x;
    return x;
}

// ------------------------------------------------------------------------------------------------------------------
// forward stage  Y = act(bn_in(X)) W^T + b  (+ batch statistics of Y and the BatchNorm record, merged after the grid rendezvous)
// ------------------------------------------------------------------------------------------------------------------
template <int KP, int MP, int NACC, int NBUF_A, int RING, int NCV, int NEPI, int NACCBUF>
struct FwdCfg {
    static constexpr int PK = KP / 32, PM = MP / 32;
    static constexpr int NWE = 4 * NEPI;                              // epilogue warps: NEPI groups of 4 (tiles j % NEPI)
    static constexpr int NT = (NWE + 2 + NCV) * 32;
    static constexpr int W_CONV0 = NWE, W_PROD = NWE + NCV, W_MMA = NWE + 1 + NCV;
    static constexpr uint32_t A_BYTES = PK * PANEL128;                 // one of hi / lo
    static constexpr uint32_t B_BYTES = PK * 2 * MP * 128u;
    static constexpr uint32_t RAW_BYTES = 128u * KP * 4u;
    static constexpr uint32_t STAGE_BYTES = PM * PANEL128;
    static constexpr uint32_t OFF_B = 0, OFF_A = OFF_B + B_BYTES, OFF_RAW = OFF_A + NBUF_A * 2 * A_BYTES,
                              OFF_STAGE = OFF_RAW + RING * RAW_BYTES, SMEM = OFF_STAGE + NEPI * STAGE_BYTES + 1024;
    static constexpr int KSTEPS = KP / 8, KPA = KSTEPS / NACC;
    static constexpr uint32_t ACC_COLS = NACC * 2 * MP, TCOLS_RAW = NACCBUF * ACC_COLS;   // NACCBUF accumulator sets (2 = double-buffered)
    static_assert(NACCBUF == 2 || NEPI == 1, "one accumulator set: one epilogue group");
    static constexpr uint32_t TCOLS = TCOLS_RAW <= 32 ? 32 : TCOLS_RAW <= 64 ? 64 : TCOLS_RAW <= 128 ? 128 : TCOLS_RAW <= 256 ? 256 : 512;
    static_assert(TCOLS_RAW <= 512, "tensor memory budget");
    static_assert(KSTEPS % NACC == 0, "k-steps per accumulator");
    static_assert(SMEM <= 227 * 1024 - 2048, "shared memory budget");
};

template <int KP, int MP, int NACC, int NBUF_A, int RING, int NCV, int NEPI, int NACCBUF>
__global__ void __launch_bounds__((4 * NEPI + 2 + NCV) * 32, 1)
lin_fwd_pipe_kernel(const LinFwdArgs a, const BnFinalArgs f, int *__restrict__ counter) {
    using C = FwdCfg<KP, MP, NACC, NBUF_A, RING, NCV, NEPI, NACCBUF>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (s_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sB = base + C::OFF_B, sA = base + C::OFF_A, sRaw = base + C::OFF_RAW, sStage = base + C::OFF_STAGE;
    __shared__ __align__(8) uint64_t bars[2 * RING + 2 * NBUF_A + 4];
    __shared__ uint32_t tmem_ptr;
    __shared__ float red[4 * NEPI][2 * MP];
    __shared__ float shift_s[NEPI][MP];
    __shared__ float ncta_s[NEPI];
    __shared__ __align__(16) float bias_sm[MP];
    const uint32_t bar0 = s_u32(bars);
    auto raw_full = [&](int s) { return bar0 + 8u * s; };
    auto raw_empty = [&](int s) { return bar0 + 8u * (RING + s); };
    auto a_full = [&](int b) { return bar0 + 8u * (2 * RING + b); };
    auto a_empty = [&](int b) { return bar0 + 8u * (2 * RING + NBUF_A + b); };
    auto acc_full = [&](int b) { return bar0 + 8u * (2 * RING + 2 * NBUF_A + b); };
    auto acc_empty = [&](int b) { return bar0 + 8u * (2 * RING + 2 * NBUF_A + 2 + b); };

    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    TL_SPAN(0);
    if (t == 0) {
        for (int s = 0; s < RING; ++s) { mbar_init(raw_full(s), 1); mbar_init(raw_empty(s), NCV); }
        for (int b = 0; b < NBUF_A; ++b) { mbar_init(a_full(b), NCV); mbar_init(a_empty(b), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full(b), 1); mbar_init(acc_empty(b), 4); }   // 4 = warps of one epilogue group
        fence_barrier_init();
    }
    if (w == C::W_MMA) tc_alloc(s_u32(&tmem_ptr), C::TCOLS);
    __syncthreads();
    // weights: W (M x K) row-major = K-major B operand, zero-padded to MP x KP, split once: per 32-float K panel the MP
    // hi rows then the MP lo rows, so that ONE MMA with N = 2 MP multiplies an A tile with [W_hi | W_lo]
    for (int i = t; i < MP * (KP / 4); i += C::NT) {
        const int m = i / (KP / 4), c = i % (KP / 4);
        float4 v = zero4();
        if (m < a.M && 4 * c < a.K)
            v = a.x_direct ? load_chunk(a.W, m, a.K, c, false) : __ldg(reinterpret_cast<const float4 *>(a.W + static_cast<size_t>(m) * a.K + 4 * c));
        store_split(sB, sB, 0, v, tile_off(m, c, 2 * MP), tile_off(MP + m, c, 2 * MP));
    }
    for (int i = t; i < MP; i += C::NT) bias_sm[i] = (a.bias != nullptr && i < a.M) ? __ldg(a.bias + i) : 0.f;
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_ptr;
    TL_SPAN(1);
    const int my_tiles = a.num_tiles > static_cast<int>(blockIdx.x) ? (a.num_tiles - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;

    if (w == C::W_PROD) {
        // ---------------------------------------------------------------- producer: raw X slabs into the ring
        if (lane == 0) {
            TL_DECL;
            for (int j = 0; j < my_tiles; ++j) {
                const int s = j % RING, use = j / RING;
                TL_WAIT(0, mbar_wait(raw_empty(s), (use & 1) ^ 1));
                const int64_t row0 = (static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(j) * gridDim.x) * 128;
                const int64_t left = a.N - row0;
                const uint32_t bytes = static_cast<uint32_t>((left < 128 ? left : 128) * a.K * 4);
                if (a.x_direct) {                      // the converters load X themselves: just hand the slot over
                    mbar_arrive(raw_full(s));
                } else {
                    mbar_expect_tx(raw_full(s), bytes);
                    bulk_g2s(sRaw + s * C::RAW_BYTES, a.X + row0 * a.K, bytes, raw_full(s));
                }
            }
            TL_DONE(0);
        }
    } else if (w == C::W_MMA) {
        // ---------------------------------------------------------------- MMA issuer
        if (lane == 0) {
            constexpr uint32_t IDESC = make_idesc(128, 2 * MP, 0, 0);
            TL_DECL;
            for (int j = 0; j < my_tiles; ++j) {
                const int b = j % NBUF_A, ub = j / NBUF_A, ab = j % NACCBUF, ua = j / NACCBUF;
                TL_WAIT(0, mbar_wait(acc_empty(ab), (ua & 1) ^ 1));
                TL_WAIT(1, mbar_wait(a_full(b), ub & 1));
                tc_fence_after();
                const uint32_t sAh = sA + b * 2 * C::A_BYTES, sAl = sAh + C::A_BYTES;
                const uint32_t d0 = tmem + ab * C::ACC_COLS;
#pragma unroll
                for (int jj = 0; jj < C::KSTEPS; ++jj) {     // all A_lo products first, into accumulator 0
                    const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u, boff = (jj >> 2) * (2 * MP * 128u) + (jj & 3) * 32u;
                    tc_mma_tf32(d0, make_desc(sAl + aoff, 16, 1024), make_desc(sB + boff, 16, 1024), IDESC, jj != 0 ? 1u : 0u);
                }
#pragma unroll
                for (int jj = 0; jj < C::KSTEPS; ++jj) {     // then the A_hi products, KPA k-steps per accumulator
                    const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u, boff = (jj >> 2) * (2 * MP * 128u) + (jj & 3) * 32u;
                    const int acc = jj / C::KPA;
                    tc_mma_tf32(d0 + acc * 2 * MP, make_desc(sAh + aoff, 16, 1024), make_desc(sB + boff, 16, 1024), IDESC,
                                (acc == 0 || (jj % C::KPA) != 0) ? 1u : 0u);
                }
                tc_commit(a_empty(b));
                tc_commit(acc_full(ab));
            }
            TL_DONE(1);
        }
    } else if (w >= C::W_CONV0 && w < C::W_PROD) {
        // ---------------------------------------------------------------- converters: raw -> bn/act -> hi/lo tiles
        constexpr int CT = NCV * 32, CH = KP / 4, RP = CT / CH;
        const int ct = t - C::W_CONV0 * 32, c_in = ct % CH, r_in = ct / CH;
        const Bn4 bi = load_bn4(a.in_bn, a.K, c_in);
        const float slope = a.in_slope;
        const bool col_ok = 4 * c_in < a.K;
        const uint32_t rpitch = static_cast<uint32_t>(a.K) * 4u;
        // rows past the end of the matrix (last tile only) are converted from whatever the slot holds: accumulator rows
        // depend on their own A row only and those rows are neither stored nor counted
        auto run = [&](auto bn_tag, auto act_tag) {
            constexpr bool BN = decltype(bn_tag)::value;
            constexpr int ACT = decltype(act_tag)::value;
            TL_DECL;
            for (int j = 0; j < my_tiles; ++j) {
                const int s = j % RING, us = j / RING, b = j % NBUF_A, ub = j / NBUF_A;
                TL_WAIT(0, mbar_wait(raw_full(s), us & 1));
                TL_WAIT(1, mbar_wait(a_empty(b), (ub & 1) ^ 1));
                const uint32_t src = sRaw + s * C::RAW_BYTES + static_cast<uint32_t>(r_in) * rpitch + c_in * 16;
                const uint32_t sAh = sA + b * 2 * C::A_BYTES;
                float4 v[128 / RP];
                if (a.x_direct) {                          // K % 4 != 0 or unaligned X: bounds-checked global loads
                    const int64_t row0 = (static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(j) * gridDim.x) * 128;
#pragma unroll
                    for (int i = 0; i < 128 / RP; ++i) {
                        const int64_t gr = row0 + r_in + RP * i;
                        v[i] = (col_ok && gr < a.N) ? load_chunk(a.X, gr, a.K, c_in, false) : zero4();
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 128 / RP; ++i) v[i] = col_ok ? lds128s(src + static_cast<uint32_t>(RP * i) * rpitch) : zero4();
                }
#pragma unroll
                for (int i = 0; i < 128 / RP; ++i) {
                    if (BN) v[i] = bn_apply(v[i], bi);
                    v[i].x = act_t<ACT>(v[i].x, slope); v[i].y = act_t<ACT>(v[i].y, slope);
                    v[i].z = act_t<ACT>(v[i].z, slope); v[i].w = act_t<ACT>(v[i].w, slope);
                    store_split_fast(sAh + tile_off(r_in + RP * i, c_in, 128), C::A_BYTES, v[i]);
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) { mbar_arrive(a_full(b)); mbar_arrive(raw_empty(s)); }
            }
            if (ct == 0) TL_DONE(2);
        };
        using T_ = std::true_type; using F_ = std::false_type;
        const int mode = (a.in_bn != nullptr ? 3 : 0) + a.in_act;
        switch (mode) {
            case 0: run(F_{}, std::integral_constant<int, DN4GL_ACT_NONE>{}); break;
            case 1: run(F_{}, std::integral_constant<int, DN4GL_ACT_RELU>{}); break;
            case 2: run(F_{}, std::integral_constant<int, DN4GL_ACT_LEAKY_RELU>{}); break;
            case 3: run(T_{}, std::integral_constant<int, DN4GL_ACT_NONE>{}); break;
            case 4: run(T_{}, std::integral_constant<int, DN4GL_ACT_RELU>{}); break;
            default: run(T_{}, std::integral_constant<int, DN4GL_ACT_LEAKY_RELU>{}); break;
        }
    } else {
        // ---------------------------------------------------------------- epilogue warps 0..3 (TMEM lane quadrant = w)
        // thread = accumulator row.  The row's MP outputs (+ bias) go to a LINEAR staging tile that mirrors the global row
        // pitch, so that ONE bulk asynchronous store (TMA engine) writes the whole tile; the 16-byte chunks of a row are
        // written in an order rotated by the lane (register butterfly, no dynamic register index), which makes the
        // thread-per-row shared-memory stores conflict-free.  Batch statistics: thread (channel, row group) re-reads the
        // staged tile column-wise (conflict-free) while the bulk store drains.
        constexpr int CH4 = MP / 4, RG4 = 128 / CH4;       // statistics pass: chunks per row, row groups
        const int eg = w >> 2, wq = w & 3, tg = t & 127;   // epilogue group (tiles j = eg, eg + NEPI, ...), lane quadrant, thread in group
        const int c_s4 = tg % CH4, rg4 = tg / CH4;
        const uint32_t sSt = sStage + eg * C::STAGE_BYTES;
        static_assert(NEPI == 1 || NEPI == 2, "one epilogue group per accumulator buffer");
        const bool stats = a.stats != 0, st_ok = 4 * c_s4 < a.M;
        const uint32_t pitch = static_cast<uint32_t>(a.M) * 4u;
        const uint32_t bias_s = s_u32(bias_sm);
        float4 S1 = zero4(), S2 = zero4(), shift4 = zero4();
        bool have_shift = false;
        float n_cta = 0.f;
        TL_DECL;
        for (int j = eg; j < my_tiles; j += NEPI) {
            const int ab = j % NACCBUF, ua = j / NACCBUF;
            const int64_t row0 = (static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(j) * gridDim.x) * 128;
            const int valid = static_cast<int>((a.N - row0) < 128 ? (a.N - row0) : 128);
            TL_WAIT(0, mbar_wait(acc_full(ab), ua & 1));
            tc_fence_after();
            [[maybe_unused]] const long long tl_p0 = clock64();
            const uint32_t tacc = tmem + ab * C::ACC_COLS + (static_cast<uint32_t>(wq * 32) << 16);
            if (tg == 0) bulk_wait_read0();                 // the previous tile's store has read the staging tile
            named_bar_sync<128>(1 + eg);                        // ... and its statistics pass is over
#pragma unroll
            for (int cb = 0; cb < C::PM; ++cb) {
                float v[32];
                tc_ld_sum2<2 * NACC>(tacc + cb * 32, MP, v);
                if (cb == C::PM - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty(ab));     // the accumulators are free for tile j + 2
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 b4 = lds128s(bias_s + (cb * 8 + q) * 16);
                    v[4 * q] += b4.x; v[4 * q + 1] += b4.y; v[4 * q + 2] += b4.z; v[4 * q + 3] += b4.w;
                }
                lane_rotate_chunks(v, lane);               // register chunk p now holds the row's chunk p ^ (lane & 7)
#pragma unroll
                for (int p = 0; p < 8; ++p) {
                    const int chunk = cb * 8 + (p ^ (lane & 7));
                    if (4 * chunk < a.M)
                        sts128(sSt + static_cast<uint32_t>(tg) * pitch + chunk * 16, make_float4(v[4 * p], v[4 * p + 1], v[4 * p + 2], v[4 * p + 3]));
                }
            }
            fence_async_smem();
            named_bar_sync<128>(1 + eg);
#ifdef DN4GL_PIPE_TL
            const long long tl_p1 = clock64();
            tl_w[1] += tl_p1 - tl_p0;
#endif
            if (tg == 0) {
                bulk_s2g(a.Y + row0 * a.M, sSt, static_cast<uint32_t>(valid) * pitch);
                bulk_commit();
            }
            if (stats && st_ok) {
                // thread (chunk c_s4, row group rg4): 128-bit reads of its 4 channels, rows rg4, rg4 + RG4, ...
                if (!have_shift) {
                    shift4 = lds128s(sSt + c_s4 * 16);
                    have_shift = true;
                }
                uint32_t addr = sSt + static_cast<uint32_t>(rg4) * pitch + c_s4 * 16;
                for (int r = rg4; r < valid; r += RG4, addr += RG4 * pitch) {
                    const float4 y = lds128s(addr);
                    const float dx = y.x - shift4.x, dy = y.y - shift4.y, dz = y.z - shift4.z, dw = y.w - shift4.w;
                    S1.x += dx; S1.y += dy; S1.z += dz; S1.w += dw;
                    S2.x = fmaf(dx, dx, S2.x); S2.y = fmaf(dy, dy, S2.y); S2.z = fmaf(dz, dz, S2.z); S2.w = fmaf(dw, dw, S2.w);
                }
            }
            n_cta += static_cast<float>(valid);
#ifdef DN4GL_PIPE_TL
            tl_w[2] += clock64() - tl_p1;
#endif
        }
        if (tg == 0) bulk_wait_all0();
        if (t == 0) TL_DONE(3);
        if (stats) {
            // lanes l, l + CH4, ... of a warp hold the same chunk: fixed butterfly; then the warps of the group through
            // shared memory; with two groups, group 1's sums are re-centred on group 0's shift (double, fixed formula)
            chunk_allreduce<CH4>(S1);
            chunk_allreduce<CH4>(S2);
            if (lane < (CH4 < 32 ? CH4 : 32)) {
                float *p = &red[w][0];
                const int c0 = 4 * c_s4;
                p[c0] = S1.x; p[c0 + 1] = S1.y; p[c0 + 2] = S1.z; p[c0 + 3] = S1.w;
                p[MP + c0] = S2.x; p[MP + c0 + 1] = S2.y; p[MP + c0 + 2] = S2.z; p[MP + c0 + 3] = S2.w;
            }
            if (rg4 == 0) {
                const int c0 = 4 * c_s4;
                shift_s[eg][c0] = shift4.x; shift_s[eg][c0 + 1] = shift4.y; shift_s[eg][c0 + 2] = shift4.z; shift_s[eg][c0 + 3] = shift4.w;
            }
            if (tg == 0) ncta_s[eg] = n_cta;
            asm volatile("bar.sync 3, %0;" ::"n"(128 * NEPI) : "memory");
            if (t < MP) {
                float s1 = 0.f, s2 = 0.f;
#pragma unroll
                for (int ww = 0; ww < 4; ++ww) { s1 += red[ww][t]; s2 += red[ww][MP + t]; }
                float n = ncta_s[0];
                if (NEPI == 2 && ncta_s[NEPI - 1] > 0.f) {
                    float u1 = 0.f, u2 = 0.f;
#pragma unroll
                    for (int ww = 4; ww < 4 * NEPI; ++ww) { u1 += red[ww][t]; u2 += red[ww][MP + t]; }
                    const double n1 = ncta_s[NEPI - 1], d = static_cast<double>(shift_s[NEPI - 1][t]) - static_cast<double>(shift_s[0][t]);
                    const double nd = n1 * d;
                    s1 = static_cast<float>(static_cast<double>(s1) + (static_cast<double>(u1) + nd));
                    s2 = static_cast<float>(static_cast<double>(s2) + (static_cast<double>(u2) + d * (2.0 * static_cast<double>(u1) + nd)));
                    n += ncta_s[NEPI - 1];
                }
                reinterpret_cast<float4 *>(a.part)[static_cast<size_t>(blockIdx.x) * MP + t] = make_float4(n, shift_s[0][t], s1, s2);
            }
        }
    }
    // ---- teardown; with statistics: grid rendezvous, then CTA b merges channels b, b + G, ... into the BatchNorm record
    tc_fence_before();
    __syncthreads();
    TL_SPAN(2);
    if (w == C::W_MMA) tc_dealloc(tmem, C::TCOLS);
    if (!a.stats) { TL_SPAN(3); return; }
    const int G = static_cast<int>(gridDim.x);
    const bool merger = static_cast<int>(blockIdx.x) < a.M;
    const int n_mergers = G < a.M ? G : a.M;
    const int passed = grid_arrive(counter, counter + 1, G, merger);
    if (!merger) { TL_SPAN(3); return; }
    {
        // one warp per channel, lanes over the per-CTA partials {n, a, S1 = sum (y - a), S2 = sum (y - a)^2}.  Every partial
        // is re-centred on K* = the mean of CTA 0's rows (exact in double): with d = a - K*,
        //   sum (y - K*) = S1 + n d,   sum (y - K*)^2 = S2 + d (2 S1 + n d),
        // so T2 - T1^2 / N has no cancellation to speak of.  Lane l adds partials l, l + 32, ... in that order, then a
        // fixed butterfly over the lanes: a fixed summation tree, double arithmetic, no divisions in the loop.
        const float4 *part = reinterpret_cast<const float4 *>(a.part);
        for (int c = static_cast<int>(blockIdx.x) + G * w; c < a.M; c += G * (C::NT / 32)) {
            const float4 p0 = __ldcg(part + c);
            double A1 = 0.0, A2 = 0.0, kstar = 0.0;
            constexpr int UNR = 5;      // 5 x 32 lanes >= 148 CTAs: one round of loads
            for (int q0 = 0; q0 < G; q0 += 32 * UNR) {
                float4 v[UNR];
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const int q = q0 + lane + 32 * u;
                    v[u] = (q < G) ? __ldcg(part + static_cast<size_t>(q) * MP + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                if (q0 == 0) kstar = static_cast<double>(p0.y) + static_cast<double>(p0.z) / static_cast<double>(p0.x);
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const double n = v[u].x, s1 = v[u].z, s2 = v[u].w;
                    const double d = static_cast<double>(v[u].y) - kstar, nd = n * d;
                    if (v[u].x > 0.f) {
                        A1 += s1 + nd;
                        A2 += s2 + d * (2.0 * s1 + nd);
                    }
                }
            }
            const double a1 = warp_sum_f64(A1), a2 = warp_sum_f64(A2);
            if (lane == 0) {
                const double Nd = static_cast<double>(a.N);
                const double mean = kstar + a1 / Nd;
                double m2 = a2 - a1 * a1 / Nd;
                if (m2 < 0.0) m2 = 0.0;
                const double var = m2 / Nd;
                const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(f.eps)));
                const float gam = f.gamma ? f.gamma[c] : 1.f, bet = f.beta ? f.beta[c] : 0.f;
                const int M = a.M;
                f.bn_out[c] = static_cast<float>(mean);
                f.bn_out[M + c] = rstd;
                f.bn_out[2 * M + c] = gam * rstd;
                f.bn_out[3 * M + c] = bet;
                if (f.run_mean) f.run_mean[c] = (1.f - f.momentum) * f.run_mean[c] + f.momentum * static_cast<float>(mean);
                if (f.run_var) {
                    const double unb = a.N > 1 ? m2 / (Nd - 1.0) : var;
                    f.run_var[c] = (1.f - f.momentum) * f.run_var[c] + f.momentum * static_cast<float>(unb);
                }
            }
        }
        if (blockIdx.x == 0 && t == 0 && f.nbt) *f.nbt += 1;
        grid_depart(counter, counter + 1, passed, n_mergers);
        TL_SPAN(3);
    }
}

template <int KP, int MP, int NACC, int NBUF_A, int RING, int NCV, int NEPI, int NACCBUF>
int launch_fwd_pipe(const LinFwdArgs &a, const BnFinalArgs &f, int *counter, cudaStream_t s) {
    using C = FwdCfg<KP, MP, NACC, NBUF_A, RING, NCV, NEPI, NACCBUF>;
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(lin_fwd_pipe_kernel<KP, MP, NACC, NBUF_A, RING, NCV, NEPI, NACCBUF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(C::SMEM)) != cudaSuccess)
            return -1;
        attr_done = true;
    }
    const int sms = dn4gl_num_sms();
    const int grid = a.num_tiles < sms ? a.num_tiles : sms;
    if (a.stats) {      // the statistics merge rendezvouses the grid: every CTA must be resident
        if (launch_coop(lin_fwd_pipe_kernel<KP, MP, NACC, NBUF_A, RING, NCV, NEPI, NACCBUF>, grid, C::NT, C::SMEM, s, a, f, counter) != cudaSuccess)
            return -1;
    } else {
        lin_fwd_pipe_kernel<KP, MP, NACC, NBUF_A, RING, NCV, NEPI, NACCBUF><<<grid, C::NT, C::SMEM, s>>>(a, f, counter);
    }
    return grid;
}


// ------------------------------------------------------------------------------------------------------------------
// backward stage:  gY = BatchNorm(+ReLU) backward of (G + Gseg[row2seg]),  GX = (gY W) * act'(bn_in(X)),
//                  dW = gY^T X',  db = colsum gY,  sums_prev = {sum GX, sum GX * xhat_in}      (see include/dn4gl.h)
// Roles as in the forward kernel.  Differences:
//   * the converters read G and Yout straight from global memory, 4 row passes ahead (register window), because the
//     operand tiles (gY twice -- K-major for the data GEMM, MN-major for the weight GEMM -- and X', hi and lo each: 96 KB
//     at 32 x 32) leave no room for a raw ring of all three inputs; X (+ the row -> graph map) comes through the TMA ring,
//     the epilogue needs it again for the activation mask;
//   * the weight-gradient accumulator starts fresh every tile (16 MMAs) and the epilogue adds it to a shared-memory copy
//     with fp32 adds, so the accumulation error does not grow with the number of tiles (DESIGN.md section 4 K6);
//   * per-CTA partials {dW, db, sums} are merged by LAST-FINISHER tickets in two levels (groups of BWD_GROUP CTAs, then
//     the groups), all additions in CTA-index order in double: deterministic, no separate reduce launch.
// ------------------------------------------------------------------------------------------------------------------
constexpr int BWD_GROUP = 12;
__host__ __device__ constexpr int bwd_pipe_part_floats(int KP, int MP) { return MP * KP + MP + 2 * KP; }

template <int KP, int MP, int RING, int NCV, int NEPI_>
struct BwdCfg {
    static constexpr int PK = KP / 32, PM = MP / 32;
    static constexpr int NEPI = NEPI_, NWE = 4 * NEPI;                                     // epilogue groups (tiles j % NEPI) of 4 warps
    static constexpr int NT = (NWE + 2 + NCV) * 32;
    static constexpr int W_CONV0 = NWE, W_PROD = NWE + NCV, W_MMA = NWE + 1 + NCV;
    static constexpr uint32_t G_BYTES = PM * PANEL128, X_BYTES = PK * PANEL128, W_BYTES = PK * MP * 128u;
    static constexpr uint32_t RAW_X = 128u * KP * 4u, RAW_SLOT = RAW_X + 512u;          // X rows + 128 row -> graph ids
    static constexpr uint32_t STAGE_BYTES = PK * PANEL128;
    static constexpr uint32_t ACCW_BYTES = 2u * MP * KP * 4u;                           // [KP/4 chunks][2 MP lanes] float4
    static constexpr uint32_t OFF_GM = 0, OFF_GK = OFF_GM + 2 * G_BYTES, OFF_X = OFF_GK + 2 * G_BYTES, OFF_W = OFF_X + 2 * X_BYTES,
                              OFF_RAW = OFF_W + 2 * W_BYTES, OFF_STAGE = OFF_RAW + RING * RAW_SLOT, OFF_ACCW = OFF_STAGE + NEPI * STAGE_BYTES,
                              SMEM = OFF_ACCW + NEPI * ACCW_BYTES + 1024;
    static constexpr int KS_D = MP / 8;
    static constexpr uint32_t ACC_COLS = 4 * KP;                                        // data accumulator 2 KP + weight accumulator 2 KP
    static constexpr uint32_t TCOLS = 2 * ACC_COLS <= 256 ? 256 : 512;
    static_assert(2 * ACC_COLS <= 512, "tensor memory budget");
    static_assert(2 * MP <= 128, "the weight-gradient MMA stacks gY hi and lo along M = 128");
    static_assert(SMEM <= 227 * 1024 - 3072, "shared memory budget");
};

template <int KP, int MP, int RING, int NCV, int NEPI_>
__global__ void __launch_bounds__((4 * NEPI_ + 2 + NCV) * 32, 1)
lin_bwd_pipe_kernel(const LinBwdArgs a, float *__restrict__ dW, float *__restrict__ db, float *__restrict__ sums_prev,
                    float *__restrict__ gpart, int *__restrict__ counters) {
    using C = BwdCfg<KP, MP, RING, NCV, NEPI_>;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (s_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sGm = base + C::OFF_GM, sGk = base + C::OFF_GK, sX = base + C::OFF_X, sW = base + C::OFF_W,
                   sRaw = base + C::OFF_RAW, sStage = base + C::OFF_STAGE, sAccW = base + C::OFF_ACCW;
    __shared__ __align__(8) uint64_t bars[2 * RING + 2 + 4];
    __shared__ uint32_t tmem_ptr;
    __shared__ float red_db[NCV][MP];
    __shared__ float red_sp[4 * C::NEPI][2 * KP];
    const uint32_t bar0 = s_u32(bars);
    auto raw_full = [&](int s) { return bar0 + 8u * s; };
    auto raw_empty = [&](int s) { return bar0 + 8u * (RING + s); };
    const uint32_t a_full = bar0 + 8u * (2 * RING), a_empty = bar0 + 8u * (2 * RING + 1);
    auto acc_full = [&](int b) { return bar0 + 8u * (2 * RING + 2 + b); };
    auto acc_empty = [&](int b) { return bar0 + 8u * (2 * RING + 4 + b); };

    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    TL_SPAN(0);
    if (t == 0) {
        for (int s = 0; s < RING; ++s) { mbar_init(raw_full(s), 1); mbar_init(raw_empty(s), NCV + 4); }   // converter warps + the 4 warps of the tile's epilogue group
        mbar_init(a_full, NCV); mbar_init(a_empty, 1);
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full(b), 1); mbar_init(acc_empty(b), 4); }
        fence_barrier_init();
    }
    if (w == C::W_MMA) tc_alloc(s_u32(&tmem_ptr), C::TCOLS);
    __syncthreads();
    const bool want_gx = a.GX != nullptr, has_bn = a.bn != nullptr, has_bn_in = a.in_bn != nullptr, has_seg = a.Gseg != nullptr;
    // weights as they are stored: rows m (the data GEMM's K), k contiguous (its N) -> MN-major B operand, hi panels then lo
    if (want_gx) {
        for (int i = t; i < MP * (KP / 4); i += C::NT) {
            const int m = i / (KP / 4), c = i % (KP / 4);
            float4 v = zero4();
            if (m < a.M && 4 * c < a.K) v = __ldg(reinterpret_cast<const float4 *>(a.W + static_cast<size_t>(m) * a.K + 4 * c));
            store_split(sW, sW + C::W_BYTES, tile_off_mn(m, c, MP), v, 0, 0);
        }
    }
    for (uint32_t i = t * 16u; i < C::NEPI * C::ACCW_BYTES; i += C::NT * 16u) sts128(sAccW + i, zero4());
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_ptr;
    TL_SPAN(1);
    const int my_tiles = a.num_tiles > static_cast<int>(blockIdx.x) ? (a.num_tiles - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;
    auto tile_row0 = [&](int j) { return (static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(j) * gridDim.x) * 128; };
    const bool need_mask = want_gx && (a.in_act != DN4GL_ACT_NONE || has_bn_in);
    float *part = reinterpret_cast<float *>(a.part) + static_cast<size_t>(blockIdx.x) * bwd_pipe_part_floats(KP, MP);

    if (w == C::W_PROD) {
        // ---------------------------------------------------------------- producer: raw X slabs (+ row -> graph ids)
        if (lane == 0) {
            TL_DECL;
            if (my_tiles > 1) {                                  // tile 1's G / Yout slabs (tile 0 is loaded right away)
                const int64_t prow = tile_row0(1), pleft = a.N - prow;
                const uint32_t pb = static_cast<uint32_t>(pleft < 128 ? pleft : 128) * a.M * 4u;
                if (a.G != nullptr) bulk_prefetch_l2(a.G + prow * a.M, pb);
                if (has_bn) bulk_prefetch_l2(a.Yo + prow * a.M, pb);
            }
            for (int j = 0; j < my_tiles; ++j) {
                const int s = j % RING, use = j / RING;
                TL_WAIT(0, mbar_wait(raw_empty(s), (use & 1) ^ 1));
                const int64_t row0 = tile_row0(j), left = a.N - row0;
                const uint32_t rows = static_cast<uint32_t>(left < 128 ? left : 128);
                const uint32_t xb = rows * a.K * 4u, sb = has_seg ? ((rows * 4u + 15u) & ~15u) : 0u;
                if (a.x_direct && !has_seg) {
                    mbar_arrive(raw_full(s));              // nothing to stage: the converters load X themselves
                } else {
                    mbar_expect_tx(raw_full(s), (a.x_direct ? 0u : xb) + sb);
                    if (!a.x_direct) bulk_g2s(sRaw + s * C::RAW_SLOT, a.X + row0 * a.K, xb, raw_full(s));
                    if (has_seg) bulk_g2s(sRaw + s * C::RAW_SLOT + C::RAW_X, a.row2seg + row0, sb, raw_full(s));
                }
                // G and Yout are read by the converters with plain loads one tile ahead: pull their slabs into L2 early
                // (TMA L2 prefetch), so that those loads see L2 latency instead of a loaded HBM queue
                if (j + 2 < my_tiles) {
                    const int64_t prow = tile_row0(j + 2), pleft = a.N - prow;
                    const uint32_t pb = static_cast<uint32_t>(pleft < 128 ? pleft : 128) * a.M * 4u;
                    if (a.G != nullptr) bulk_prefetch_l2(a.G + prow * a.M, pb);
                    if (has_bn) bulk_prefetch_l2(a.Yo + prow * a.M, pb);
                }
            }
            TL_DONE(0);
        }
    } else if (w == C::W_MMA) {
        // ---------------------------------------------------------------- MMA issuer
        if (lane == 0) {
            constexpr uint32_t IDESC_DATA = make_idesc(128, 2 * KP, 0, 1);   // gY (K-major) x [W_hi | W_lo] (MN-major)
            constexpr uint32_t IDESC_WGT = make_idesc(128, 2 * KP, 1, 1);    // [gY_hi ; gY_lo]^T (MN-major) x [X'_hi | X'_lo] (MN-major)
            const uint32_t sGh = sGk, sGl = sGk + C::G_BYTES;
            TL_DECL;
            for (int j = 0; j < my_tiles; ++j) {
                const int ab = j & 1, ua = j >> 1;
                TL_WAIT(0, mbar_wait(acc_empty(ab), (ua & 1) ^ 1));
                TL_WAIT(1, mbar_wait(a_full, j & 1));
                tc_fence_after();
                const uint32_t dD = tmem + ab * C::ACC_COLS, dWt = dD + 2 * KP;
                if (want_gx) {
#pragma unroll
                    for (int jj = 0; jj < C::KS_D; ++jj) {     // gY_lo products first (see the header of this file)
                        const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u;
                        tc_mma_tf32(dD, make_desc(sGl + aoff, 16, 1024), make_desc_mn(sW + jj * 1024u, MP * 128u), IDESC_DATA, jj != 0 ? 1u : 0u);
                    }
#pragma unroll
                    for (int jj = 0; jj < C::KS_D; ++jj) {
                        const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u;
                        tc_mma_tf32(dD, make_desc(sGh + aoff, 16, 1024), make_desc_mn(sW + jj * 1024u, MP * 128u), IDESC_DATA, 1u);
                    }
                }
#pragma unroll
                for (int jj = 0; jj < 16; ++jj)                 // weight gradient of this tile: k-steps of 8 rows, fresh accumulator
                    tc_mma_tf32(dWt, make_desc_mn(sGm + jj * 1024u, PANEL128), make_desc_mn(sX + jj * 1024u, PANEL128), IDESC_WGT,
                                jj != 0 ? 1u : 0u);
                tc_commit(a_empty);
                tc_commit(acc_full(ab));
            }
            TL_DONE(1);
        }
    } else if (w >= C::W_CONV0 && w < C::W_PROD) {
        // ---------------------------------------------------------------- converters
        constexpr int CT = NCV * 32, CHm = MP / 4, RPm = CT / CHm, NPm = 128 / RPm, CHk = KP / 4, RPk = CT / CHk, NPk = 128 / RPk;
        constexpr int PF = 4;                                  // row passes of G / Yout in flight (register window)
        static_assert(NPm % PF == 0, "window slots must be static");
        const int ct = t - C::W_CONV0 * 32, c_m = ct % CHm, r_m = ct / CHm, c_k = ct % CHk, r_k = ct / CHk;
        const bool colm_ok = 4 * c_m < a.M, colk_ok = 4 * c_k < a.K;
        const Bn4 bo = load_bn4(a.bn, a.M, c_m), bi = load_bn4(a.in_bn, a.K, c_k);
        float4 m1 = zero4(), m2r = zero4();
        if (has_bn) {
            const float invN = 1.f / static_cast<float>(a.N);
            const float4 s1 = load_vec4(a.sums, a.M, c_m), s2 = load_vec4(a.sums + a.M, a.M, c_m);
            m1 = make_float4(s1.x * invN, s1.y * invN, s1.z * invN, s1.w * invN);
            m2r = make_float4(s2.x * invN * bo.rstd.x, s2.y * invN * bo.rstd.y, s2.z * invN * bo.rstd.z, s2.w * invN * bo.rstd.w);
        }
        const bool g_masked = a.g_masked != 0;
        const int in_act = a.in_act;
        const float in_slope = a.in_slope;
        const uint32_t rpitch = static_cast<uint32_t>(a.K) * 4u;
        float4 db4 = zero4();
        float4 gw[PF], yw[PF];
        auto issue = [&](int j, int i, float4 &gd, float4 &yd) {
            gd = zero4(); yd = zero4();
            if (j >= my_tiles || !colm_ok) return;
            const int64_t row = tile_row0(j) + r_m + RPm * i;
            if (row >= a.N) return;
            if (a.G != nullptr) gd = __ldg(reinterpret_cast<const float4 *>(a.G + row * a.M + 4 * c_m));
            if (has_bn) yd = __ldg(reinterpret_cast<const float4 *>(a.Yo + row * a.M + 4 * c_m));
        };
#pragma unroll
        for (int i = 0; i < PF; ++i) issue(0, i, gw[i], yw[i]);
        TL_DECL;
        for (int j = 0; j < my_tiles; ++j) {
            const int s = j % RING, us = j / RING;
            const int64_t row0 = tile_row0(j);
            const int valid = static_cast<int>((a.N - row0) < 128 ? (a.N - row0) : 128);
            TL_WAIT(0, mbar_wait(raw_full(s), us & 1));
            TL_WAIT(1, mbar_wait(a_empty, (j & 1) ^ 1));
            const uint32_t slab = sRaw + s * C::RAW_SLOT;
            // ---- gY (BatchNorm backward folded in) -> K-major copy (data GEMM) + MN-major copy (weight GEMM), hi and lo
#pragma unroll
            for (int i = 0; i < NPm; ++i) {
                const int r = r_m + RPm * i;
                float4 g = gw[i % PF];
                const float4 y = yw[i % PF];
                if (i + PF < NPm) issue(j, i + PF, gw[i % PF], yw[i % PF]);      // later passes of THIS tile
                if (r < valid && colm_ok) {
                    if (has_seg) {
                        const int seg = static_cast<int>(lds32f_i(slab + C::RAW_X + r * 4));
                        const float4 gs = __ldg(reinterpret_cast<const float4 *>(a.Gseg + static_cast<size_t>(seg) * a.M + 4 * c_m));
                        g.x += gs.x; g.y += gs.y; g.z += gs.z; g.w += gs.w;
                    }
                    if (has_bn) {
                        const float4 xc = make_float4(y.x - bo.mean.x, y.y - bo.mean.y, y.z - bo.mean.z, y.w - bo.mean.w);
                        if (!g_masked) {
                            if (!(fmaf(xc.x, bo.k.x, bo.beta.x) > 0.f)) g.x = 0.f;
                            if (!(fmaf(xc.y, bo.k.y, bo.beta.y) > 0.f)) g.y = 0.f;
                            if (!(fmaf(xc.z, bo.k.z, bo.beta.z) > 0.f)) g.z = 0.f;
                            if (!(fmaf(xc.w, bo.k.w, bo.beta.w) > 0.f)) g.w = 0.f;
                        }
                        g.x = bo.k.x * (g.x - m1.x - xc.x * m2r.x);
                        g.y = bo.k.y * (g.y - m1.y - xc.y * m2r.y);
                        g.z = bo.k.z * (g.z - m1.z - xc.z * m2r.z);
                        g.w = bo.k.w * (g.w - m1.w - xc.w * m2r.w);
                    }
                    db4.x += g.x; db4.y += g.y; db4.z += g.z; db4.w += g.w;
                } else {
                    g = zero4();
                }
                float4 h, l;
                split_fast(g.x, h.x, l.x); split_fast(g.y, h.y, l.y); split_fast(g.z, h.z, l.z); split_fast(g.w, h.w, l.w);
                const uint32_t ok = tile_off(r, c_m, 128), om = tile_off_mn(r, c_m, 128);
                sts128(sGk + ok, h); sts128(sGk + C::G_BYTES + ok, l);
                sts128(sGm + om, h); sts128(sGm + C::G_BYTES + om, l);
            }
            // ---- X' = act(bn_in(X)) as the GEMM saw it -> MN-major, hi and lo
#pragma unroll
            for (int i = 0; i < NPk; ++i) {
                const int r = r_k + RPk * i;
                float4 v = zero4();
                if (r < valid && colk_ok) {
                    v = a.x_direct ? load_chunk(a.X, row0 + r, a.K, c_k, false) : lds128s(slab + static_cast<uint32_t>(r) * rpitch + c_k * 16);
                    if (has_bn_in) v = bn_apply(v, bi);
                    v.x = act_f(v.x, in_act, in_slope); v.y = act_f(v.y, in_act, in_slope);
                    v.z = act_f(v.z, in_act, in_slope); v.w = act_f(v.w, in_act, in_slope);
                }
                store_split_fast(sX + tile_off_mn(r, c_k, 128), C::X_BYTES, v);
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) { mbar_arrive(a_full); mbar_arrive(raw_empty(s)); }
            // the first passes of the NEXT tile, issued only now: the proxy fence above is a full memory barrier and would
            // wait for them (one HBM round trip per tile, measured); they fly while this warp waits for the MMAs, and the
            // producer has pulled their slabs into L2 a tile earlier
#pragma unroll
            for (int i = 0; i < PF; ++i) issue(j + 1, i, gw[i], yw[i]);
        }
        if (ct == 0) TL_DONE(2);
        // db: lanes sharing a chunk (fixed butterfly), then the converter warps through shared memory
        chunk_allreduce<CHm>(db4);
        if (lane < (CHm < 32 ? CHm : 32)) {
            float *p = &red_db[w - C::W_CONV0][4 * c_m];
            p[0] = db4.x; p[1] = db4.y; p[2] = db4.z; p[3] = db4.w;
        }
        asm volatile("bar.sync 4, %0;" ::"n"(NCV * 32) : "memory");   // ids 1, 2: epilogue groups, 3: both groups
        if (ct < MP) {
            float sum = 0.f;
#pragma unroll
            for (int ww = 0; ww < NCV; ++ww) sum += red_db[ww][ct];
            part[MP * KP + ct] = sum;
        }
    } else {
        // ---------------------------------------------------------------- epilogue warps 0..3 (TMEM lane quadrant = w)
        constexpr int CHk = KP / 4, RPe = 128 / CHk, NPe = 128 / RPe;
        const int eg = w >> 2, wq = w & 3, tg = t & 127;   // epilogue group (tiles j = eg, eg + NEPI, ...), lane quadrant, thread in group
        const int c_k = tg % CHk, r_k = tg / CHk;
        const uint32_t sSt = sStage + eg * C::STAGE_BYTES, sAw = sAccW + eg * C::ACCW_BYTES;
        const bool colk_ok = 4 * c_k < a.K;
        const Bn4 bi = load_bn4(a.in_bn, a.K, c_k);
        const int in_act = a.in_act;
        const float in_slope = a.in_slope;
        const uint32_t pitch = static_cast<uint32_t>(a.K) * 4u;
        float4 sp1 = zero4(), sp2 = zero4();
        TL_DECL;
        for (int j = eg; j < my_tiles; j += C::NEPI) {
            const int ab = j & 1, ua = j >> 1, s = j % RING;
            const int64_t row0 = tile_row0(j);
            const int valid = static_cast<int>((a.N - row0) < 128 ? (a.N - row0) : 128);
            TL_WAIT(0, mbar_wait(acc_full(ab), ua & 1));
            tc_fence_after();
            [[maybe_unused]] const long long tl_p0 = clock64();
            const uint32_t tacc = tmem + ab * C::ACC_COLS + (static_cast<uint32_t>(wq * 32) << 16);
            // ---- this tile's weight-gradient blocks += the CTA's shared-memory copy.  Accumulator row = lane: rows
            // [0, MP) are gY_hi^T [X'_hi | X'_lo], rows [MP, 2 MP) gY_lo^T [X'_hi | (X'_lo: 2^-22, dropped)]
            if (wq * 32 < 2 * MP) {
                const bool lo_row = tg >= MP;
#pragma unroll
                for (int cb = 0; cb < C::PK; ++cb) {
                    float v[32];
                    tc_ld32_nowait(tacc + 2 * KP + cb * 32, v);
                    if (!lo_row) {
                        float u[32];
                        tc_ld32_nowait(tacc + 2 * KP + KP + cb * 32, u);
                        tc_wait_ld();
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] += u[i];
                    } else {
                        tc_wait_ld();
                    }
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const uint32_t slot = sAw + static_cast<uint32_t>(((cb * 8 + q) * 2 * MP + tg) * 16);
                        const float4 p = lds128s(slot);
                        sts128(slot, make_float4(p.x + v[4 * q], p.y + v[4 * q + 1], p.z + v[4 * q + 2], p.w + v[4 * q + 3]));
                    }
                }
            }
            if (!want_gx) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { mbar_arrive(acc_empty(ab)); mbar_arrive(raw_empty(s)); }
                continue;
            }
            if (tg == 0) bulk_wait_read0();
            named_bar_sync<128>(1 + eg);
#pragma unroll
            for (int cb = 0; cb < C::PK; ++cb) {
                float v[32];
                tc_ld_sum2<2>(tacc + cb * 32, KP, v);
                if (cb == C::PK - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty(ab));
                }
                lane_rotate_chunks(v, lane);
#pragma unroll
                for (int p = 0; p < 8; ++p) {
                    const int chunk = cb * 8 + (p ^ (lane & 7));
                    if (4 * chunk < a.K)
                        sts128(sSt + static_cast<uint32_t>(tg) * pitch + chunk * 16, make_float4(v[4 * p], v[4 * p + 1], v[4 * p + 2], v[4 * p + 3]));
                }
            }
            if (need_mask) {
                // ---- activation mask of the previous stage + its BatchNorm-backward sums, in place on the staged tile
                named_bar_sync<128>(1 + eg);
                const uint32_t slab = sRaw + s * C::RAW_SLOT;
                if (colk_ok) {
#pragma unroll 4
                    for (int i = 0; i < NPe; ++i) {
                        const int r = r_k + RPe * i;
                        if (r < valid) {
                            const uint32_t ga = sSt + static_cast<uint32_t>(r) * pitch + c_k * 16;
                            float4 g = lds128s(ga);
                            const float4 x = lds128s(slab + static_cast<uint32_t>(r) * pitch + c_k * 16);
                            if (has_bn_in) {
                                const float4 xc = make_float4(x.x - bi.mean.x, x.y - bi.mean.y, x.z - bi.mean.z, x.w - bi.mean.w);
                                g.x *= dact_f(fmaf(xc.x, bi.k.x, bi.beta.x), in_act, in_slope);
                                g.y *= dact_f(fmaf(xc.y, bi.k.y, bi.beta.y), in_act, in_slope);
                                g.z *= dact_f(fmaf(xc.z, bi.k.z, bi.beta.z), in_act, in_slope);
                                g.w *= dact_f(fmaf(xc.w, bi.k.w, bi.beta.w), in_act, in_slope);
                                sp1.x += g.x; sp1.y += g.y; sp1.z += g.z; sp1.w += g.w;
                                sp2.x = fmaf(g.x, xc.x * bi.rstd.x, sp2.x); sp2.y = fmaf(g.y, xc.y * bi.rstd.y, sp2.y);
                                sp2.z = fmaf(g.z, xc.z * bi.rstd.z, sp2.z); sp2.w = fmaf(g.w, xc.w * bi.rstd.w, sp2.w);
                            } else {
                                g.x *= dact_f(x.x, in_act, in_slope); g.y *= dact_f(x.y, in_act, in_slope);
                                g.z *= dact_f(x.z, in_act, in_slope); g.w *= dact_f(x.w, in_act, in_slope);
                            }
                            sts128(ga, g);
                        }
                    }
                }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(raw_empty(s));
            named_bar_sync<128>(1 + eg);
#ifdef DN4GL_PIPE_TL
            tl_w[1] += clock64() - tl_p0;
#endif
            if (tg == 0) {
                bulk_s2g(a.GX + row0 * a.K, sSt, static_cast<uint32_t>(valid) * pitch);
                bulk_commit();
            }
        }
        if (tg == 0) bulk_wait_all0();
        if (t == 0) TL_DONE(3);
        // previous-stage sums: lanes sharing a chunk, then the 4 warps
        chunk_allreduce<CHk>(sp1);
        chunk_allreduce<CHk>(sp2);
        if (lane < (CHk < 32 ? CHk : 32)) {
            float *p = &red_sp[w][4 * c_k];
            p[0] = sp1.x; p[1] = sp1.y; p[2] = sp1.z; p[3] = sp1.w;
            p[KP] = sp2.x; p[KP + 1] = sp2.y; p[KP + 2] = sp2.z; p[KP + 3] = sp2.w;
        }
        asm volatile("bar.sync 3, %0;" ::"n"(128 * C::NEPI) : "memory");
        for (int i = t; i < 2 * KP; i += 128 * C::NEPI) {
            float sum = 0.f;
#pragma unroll
            for (int ww = 0; ww < 4 * C::NEPI; ++ww) sum += red_sp[ww][i];
            part[MP * KP + MP + i] = sum;
        }
        // the CTA's weight gradient: dW[m][k] = sum over the epilogue groups of (hi row m: hh + hl) + (lo row MP + m: lh)
        for (int e = t; e < MP * (KP / 4); e += 128 * C::NEPI) {
            const int m = e % MP, q = e / MP;
            float4 acc = zero4();
#pragma unroll
            for (int g = 0; g < C::NEPI; ++g) {
                const float4 hi = lds128s(sAccW + g * C::ACCW_BYTES + static_cast<uint32_t>((q * 2 * MP + m) * 16));
                const float4 lo = lds128s(sAccW + g * C::ACCW_BYTES + static_cast<uint32_t>((q * 2 * MP + MP + m) * 16));
                acc.x += hi.x + lo.x; acc.y += hi.y + lo.y; acc.z += hi.z + lo.z; acc.w += hi.w + lo.w;
            }
            *reinterpret_cast<float4 *>(part + m * KP + 4 * q) = acc;
        }
    }
    // ---- teardown + merge of the per-CTA partials {dW, db, sums}: grid rendezvous, then CTA b merges entries
    // [b per, (b + 1) per) -- a warp per entry, lane l adds partials l, l + 32, ... in that order (double), then a fixed
    // butterfly over the lanes; small grids (<= 16 CTAs): a thread per entry, partials in CTA order
    tc_fence_before();
    __syncthreads();
    TL_SPAN(2);
    if (w == C::W_MMA) tc_dealloc(tmem, C::TCOLS);
    constexpr int P = bwd_pipe_part_floats(KP, MP);
    const int G = static_cast<int>(gridDim.x);
    const int per = (P + G - 1) / G, e_begin = static_cast<int>(blockIdx.x) * per, e_end = (e_begin + per < P) ? e_begin + per : P;
    const bool merger = e_begin < P;
    const int passed = grid_arrive(counters, counters + 1, G, merger);
    if (!merger) { TL_SPAN(3); return; }
    const float *pbase = reinterpret_cast<const float *>(a.part);
    auto emit = [&](int e, float r) {
        if (e < MP * KP) {
            const int m = e / KP, kk = e % KP;
            if (dW != nullptr && m < a.M && kk < a.K) dW[m * a.K + kk] = r;
        } else if (e < MP * KP + MP) {
            const int m = e - MP * KP;
            if (db != nullptr && m < a.M) db[m] = r;
        } else {
            const int i2 = e - MP * KP - MP, which = i2 / KP, kk = i2 % KP;
            if (sums_prev != nullptr && kk < a.K) sums_prev[which * a.K + kk] = r;
        }
    };
    if (G > 16) {
        const int lane_ = t & 31;
        for (int e = e_begin + w; e < e_end; e += C::NT / 32) {
            double acc = 0.0;
            constexpr int UNR = 5;
            for (int q0 = 0; q0 < G; q0 += 32 * UNR) {
                float v[UNR];
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const int q = q0 + lane_ + 32 * u;
                    v[u] = (q < G) ? __ldcg(pbase + static_cast<size_t>(q) * P + e) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < UNR; ++u) acc += static_cast<double>(v[u]);
            }
            acc = warp_sum_f64(acc);
            if (lane_ == 0) emit(e, static_cast<float>(acc));
        }
    } else {
        for (int e = e_begin + t; e < e_end; e += C::NT) {
            float v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = (u < G) ? __ldcg(pbase + static_cast<size_t>(u) * P + e) : 0.f;
            double acc = 0.0;
#pragma unroll
            for (int u = 0; u < 16; ++u) acc += static_cast<double>(v[u]);
            emit(e, static_cast<float>(acc));
        }
    }
    grid_depart(counters, counters + 1, passed, (P + per - 1) / per);
    TL_SPAN(3);
}

template <int KP, int MP, int RING, int NCV, int NEPI_>
int launch_bwd_pipe(const LinBwdArgs &a, float *dW, float *db, float *sums_prev, float *gpart, int *counters, cudaStream_t s) {
    using C = BwdCfg<KP, MP, RING, NCV, NEPI_>;
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(lin_bwd_pipe_kernel<KP, MP, RING, NCV, NEPI_>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(C::SMEM)) != cudaSuccess)
            return -1;
        attr_done = true;
    }
    const int sms = dn4gl_num_sms();
    const int grid = a.num_tiles < sms ? a.num_tiles : sms;
    if (launch_coop(lin_bwd_pipe_kernel<KP, MP, RING, NCV, NEPI_>, grid, C::NT, C::SMEM, s, a, dW, db, sums_prev, gpart, counters) != cudaSuccess)
        return -1;
    return grid;
}

}  // namespace

#ifdef DN4GL_PIPE_TL
extern "C" int dn4gl_debug_read_pipe_timeline(long long *host_out) {
    return cudaMemcpyFromSymbol(host_out, g_pipe_tl, sizeof(long long) * 148 * 16) == cudaSuccess ? 0 : -2;
}
extern "C" int dn4gl_debug_read_pipe_span(unsigned long long *host_out) {
    return cudaMemcpyFromSymbol(host_out, g_pipe_span, sizeof(unsigned long long) * 148 * 4) == cudaSuccess ? 0 : -2;
}
#endif

// -> number of CTAs launched (> 0), 0 if this shape has no pipelined instantiation, -1 on a CUDA error.
// Preconditions (checked by the caller): K % 4 == 0, M % 4 == 0, X / Y / W 16-byte aligned, counter zero on entry.
int dn4gl_pipe_lin_fwd(const LinFwdArgs &a, const BnFinalArgs &f, int *counter, cudaStream_t s) {
    const int KP = a.K <= 32 ? 32 : 64, MP = a.M <= 32 ? 32 : 64;
    if (a.K > 64 || a.M > 64) return 0;
    //                                                  KP  MP NACC NBUF_A RING NCV NEPI NACCBUF
    if (KP == 32 && MP == 32) return launch_fwd_pipe<32, 32, 1, 2, 4, 8, 2, 2>(a, f, counter, s);
    if (KP == 32 && MP == 64) return launch_fwd_pipe<32, 64, 1, 2, 4, 8, 2, 2>(a, f, counter, s);
    // K = 64: 8 k-steps.  Four accumulators of two A_hi k-steps each (one accumulator set, 512 tensor-memory columns at
    // M = 64): the truncation bias of the accumulation is what the counting models' 1e-5 bar is sensitive to (DESIGN.md)
    if (KP == 64 && MP == 32) return launch_fwd_pipe<64, 32, 4, 1, 3, 8, 2, 2>(a, f, counter, s);
    return launch_fwd_pipe<64, 64, 4, 1, 2, 8, 1, 1>(a, f, counter, s);
}

// workspace of the pipelined backward: per-CTA partials (floats), then the group partials (doubles)
size_t dn4gl_pipe_lin_bwd_ws_bytes(int K, int M) {
    const int KP = K <= 32 ? 32 : 64, MP = M <= 32 ? 32 : 64;
    const size_t P = static_cast<size_t>(bwd_pipe_part_floats(KP, MP));
    const size_t ctas = static_cast<size_t>(dn4gl_num_sms());
    return align_up(ctas * P * sizeof(float), 256) + align_up(((ctas + BWD_GROUP - 1) / BWD_GROUP) * P * sizeof(float), 256);
}
// -> CTAs launched (> 0), 0 if the shape has no pipelined instantiation, -1 on a CUDA error.  Preconditions (caller):
// K % 4 == 0, M % 4 == 0, all matrices 16-byte aligned, counters zero on entry (left zero), ws >= the size above.
int dn4gl_pipe_lin_bwd(LinBwdArgs a, float *dW, float *db, float *sums_prev, void *ws, int *counters, cudaStream_t s) {
    if (a.K > 64 || a.M > 64) return 0;
    if (a.x_direct && a.GX != nullptr) return 0;      // the mask pass of the data gradient reads the staged X slab
    const int KP = a.K <= 32 ? 32 : 64, MP = a.M <= 32 ? 32 : 64;
    if (KP == 64 || MP == 64) return 0;          // 64-wide shapes: operand tiles alone exceed one CTA's shared memory (mlp_tc.cu path)
    const size_t P = static_cast<size_t>(bwd_pipe_part_floats(KP, MP));
    a.part = static_cast<float *>(ws);
    float *gpart = reinterpret_cast<float *>(static_cast<char *>(ws) + align_up(static_cast<size_t>(dn4gl_num_sms()) * P * sizeof(float), 256));
    return launch_bwd_pipe<32, 32, 3, 8, 1>(a, dW, db, sums_prev, gpart, counters, s);
}
