// libdn4gl.so -- general fp32 GEMM on the tensor cores:  C (N x M) = A (N x K) B (+ bias),  B given as the nn.Linear
// weight (M x K: y = x W^T, rgin.py:52 / dmpnn.py:47 style layers, the data gradient of `x @ w`) or as a (K x M) matrix
// (`x @ w`: the relation / loop / P|Q / T products of rgin.py:137-154, dmpnn.py:111-156, rgconv.py:48-51, and the data
// gradient of nn.Linear).  N is tall (nodes / edges), K and M are 1 .. ~1200.
//
// These products used to run as library SIMT SGEMMs (25-35 % of a C3 / C4 step, profiles/r3t_*): fp32 on the FMA pipe
// is what "within 1e-5" needs from a library, and a single-pass TF32 GEMM is 1e-3.  Here: 3xTF32 on tcgen05 -- every
// operand is split x = hi + lo (both exactly representable in tf32), the products hi*hi + hi*lo + lo*hi are formed by
// the tensor core, and ALL additions across the contraction index beyond one 32-wide chunk are done in fp32 registers
// with round-to-nearest: the tensor core truncates after each accumulation (a biased error that grows with the number of
// MMAs added into one accumulator, DESIGN.md section 4 K6), so an accumulator only ever holds the products of ONE chunk
// (lo products first), is drained by the epilogue warps and starts fresh.
//
// Structure (one persistent CTA per SM, warp-specialised, as csrc/mlp_pipe.cu):
//   prep kernel     B -> per (column tile, k-chunk) a block [B_hi ; B_lo] of 2 MT rows x 32 k, already in the 128-byte
//                   swizzled K-major layout the MMA reads: the main kernel moves it with ONE bulk copy per chunk
//   producer warp   cp.async.bulk of the B blocks into the stage ring; L2 prefetch of the A rows a few chunks ahead
//   4 loader warps      A chunk (128 rows x 32 k) global -> raw ring in shared memory by 16-byte cp.async (5 chunks in flight)
//   4 converter warps   raw chunk -> hi / lo -> swizzled operand tiles, fence.proxy.async
//   MMA warp        per chunk 4 k-steps x {A_lo B_hi, A_hi B_lo, A_hi B_hi} into one of two tensor-memory accumulators
//   epilogue warps  tcgen05.ld of the chunk's accumulator, += into up to 64 fp32 registers per thread; after
//                   the last chunk: bias, store.  MT = 128: two epilogue groups of 64 columns each.
#include "tc_common.cuh"

#ifdef DN4GL_GEMM_TL
// debug build (make libdn4gl_exp.so EXP_FLAGS=-DDN4GL_GEMM_TL, tools/gemm_timeline.py): per role the cycles of its chunk loop and
// the cycles blocked in each of its waits, for the first 148 CTAs of the last launch
__device__ long long g_gemm_tl[148 * 5 * 4];
#define GTL_DECL long long gtl_t0 = clock64(), gtl_w[3] = {0, 0, 0}
#define GTL_WAIT(k, stmt) do { const long long c0__ = clock64(); stmt; gtl_w[k] += clock64() - c0__; } while (0)
#define GTL_DONE(role) do { if (blockIdx.x < 148) { long long *p__ = g_gemm_tl + (blockIdx.x * 5 + (role)) * 4; \
    p__[0] = clock64() - gtl_t0; p__[1] = gtl_w[0]; p__[2] = gtl_w[1]; p__[3] = gtl_w[2]; } } while (0)
#else
#define GTL_DECL do { } while (0)
#define GTL_WAIT(k, stmt) stmt
#define GTL_DONE(role) do { } while (0)
#endif

namespace {

struct GemmArgs {
    const float *A;        // N x K, leading dimension lda
    int64_t N;
    int K, lda;
    const float *Bp;       // prepared blocks, see prep kernel
    const float *bias;     // M or NULL
    float *C;              // N x M, leading dimension ldc
    int M, ldc;
    int row_tiles, col_tiles, kchunks;
};

__device__ __forceinline__ void split_rn(float x, float &hi, float &lo) {      // as mlp_pipe.cu split_fast
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
    lo = x - hi;
}
__device__ __forceinline__ void mbar_arrive_g(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// ---- B -> [hi ; lo] blocks.  layout 0: B is (M x K) row-major (ldb >= K);  layout 1: B is (K x M) row-major (ldb >= M).
// block (ct, kc) at Bp + (ct * kchunks + kc) * MT * 64 floats; row r < MT: hi of column ct * MT + r, row MT + r: its lo;
// 16-byte chunk c of a row (k = kc * 32 + 4 c ..) at byte  r * 128 + ((c ^ (r & 7)) << 4)
template <int MT>
__global__ void __launch_bounds__(256) gemm3x_prep_kernel(const float *__restrict__ B, int ldb, int layout, int K, int M, int kchunks,
                                                          float *__restrict__ Bp) {
    const int kc = blockIdx.x, ct = blockIdx.y;
    char *blk = reinterpret_cast<char *>(Bp) + (static_cast<size_t>(ct) * kchunks + kc) * MT * 256;
    for (int idx = threadIdx.x; idx < MT * 8; idx += 256) {
        // layout 1 reads are contiguous in m: let consecutive threads take consecutive m
        const int m = layout == 0 ? idx >> 3 : idx % MT, c = layout == 0 ? idx & 7 : idx / MT;
        const int col = ct * MT + m, k0 = kc * 32 + 4 * c;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + j;
            v[j] = (col < M && k < K) ? (layout == 0 ? __ldg(B + static_cast<size_t>(col) * ldb + k) : __ldg(B + static_cast<size_t>(k) * ldb + col)) : 0.f;
        }
        float4 h, l;
        split_rn(v[0], h.x, l.x); split_rn(v[1], h.y, l.y); split_rn(v[2], h.z, l.z); split_rn(v[3], h.w, l.w);
        *reinterpret_cast<float4 *>(blk + m * 128 + ((c ^ (m & 7)) << 4)) = h;
        const int r = MT + m;
        *reinterpret_cast<float4 *>(blk + r * 128 + ((c ^ (r & 7)) << 4)) = l;
    }
}

template <int MT>
struct GemmCfg {
    static constexpr int NCV = 4;
    static constexpr int NEG = MT == 128 ? 2 : 1;               // epilogue groups (64 output columns each at MT = 128)
    static constexpr int NWE = 4 * NEG;
    static constexpr int NLD = 4;                                // loader warps: global A -> registers -> raw ring
    static constexpr int W_CONV0 = NWE, W_LOAD0 = NWE + NCV, W_PROD = NWE + NCV + NLD, W_MMA = NWE + NCV + NLD + 1;
    static constexpr int NT = (NWE + NCV + NLD + 2) * 32;
    static constexpr int STAGES = MT == 128 ? 2 : 3;             // ring of {A_hi, A_lo, [B_hi ; B_lo]}
    static constexpr int RS = 5;                                 // raw ring: A chunks as they lie in memory (16 KB each)
    static constexpr uint32_t A_BYTES = 128u * 128u;             // one of A_hi / A_lo: 128 rows x 32 floats
    static constexpr uint32_t B_BYTES = MT * 256u;               // [B_hi ; B_lo]: 2 MT rows x 32 floats
    static constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + B_BYTES;
    static constexpr int ACC_COLS = MT < 32 ? 32 : MT;           // one accumulator: all three products of a chunk
    static constexpr int TCOLS = 2 * ACC_COLS;                   // two accumulator buffers
    static constexpr int CPT = MT < 64 ? MT : 64;                // output columns per epilogue thread
    static constexpr size_t SMEM = 1024 + static_cast<size_t>(STAGES) * STAGE_BYTES + static_cast<size_t>(RS) * A_BYTES;
};

template <int MT>
__global__ void __launch_bounds__(GemmCfg<MT>::NT, 1) gemm3x_kernel(const GemmArgs a) {
    using C = GemmCfg<MT>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * C::STAGES + 4 + 2 * C::RS];
    __shared__ uint32_t tmem_ptr;
    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    const uint32_t base = (s_u32(smem_raw) + 1023u) & ~1023u;
    auto a_full = [&](int s) { return s_u32(&bars[s]); };
    auto a_empty = [&](int s) { return s_u32(&bars[C::STAGES + s]); };
    auto acc_full = [&](int b) { return s_u32(&bars[2 * C::STAGES + b]); };
    auto acc_empty = [&](int b) { return s_u32(&bars[2 * C::STAGES + 2 + b]); };
    auto raw_full = [&](int r) { return s_u32(&bars[2 * C::STAGES + 4 + r]); };
    auto raw_empty = [&](int r) { return s_u32(&bars[2 * C::STAGES + 4 + C::RS + r]); };
    const uint32_t sRaw = base + C::STAGES * C::STAGE_BYTES;
    if (t == 0) {
        for (int r = 0; r < C::RS; ++r) {
            mbar_init(raw_full(r), C::NLD * 32);     // every loader thread (its copies' completion, or its own stores)
            mbar_init(raw_empty(r), C::NCV);         // converter warps
        }
        for (int s = 0; s < C::STAGES; ++s) {
            mbar_init(a_full(s), C::NCV + 1);        // converter warps + the producer's expect_tx arrival
            mbar_init(a_empty(s), 1);                // tcgen05.commit
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full(b), 1);
            mbar_init(acc_empty(b), C::NWE);
        }
        fence_barrier_init();
    }
    if (w == C::W_MMA) tc_alloc(s_u32(&tmem_ptr), C::TCOLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_ptr;
    const int total_tiles = a.row_tiles * a.col_tiles;
    const int KC = a.kchunks;
    // this CTA's chunk sequence: chunk j of the CTA is k-chunk j % KC of its (j / KC)-th tile
    auto chunk_at = [&](int j, int64_t &row0, int &kc) -> bool {
        const int tile = static_cast<int>(blockIdx.x) + (j / KC) * static_cast<int>(gridDim.x);
        if (tile >= total_tiles) return false;
        row0 = static_cast<int64_t>(tile / a.col_tiles) * 128;
        kc = j % KC;
        return true;
    };

    if (w == C::W_PROD) {
        // ------------------------------------------------------------ producer: B blocks (lane 0) + L2 prefetch of A
        // A is loaded by the loader warps (row pieces of 128 bytes are too small for bulk copies: 128 of them per chunk
        // took 4 us, profiles/r4f_bench_gemm.txt).  The 32 lanes of this warp pull the A rows of the chunk PF steps ahead
        // into L2 (one line per row and chunk, 4 per lane), paced by the same "stage free" barrier as everything else, so
        // those loads hit L2.
        constexpr int PF = C::STAGES + 2;
        auto prefetch_chunk = [&](int j) {
            int64_t row0;
            int kc;
            if (!chunk_at(j, row0, kc) || kc * 32 >= a.K) return;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int64_t row = row0 + lane + 32 * i;
                if (row < a.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.A + row * a.lda + kc * 32));
            }
        };
        for (int j = 0; j < PF; ++j) prefetch_chunk(j);
        int q = 0;
        GTL_DECL;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int ct = tile % a.col_tiles;
            const char *src = reinterpret_cast<const char *>(a.Bp) + static_cast<size_t>(ct) * KC * C::B_BYTES;
            for (int kc = 0; kc < KC; ++kc, ++q) {
                const int s = q % C::STAGES, us = q / C::STAGES;
                GTL_WAIT(0, mbar_wait(a_empty(s), (us & 1) ^ 1));
                if (lane == 0) {
                    mbar_expect_tx(a_full(s), C::B_BYTES);
                    bulk_g2s(base + s * C::STAGE_BYTES + 2 * C::A_BYTES, src + static_cast<size_t>(kc) * C::B_BYTES, C::B_BYTES, a_full(s));
                }
                prefetch_chunk(q + PF);
                __syncwarp();
            }
        }
        if (lane == 0) GTL_DONE(0);
    } else if (w == C::W_MMA) {
        // ------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            constexpr uint32_t IDESC = make_idesc(128, MT, 0, 0);
            constexpr uint32_t B_LO = MT * 128u;                 // B_lo rows follow the MT rows of B_hi
            int q = 0;
            GTL_DECL;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                for (int kc = 0; kc < KC; ++kc, ++q) {
                    const int s = q % C::STAGES, us = q / C::STAGES, ab = q & 1, ua = q >> 1;
                    GTL_WAIT(0, mbar_wait(acc_empty(ab), (ua & 1) ^ 1));
                    GTL_WAIT(1, mbar_wait(a_full(s), us & 1));
                    tc_fence_after();
                    const uint32_t sAh = base + s * C::STAGE_BYTES, sAl = sAh + C::A_BYTES, sB = sAh + 2 * C::A_BYTES;
                    const uint32_t d = tmem + ab * C::ACC_COLS;
                    // the small products first (2^-11 of the result: the tensor core's truncation there is harmless), all
                    // three into ONE accumulator: the epilogue's drain is bound by the tensor-memory read rate (64 B / clock),
                    // so separate hh | hl halves (one N = 2 MT instruction instead of two) cost more than they saved
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        tc_mma_tf32(d, make_desc(sAl + ks * 32u, 16, 1024), make_desc(sB + ks * 32u, 16, 1024), IDESC, ks != 0 ? 1u : 0u);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        tc_mma_tf32(d, make_desc(sAh + ks * 32u, 16, 1024), make_desc(sB + B_LO + ks * 32u, 16, 1024), IDESC, 1u);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        tc_mma_tf32(d, make_desc(sAh + ks * 32u, 16, 1024), make_desc(sB + ks * 32u, 16, 1024), IDESC, 1u);
                    tc_commit(a_empty(s));
                    tc_commit(acc_full(ab));
                }
            }
            GTL_DONE(1);
        }
    } else if (w >= C::W_LOAD0 && w < C::W_PROD) {
        // ------------------------------------------------------------ loaders: A chunk global -> registers -> raw ring
        // Separate from the converters on purpose: a converter must execute fence.proxy.async after its shared stores, which
        // compiles to MEMBAR.ALL.CTA and waits for EVERY outstanding load of the thread -- with the loads in the converter
        // threads (first versions) each chunk cost one memory round trip (1.6 us per chunk however deep the register
        // prefetch).  These warps never fence: two chunks of loads stay in flight per thread.
        const int lt = t - C::W_LOAD0 * 32, c_in = lt & 7, r_in = lt >> 3;         // 16 rows per pass, 8 passes
        const bool vec = (a.lda % 4 == 0) && aligned16_dev(a.A);
        auto load = [&](int j, float4 (&v)[8]) {
            int64_t row0;
            int kc;
            if (!chunk_at(j, row0, kc)) return;
            const int k0 = kc * 32 + 4 * c_in;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int64_t row = row0 + r_in + 16 * i;
                v[i] = zero4();
                if (row < a.N && k0 < a.K) {
                    const float *p = a.A + row * a.lda + k0;
                    if (vec && k0 + 3 < a.K) {
                        v[i] = __ldg(reinterpret_cast<const float4 *>(p));
                    } else {
                        v[i].x = __ldg(p);
                        if (k0 + 1 < a.K) v[i].y = __ldg(p + 1);
                        if (k0 + 2 < a.K) v[i].z = __ldg(p + 2);
                        if (k0 + 3 < a.K) v[i].w = __ldg(p + 3);
                    }
                }
            }
        };
        int q = 0;
        GTL_DECL;
        if (vec && a.K % 4 == 0) {
            // 16-byte asynchronous copies (cp.async, global -> shared without registers): a thread issues its 8 pieces of a
            // chunk and moves on; the copies signal the slot's barrier when they land.  RS chunks (80 KB) are in flight per
            // SM -- with register staging it was two (32 KB), and the kernel ran at latency x concurrency = 2.7 TB/s
            // (profiles/r4i_gemm_timeline.txt: loader 97 % busy, converters waiting for it 45-70 % of the time).
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int64_t row0 = static_cast<int64_t>(tile / a.col_tiles) * 128;
                for (int kc = 0; kc < KC; ++kc, ++q) {
                    const int rs = q % C::RS, ur = q / C::RS;
                    GTL_WAIT(0, mbar_wait(raw_empty(rs), (ur & 1) ^ 1));
                    const uint32_t dst = sRaw + rs * C::A_BYTES + static_cast<uint32_t>(r_in) * 128u + c_in * 16u;
                    const int k0 = kc * 32 + 4 * c_in;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int64_t row = row0 + r_in + 16 * i;
                        const bool ok = row < a.N && k0 < a.K;
                        const float *src = ok ? a.A + row * a.lda + k0 : a.A;
                        const uint32_t nbytes = ok ? 16u : 0u;           // fewer source bytes than 16: the rest is zero-filled
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + static_cast<uint32_t>(i) * 2048u), "l"(src), "r"(nbytes) : "memory");
                    }
                    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(raw_full(rs)) : "memory");
                }
            }
        } else {
            float4 b0[8], b1[8];             // unaligned A: chunks q, q + 1 through registers
            load(0, b0);
            load(1, b1);
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                for (int kc = 0; kc < KC; ++kc, ++q) {
                    const int rs = q % C::RS, ur = q / C::RS;
                    GTL_WAIT(0, mbar_wait(raw_empty(rs), (ur & 1) ^ 1));
                    const uint32_t dst = sRaw + rs * C::A_BYTES + static_cast<uint32_t>(r_in) * 128u + c_in * 16u;
#pragma unroll
                    for (int i = 0; i < 8; ++i) sts128(dst + static_cast<uint32_t>(i) * 2048u, b0[i]);
                    mbar_arrive_g(raw_full(rs));
#pragma unroll
                    for (int i = 0; i < 8; ++i) b0[i] = b1[i];
                    load(q + 2, b1);
                }
            }
        }
        if (lt == 0) GTL_DONE(3);
    } else if (w >= C::W_CONV0 && w < C::W_LOAD0) {
        // ------------------------------------------------------------ converters: raw A chunk -> hi / lo swizzled tiles
        const int ct_ = t - C::W_CONV0 * 32, c_in = ct_ & 7, r_in = ct_ >> 3;
        int q = 0;
        GTL_DECL;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            for (int kc = 0; kc < KC; ++kc, ++q) {
                const int s = q % C::STAGES, us = q / C::STAGES, rs = q % C::RS, ur = q / C::RS;
                GTL_WAIT(0, mbar_wait(raw_full(rs), ur & 1));
                const uint32_t src = sRaw + rs * C::A_BYTES + static_cast<uint32_t>(r_in) * 128u + c_in * 16u;
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = lds128s(src + static_cast<uint32_t>(i) * 2048u);
                __syncwarp();
                if (lane == 0) mbar_arrive_g(raw_empty(rs));
                GTL_WAIT(1, mbar_wait(a_empty(s), (us & 1) ^ 1));
                const uint32_t sAh = base + s * C::STAGE_BYTES;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = r_in + 16 * i;
                    float4 h, l;
                    split_rn(v[i].x, h.x, l.x); split_rn(v[i].y, h.y, l.y); split_rn(v[i].z, h.z, l.z); split_rn(v[i].w, h.w, l.w);
                    const uint32_t off = static_cast<uint32_t>(r) * 128u + static_cast<uint32_t>((c_in ^ (r & 7)) << 4);
                    sts128(sAh + off, h);
                    sts128(sAh + C::A_BYTES + off, l);
                }
                GTL_WAIT(2, fence_async_smem());
                __syncwarp();
                if (lane == 0) mbar_arrive_g(a_full(s));
            }
        }
        if (ct_ == 0) GTL_DONE(2);
    } else {
        // ------------------------------------------------------------ epilogue: drain every chunk into registers, store at the end
        const int eg = w >> 2, wq = w & 3;                       // column group, TMEM lane quadrant
        const int col_e = eg * 64;                               // first output column of this group inside the tile
        const bool vec = (a.ldc % 4 == 0) && aligned16_dev(a.C);
        int q = 0;
        GTL_DECL;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            float acc[C::CPT];
#pragma unroll
            for (int i = 0; i < C::CPT; ++i) acc[i] = 0.f;
            for (int kc = 0; kc < KC; ++kc, ++q) {
                const int ab = q & 1, ua = q >> 1;
                GTL_WAIT(0, mbar_wait(acc_full(ab), ua & 1));
                tc_fence_after();
                [[maybe_unused]] const long long gtl_e0 = clock64();
                const uint32_t tacc = tmem + ab * C::ACC_COLS + (static_cast<uint32_t>(wq * 32) << 16);
                if constexpr (MT == 16) {
                    float v[32];                                 // the buffer is 32 columns wide, 16 are written
                    tc_ld32(tacc, v);
                    tc_wait_ld();
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[i] += v[i];
                } else {
#pragma unroll
                    for (int cb = 0; cb < C::CPT / 32; ++cb) {
                        float v[32];
                        tc_ld32(tacc + col_e + cb * 32, v);
                        tc_wait_ld();
#pragma unroll
                        for (int i = 0; i < 32; ++i) acc[cb * 32 + i] += v[i];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_g(acc_empty(ab));
#ifdef DN4GL_GEMM_TL
                gtl_w[1] += clock64() - gtl_e0;
#endif
            }
            [[maybe_unused]] const long long gtl_s0 = clock64();
            const int64_t row = static_cast<int64_t>(tile / a.col_tiles) * 128 + wq * 32 + lane;
            const int col0 = (tile % a.col_tiles) * MT + col_e;
            if (row < a.N) {
                float *dst = a.C + row * a.ldc + col0;
#pragma unroll
                for (int i = 0; i < C::CPT; i += 4) {
                    const int col = col0 + i;
                    if (col >= a.M) break;
                    float4 o = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
                    if (a.bias != nullptr) {
                        o.x += __ldg(a.bias + col);
                        if (col + 1 < a.M) o.y += __ldg(a.bias + col + 1);
                        if (col + 2 < a.M) o.z += __ldg(a.bias + col + 2);
                        if (col + 3 < a.M) o.w += __ldg(a.bias + col + 3);
                    }
                    if (vec && col + 3 < a.M) {
                        *reinterpret_cast<float4 *>(dst + i) = o;
                    } else {
                        dst[i] = o.x;
                        if (col + 1 < a.M) dst[i + 1] = o.y;
                        if (col + 2 < a.M) dst[i + 2] = o.z;
                        if (col + 3 < a.M) dst[i + 3] = o.w;
                    }
                }
            }
#ifdef DN4GL_GEMM_TL
            gtl_w[2] += clock64() - gtl_s0;
#endif
        }
        if (t == 0) GTL_DONE(4);
    }
    tc_fence_before();
    __syncthreads();
    if (w == C::W_MMA) tc_dealloc(tmem, C::TCOLS);
}

static int pick_mt(int M) { return M <= 16 ? 16 : (M <= 32 ? 32 : (M <= 64 ? 64 : 128)); }

template <int MT>
static int launch_gemm(const GemmArgs &a, const float *B, int ldb, int layout, float *Bp, cudaStream_t s) {
    using C = GemmCfg<MT>;
    static bool attr_done = false;
    if (!attr_done) {
        if (cudaFuncSetAttribute(gemm3x_kernel<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(C::SMEM)) != cudaSuccess)
            return -1;
        attr_done = true;
    }
    gemm3x_prep_kernel<MT><<<dim3(a.kchunks, a.col_tiles), 256, 0, s>>>(B, ldb, layout, a.K, a.M, a.kchunks, Bp);
    const int tiles = a.row_tiles * a.col_tiles, sms = dn4gl_num_sms();
    gemm3x_kernel<MT><<<tiles < sms ? tiles : sms, C::NT, C::SMEM, s>>>(a);
    return 0;
}

}  // namespace

extern "C" size_t dn4gl_gemm_workspace_bytes(int32_t K, int32_t M) {
    if (K <= 0 || M <= 0) return 0;
    const int MT = pick_mt(M);
    const size_t col_tiles = (static_cast<size_t>(M) + MT - 1) / MT, kchunks = (static_cast<size_t>(K) + 31) / 32;
    return col_tiles * kchunks * MT * 256;
}

extern "C" int dn4gl_gemm_f32(const float *A, int64_t N, int32_t K, int32_t lda, const float *B, int32_t ldb, int32_t b_layout,
                              int32_t M, const float *bias, float *C, int32_t ldc, void *ws, size_t ws_bytes, void *stream) {
    DN_ARG(N >= 0 && K >= 0 && M >= 0 && (b_layout == 0 || b_layout == 1));
    if (N == 0 || M == 0) return DN4GL_OK;
    DN_ARG(C != nullptr && ldc >= M && N < (1ll << 31) * 64);
    DN_ARG(K == 0 || (A != nullptr && B != nullptr && lda >= K && ldb >= (b_layout == 0 ? K : M)));
    DN_ARG(K == 0 || (ws != nullptr && ws_bytes >= dn4gl_gemm_workspace_bytes(K, M) && aligned16(ws)));
    cudaStream_t s = as_stream(stream);
    const int MT = pick_mt(M);
    GemmArgs a;
    a.A = A; a.N = N; a.K = K; a.lda = lda; a.Bp = static_cast<const float *>(ws); a.bias = bias; a.C = C; a.M = M; a.ldc = ldc;
    a.row_tiles = static_cast<int>((N + 127) / 128);
    a.col_tiles = (M + MT - 1) / MT;
    a.kchunks = K > 0 ? (K + 31) / 32 : 0;
    DN_ARG(K > 0);      // an empty contraction is the caller's bias broadcast, not a GEMM
    int rc;
    switch (MT) {
    case 16: rc = launch_gemm<16>(a, B, ldb, b_layout, static_cast<float *>(ws), s); break;
    case 32: rc = launch_gemm<32>(a, B, ldb, b_layout, static_cast<float *>(ws), s); break;
    case 64: rc = launch_gemm<64>(a, B, ldb, b_layout, static_cast<float *>(ws), s); break;
    default: rc = launch_gemm<128>(a, B, ldb, b_layout, static_cast<float *>(ws), s); break;
    }
    if (rc != 0) { dn4gl_set_error("dn4gl_gemm_f32: shared-memory configuration refused"); return DN4GL_ECUDA; }
    DN_LAUNCHED_N(2);
    return DN4GL_OK;
}

#ifdef DN4GL_GEMM_TL
extern "C" int dn4gl_debug_read_gemm_timeline(long long *host_out) {
    return cudaMemcpyFromSymbol(host_out, g_gemm_tl, sizeof(long long) * 148 * 5 * 4) == cudaSuccess ? 0 : -1;
}
#endif
