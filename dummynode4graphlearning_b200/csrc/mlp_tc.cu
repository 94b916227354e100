// libdn4gl.so -- the dense per-node / per-edge MLP stages on the 5th-generation tensor cores (tcgen05 + TMEM).
//
// The MLPs on the path (gconv.py:190-196 Linear,BN,ReLU,Linear,BN,ReLU; rgin.py:52 / dmpnn.py:47,55 Linear,act,Linear)
// multiply a tall matrix of node / edge rows (1e4..1e7 x D) by a tiny D x D weight: 8..64 flop per byte, i.e. above what
// the fp32 FMA pipe delivers at full HBM rate, far below the tensor pipe.  Each "stage" kernel therefore streams row
// tiles of 128 rows ONCE through shared memory, does the GEMM as 3xTF32 (error-compensated split x = hi + lo, three
// tcgen05.mma.kind::tf32 passes hi*hi + lo*hi + hi*lo accumulated in fp32 in tensor memory; products are exact to
// ~2^-21, see DESIGN.md) and fuses everything elementwise around it:
//
//   dn4gl_lin_fwd_f32   Y = act(bn_in(X)) W^T + b        prologue: BatchNorm-apply + activation of the PREVIOUS stage
//                                                        epilogue: bias, per-channel batch statistics of Y -> the
//                                                        BatchNorm record {mean, rstd, gamma*rstd, beta} (+ running stats)
//   dn4gl_lin_bwd_f32   gX = (gY W) * act'(bn_in(X)),  dW = gY^T act(bn_in(X)),  db = colsum gY
//                                                        prologue: BatchNorm backward of the stage output (gY from the
//                                                        upstream gradient, Y and the two batch sums), epilogue:
//                                                        activation mask + the batch sums the previous stage needs;
//                                                        dW accumulates in tensor memory over all tiles of the CTA.
//
// Operand tiles live in shared memory in the canonical 128-byte-swizzled layout ("panels" of 32 floats x rows, 16-byte
// chunk index XOR (row & 7)); the same physical tile is read K-major (rows = M) by the data GEMM and MN-major
// (rows = K) by the weight-gradient GEMM.  One thread issues the MMAs; completion arrives on an mbarrier through
// tcgen05.commit; accumulators come back with tcgen05.ld (32 lanes x 32 columns per warp) and leave through a staging
// tile so that global stores are 128-bit and coalesced.  All reductions are fixed-order (no float atomics).
#include "common.cuh"
#include "tc_common.cuh"

int dn4gl_pipe_lin_fwd(const LinFwdArgs &a, const BnFinalArgs &f, int *counter, cudaStream_t s);   // mlp_pipe.cu
size_t dn4gl_pipe_lin_bwd_ws_bytes(int K, int M);
int dn4gl_pipe_lin_bwd(LinBwdArgs a, float *dW, float *db, float *sums_prev, void *ws, int *counters, cudaStream_t s);

namespace {


// ------------------------------------------------------------------------------------------------------------------
// forward stage
// ------------------------------------------------------------------------------------------------------------------

// B operand tile: per 32-float K panel the MP hi rows then the MP lo rows, so that ONE MMA with N = 2 MP multiplies
// an A tile with [W_hi | W_lo]; accumulator columns [0, MP) and [MP, 2 MP) are added in the epilogue (all four
// hi/lo products: 2 MMAs per k-step instead of 3, and the lo*lo term comes for free).
template <int KP, int MP, int RING, int NT>
__global__ void __launch_bounds__(NT) lin_fwd_kernel(const LinFwdArgs a) {
    extern __shared__ uint8_t smem_raw[];
    constexpr int PK = KP / 32, PM = MP / 32;
    constexpr uint32_t A_BYTES = PK * PANEL128, B_BYTES = PK * 2 * MP * 128u, RAW_BYTES = 128u * KP * 4u;
    const uint32_t base = (s_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sAh = base, sAl = sAh + A_BYTES, sB = sAl + A_BYTES, sRing = sB + B_BYTES;
    const uint32_t sStage = sAh;      // the operand tiles are dead once the tile's MMAs have completed
    static_assert(2 * PK >= PM, "staging tile must fit the A operand tiles");
    __shared__ __align__(8) uint64_t bar_mem;
    __shared__ __align__(8) uint64_t full_mem[RING > 0 ? RING : 1];
    __shared__ uint32_t tmem_ptr;
    constexpr int NW = NT / 32;
    __shared__ float red[NW][MP * 2];
    __shared__ float shift_s[MP];

    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    const uint32_t bar = s_u32(&bar_mem);
    // The tensor core adds every MMA into the fp32 accumulator with truncation (measured: the error grows linearly with
    // the number of MMAs accumulated, ~2^-24 each: 4e-7 relative at 8 MMAs, 2e-7 when the k-steps are spread over
    // accumulators of 4 MMAs that the epilogue adds in round-to-nearest).  Splitting costs tensor-memory read bandwidth
    // (64 B/clk/SM: +57 % time at 1M x 32 with TC_SPLIT_ACC = 2), so the default is one accumulator.
    constexpr int KSTEPS = KP / 8, NACC = (TC_SPLIT_ACC < KSTEPS / 2 ? TC_SPLIT_ACC : KSTEPS / 2), KPA = KSTEPS / NACC;
    constexpr uint32_t TCOLS = NACC * 2 * MP;
    if (t == 0) {
        mbar_init(bar, 1);
        for (int s = 0; s < RING; ++s) mbar_init(s_u32(&full_mem[s]), 1);
        fence_barrier_init();
    }
    if (w == 0) tc_alloc(s_u32(&tmem_ptr), TCOLS);
    __syncthreads();
    // raw ring: tile j of this CTA lives in slot j % RING
    auto issue = [&](int j) {
        const int64_t tile = static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(j) * gridDim.x;
        if (tile >= a.num_tiles) return;
        const int64_t row0 = tile * 128, left = a.N - row0;
        const uint32_t bytes = static_cast<uint32_t>((left < 128 ? left : 128) * a.K * 4);
        const uint32_t fb = s_u32(&full_mem[j % (RING > 0 ? RING : 1)]);
        mbar_expect_tx(fb, bytes);
        bulk_g2s(sRing + (j % (RING > 0 ? RING : 1)) * RAW_BYTES, a.X + row0 * a.K, bytes, fb);
    };
    if (RING > 0 && t == 0)
        for (int j = 0; j < RING - 1; ++j) issue(j);
    // weights: W (M x K) row-major = K-major B operand; zero-padded to MP x KP, split once
    const bool vecW = (a.K % 4 == 0) && aligned16_dev(a.W);
    for (int i = t; i < MP * (KP / 4); i += NT) {
        const int m = i / (KP / 4), c = i % (KP / 4);
        const float4 v = (m < a.M) ? load_chunk(a.W, m, a.K, c, vecW) : zero4();
        store_split(sB, sB, 0, v, tile_off(m, c, 2 * MP), tile_off(MP + m, c, 2 * MP));
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_ptr;

    constexpr int CH = KP / 4, RP = NT / CH;       // input: chunks per row, rows per pass (CH passes)
    constexpr int CHo = MP / 4, RPo = NT / CHo;    // output
    const int c_in = t % CH, r_in = t / CH, c_out = t % CHo, r_out = t / CHo;
    const bool vecX = (a.K % 4 == 0) && aligned16_dev(a.X), vecY = (a.M % 4 == 0) && aligned16_dev(a.Y);
    const bool has_bn_in = a.in_bn != nullptr, stats = a.stats != 0;
    const Bn4 bi = load_bn4(a.in_bn, a.K, c_in);
    const float4 bias4 = load_vec4(a.bias, a.M, c_out);
    float4 S1 = zero4(), S2 = zero4(), shift4 = zero4();
    bool have_shift = false;
    float n_cta = 0.f;
    constexpr uint32_t IDESC = make_idesc(128, 2 * MP, 0, 0);
    uint32_t phase = 0;

    int j = 0;
    for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++j) {
        const int64_t row0 = static_cast<int64_t>(tile) * 128;
        uint32_t slab = 0;
        if (RING > 0) {
            if (t == 0) issue(j + RING - 1);
            mbar_wait(s_u32(&full_mem[j % (RING > 0 ? RING : 1)]), (j / (RING > 0 ? RING : 1)) & 1);
            slab = sRing + (j % (RING > 0 ? RING : 1)) * RAW_BYTES;
        }
        // ---- prologue: X tile -> bn/act -> hi/lo operand tiles
#pragma unroll
        for (int i = 0; i < 128 / RP; ++i) {
            const int r = r_in + RP * i;
            const int64_t gr = row0 + r;
            float4 v = zero4();
            if (gr < a.N) v = RING > 0 ? raw_chunk(slab, r, a.K, c_in) : load_chunk(a.X, gr, a.K, c_in, vecX);
            if (has_bn_in) v = bn_apply(v, bi);
            v.x = act_f(v.x, a.in_act, a.in_slope); v.y = act_f(v.y, a.in_act, a.in_slope);
            v.z = act_f(v.z, a.in_act, a.in_slope); v.w = act_f(v.w, a.in_act, a.in_slope);
            const uint32_t off = tile_off(r, c_in, 128);
            store_split(sAh, sAl, off, v, 0, 0);
        }
        fence_async_smem();
        __syncthreads();
        if (t == 0) {
            tc_fence_after();
#pragma unroll
            for (int jj = 0; jj < KSTEPS; ++jj) {
                const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u, boff = (jj >> 2) * (2 * MP * 128u) + (jj & 3) * 32u;
                const uint64_t bd = make_desc(sB + boff, 16, 1024);
                const uint32_t d = tmem + (jj / KPA) * 2 * MP;
                tc_mma_tf32(d, make_desc(sAh + aoff, 16, 1024), bd, IDESC, (jj % KPA) != 0 ? 1u : 0u);
                tc_mma_tf32(d, make_desc(sAl + aoff, 16, 1024), bd, IDESC, 1);
            }
            tc_commit(bar);
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        __syncwarp();
        tc_fence_after();
        // ---- accumulators -> staging tile (thread = row, warps 0..3 own the TMEM lane quadrants): columns c and
        // MP + c are the [W_hi | W_lo] halves
#pragma unroll
        for (int cb = 0; cb < (w < 4 ? PM : 0); ++cb) {
            float v[32];
            tc_ld_sum<2 * NACC>(tmem + (static_cast<uint32_t>(w * 32) << 16) + cb * 32, MP, v);
#pragma unroll
            for (int q = 0; q < 8; ++q)
                sts128(sStage + tile_off(t, cb * 8 + q, 128), make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
        }
        tc_fence_before();
        __syncthreads();
        // ---- cooperative epilogue (thread = fixed 4 channels): bias, statistics, coalesced 128-bit stores
        if (stats && !have_shift) {
            const float4 s = lds128s(sStage + tile_off(0, c_out, 128));
            shift4 = make_float4(s.x + bias4.x, s.y + bias4.y, s.z + bias4.z, s.w + bias4.w);
            have_shift = true;
        }
#pragma unroll
        for (int i = 0; i < 128 / RPo; ++i) {
            const int r = r_out + RPo * i;
            const int64_t gr = row0 + r;
            if (gr < a.N) {
                float4 v = lds128s(sStage + tile_off(r, c_out, 128));
                v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w;
                store_chunk(a.Y, gr, a.M, c_out, v, vecY);
                if (stats) {
                    const float dx = v.x - shift4.x, dy = v.y - shift4.y, dz = v.z - shift4.z, dw = v.w - shift4.w;
                    S1.x += dx; S1.y += dy; S1.z += dz; S1.w += dw;
                    S2.x = fmaf(dx, dx, S2.x); S2.y = fmaf(dy, dy, S2.y); S2.z = fmaf(dz, dz, S2.z); S2.w = fmaf(dw, dw, S2.w);
                }
            }
        }
        const int64_t left = a.N - row0;
        n_cta += left < 128 ? static_cast<float>(left) : 128.f;
        __syncthreads();   // the staging tile aliases the operand tiles the next prologue overwrites
    }

    if (stats) {
        // per-CTA partial (n, shift, S1, S2) per channel; bn_finalize_kernel merges all partials in a fixed order
        chunk_allreduce<CHo>(S1);
        chunk_allreduce<CHo>(S2);
        if (lane < (CHo < 32 ? CHo : 32)) {
            float *p = &red[w][0];
            const int c0 = 4 * c_out;
            p[c0] = S1.x; p[c0 + 1] = S1.y; p[c0 + 2] = S1.z; p[c0 + 3] = S1.w;
            p[MP + c0] = S2.x; p[MP + c0 + 1] = S2.y; p[MP + c0 + 2] = S2.z; p[MP + c0 + 3] = S2.w;
        }
        if (r_out == 0) {
            const int c0 = 4 * c_out;
            shift_s[c0] = shift4.x; shift_s[c0 + 1] = shift4.y; shift_s[c0 + 2] = shift4.z; shift_s[c0 + 3] = shift4.w;
        }
        __syncthreads();
        if (t < MP) {
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int ww = 0; ww < NW; ++ww) { s1 += red[ww][t]; s2 += red[ww][MP + t]; }
            reinterpret_cast<float4 *>(a.part)[static_cast<size_t>(blockIdx.x) * MP + t] = make_float4(n_cta, shift_s[t], s1, s2);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (w == 0) tc_dealloc(tmem, TCOLS);
}

// ------------------------------------------------------------------------------------------------------------------
// backward stage
// ------------------------------------------------------------------------------------------------------------------

// room for the shared-memory copy of the weight-gradient blocks (2 MP x 2 KP floats) next to the operand tiles and the ring
__host__ __device__ constexpr bool bwd_accw_smem(int KP, int MP) { return KP * MP <= 32 * 64; }
// per-CTA partial record: dW as the four hi/lo blocks the MMA produces ([2 MP] x [2 KP]), db (MP), previous sums (2 KP)
__host__ __device__ constexpr int bwd_part_floats(int KP, int MP) { return 4 * MP * KP + MP + 2 * KP; }

template <int KP, int MP, int RING, int NT>
__global__ void __launch_bounds__(NT) lin_bwd_kernel(const LinBwdArgs a) {
    extern __shared__ uint8_t smem_raw[];
    constexpr int PK = KP / 32, PM = MP / 32;
    constexpr uint32_t G_BYTES = PM * PANEL128, X_BYTES = PK * PANEL128, W_BYTES = PK * MP * 128u;
    constexpr uint32_t RAW_G = 128u * MP * 4u, RAW_X = 128u * KP * 4u, RAW_SLOT = 2 * RAW_G + RAW_X;
    const uint32_t base = (s_u32(smem_raw) + 1023u) & ~1023u;
    // gY is kept twice: MN-major copy (weight gradient, contraction over rows; hi panels then lo panels = the M blocks
    // of ONE MMA) first, then the K-major copy (data gradient).  X' hi then lo panels = the N blocks of that MMA.
    const uint32_t sGmh = base, sGml = sGmh + G_BYTES, sGh = sGml + G_BYTES, sGl = sGh + G_BYTES;
    const uint32_t sXh = sGl + G_BYTES, sXl = sXh + X_BYTES, sWh = sXl + X_BYTES, sWl = sWh + W_BYTES, sRing = sWl + W_BYTES;
    const uint32_t sStage = sGh;        // the K-major gY copy is dead once the tile's MMAs have completed
    // Weight-gradient accumulation across the tiles of this CTA.  Left in tensor memory it would see 16 truncating
    // accumulations per tile (error ~ 16 T 2^-24 after T tiles, biased); instead every tile starts fresh accumulators and
    // its result is added to a shared-memory copy with fp32 adds (ACCW_SMEM).  Only the 64 x 64 shape has no room for
    // that copy and keeps accumulating in tensor memory.
    constexpr bool ACCW_SMEM = bwd_accw_smem(KP, MP);
    const uint32_t sAccW = sRing + RING * RAW_SLOT;     // [2 KP / 4 float4 columns][2 MP lanes] float4, lane fastest
    static_assert(2 * PM >= PK, "staging tile must fit the K-major gY copy");
    static_assert(2 * MP <= 128, "the weight-gradient MMA stacks gY hi and lo along M = 128");
    __shared__ __align__(8) uint64_t bar_mem;
    __shared__ __align__(8) uint64_t full_mem[RING > 0 ? RING : 1];
    __shared__ uint32_t tmem_ptr;
    float (*red)[MP + 2 * KP] = reinterpret_cast<float (*)[MP + 2 * KP]>(smem_raw + (sXh - s_u32(smem_raw)));   // used after the last MMA

    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    const uint32_t bar = s_u32(&bar_mem);
    // accumulators (see lin_fwd_kernel: at most a few MMAs per accumulator): data gradient NACC_D x [2 KP] columns, then
    // weight gradient NACC_W x [2 KP] columns; the weight accumulators are re-started every tile and added to the CTA's
    // partial in global memory with fp32 adds
    // data gradient: all gY_lo products first (2^-11 of the result: their truncation is harmless), then the gY_hi k-steps
    // spread over NACC_D accumulators (2 at MP = 64: four full-magnitude accumulations each) -- the same measures as the
    // pipelined forward stage (mlp_pipe.cu header); this kernel serves the 64-wide backward of the counting models
    constexpr int KS_D = MP / 8, NACC_D = (MP >= 64 && TC_SPLIT_ACC < 2) ? 2 : TC_SPLIT_ACC, KPA_D = KS_D / NACC_D;
    constexpr int NACC_W = TC_SPLIT_ACC, KPA_W = 16 / NACC_W;
    constexpr uint32_t WBASE = NACC_D * 2 * KP;
    constexpr uint32_t TCOLS = (WBASE + NACC_W * 2 * KP) <= 128 ? 128 : ((WBASE + NACC_W * 2 * KP) <= 256 ? 256 : 512);
    static_assert(WBASE + NACC_W * 2 * KP <= 512, "tensor memory budget");
    if (t == 0) {
        mbar_init(bar, 1);
        for (int s = 0; s < RING; ++s) mbar_init(s_u32(&full_mem[s]), 1);
        fence_barrier_init();
    }
    if (w == 0) tc_alloc(s_u32(&tmem_ptr), TCOLS);
    __syncthreads();
    const bool want_gx = a.GX != nullptr, has_bn = a.bn != nullptr, has_bn_in = a.in_bn != nullptr;
    auto issue = [&](int j) {
        const int64_t tile = static_cast<int64_t>(blockIdx.x) + static_cast<int64_t>(j) * gridDim.x;
        if (tile >= a.num_tiles) return;
        const int64_t row0 = tile * 128, left = a.N - row0;
        const uint32_t rows = static_cast<uint32_t>(left < 128 ? left : 128);
        const uint32_t gb = rows * a.M * 4u, xb = rows * a.K * 4u;
        const uint32_t slot = sRing + (j % (RING > 0 ? RING : 1)) * RAW_SLOT, fb = s_u32(&full_mem[j % (RING > 0 ? RING : 1)]);
        mbar_expect_tx(fb, gb * ((has_bn ? 1u : 0u) + (a.G != nullptr ? 1u : 0u)) + xb);
        if (a.G != nullptr) bulk_g2s(slot, a.G + row0 * a.M, gb, fb);
        if (has_bn) bulk_g2s(slot + RAW_G, a.Yo + row0 * a.M, gb, fb);
        bulk_g2s(slot + 2 * RAW_G, a.X + row0 * a.K, xb, fb);
    };
    if (RING > 0 && t == 0)
        for (int j = 0; j < RING - 1; ++j) issue(j);
    // weights as they are stored: rows m (the data GEMM's K), k contiguous (its N) -> MN-major B operand,
    // hi panels then lo panels = the N blocks of one MMA
    const bool vecW = (a.K % 4 == 0) && aligned16_dev(a.W);
    if (want_gx) {
        for (int i = t; i < MP * (KP / 4); i += NT) {
            const int m = i / (KP / 4), c = i % (KP / 4);
            const float4 v = (m < a.M) ? load_chunk(a.W, m, a.K, c, vecW) : zero4();
            store_split(sWh, sWl, tile_off_mn(m, c, MP), v, 0, 0);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_ptr;

    constexpr int CHm = MP / 4, RPm = NT / CHm;    // gradient / output-channel side
    constexpr int CHk = KP / 4, RPk = NT / CHk;    // input-channel side
    const int c_m = t % CHm, r_m = t / CHm, c_k = t % CHk, r_k = t / CHk;
    const bool vecG = (a.M % 4 == 0) && aligned16_dev(a.G) && (a.Yo == nullptr || aligned16_dev(a.Yo));
    const bool vecGs = (a.M % 4 == 0) && aligned16_dev(a.Gseg);
    const bool vecX = (a.K % 4 == 0) && aligned16_dev(a.X), vecGX = (a.K % 4 == 0) && aligned16_dev(a.GX);
    const Bn4 bo = load_bn4(a.bn, a.M, c_m), bi = load_bn4(a.in_bn, a.K, c_k);
    float4 m1 = zero4(), m2 = zero4();
    if (has_bn) {
        const float invN = 1.f / static_cast<float>(a.N);
        const float4 s1 = load_vec4(a.sums, a.M, c_m), s2 = load_vec4(a.sums + a.M, a.M, c_m);
        m1 = make_float4(s1.x * invN, s1.y * invN, s1.z * invN, s1.w * invN);
        m2 = make_float4(s2.x * invN, s2.y * invN, s2.z * invN, s2.w * invN);
    }
    float4 db4 = zero4(), sp1 = zero4(), sp2 = zero4();
    constexpr uint32_t IDESC_DATA = make_idesc(128, 2 * KP, 0, 1);   // gY (K-major) x [W_hi | W_lo] (MN-major)
    constexpr uint32_t IDESC_WGT = make_idesc(128, 2 * KP, 1, 1);    // [gY_hi ; gY_lo]^T (MN-major) x [X'_hi | X'_lo] (MN-major)
    uint32_t phase = 0;
    bool first = true;
    float *part = a.part + static_cast<size_t>(blockIdx.x) * bwd_part_floats(KP, MP);

    int j = 0;
    for (int tile = blockIdx.x; tile < a.num_tiles; tile += gridDim.x, ++j) {
        const int64_t row0 = static_cast<int64_t>(tile) * 128;
        uint32_t slab = 0;
        if (RING > 0) {
            if (t == 0) issue(j + RING - 1);
            mbar_wait(s_u32(&full_mem[j % (RING > 0 ? RING : 1)]), (j / (RING > 0 ? RING : 1)) & 1);
            slab = sRing + (j % (RING > 0 ? RING : 1)) * RAW_SLOT;
        }
        // ---- prologue A: gradient of the stage's linear output, gY (BatchNorm backward folded in)
#pragma unroll
        for (int i = 0; i < 128 / RPm; ++i) {
            const int r = r_m + RPm * i;
            const int64_t gr = row0 + r;
            float4 g = zero4();
            if (gr < a.N) {
                if (a.G != nullptr) g = RING > 0 ? raw_chunk(slab, r, a.M, c_m) : load_chunk(a.G, gr, a.M, c_m, vecG);
                if (a.Gseg != nullptr) {   // + the readout gradient of this row's graph (global_add/mean_pool backward)
                    const float4 gs = load_chunk(a.Gseg, __ldg(a.row2seg + gr), a.M, c_m, vecGs);
                    g.x += gs.x; g.y += gs.y; g.z += gs.z; g.w += gs.w;
                }
                if (has_bn) {
                    const float4 y = RING > 0 ? raw_chunk(slab + RAW_G, r, a.M, c_m) : load_chunk(a.Yo, gr, a.M, c_m, vecG);
                    const float4 xc = make_float4(y.x - bo.mean.x, y.y - bo.mean.y, y.z - bo.mean.z, y.w - bo.mean.w);
                    if (!a.g_masked) {
                        if (!(fmaf(xc.x, bo.k.x, bo.beta.x) > 0.f)) g.x = 0.f;
                        if (!(fmaf(xc.y, bo.k.y, bo.beta.y) > 0.f)) g.y = 0.f;
                        if (!(fmaf(xc.z, bo.k.z, bo.beta.z) > 0.f)) g.z = 0.f;
                        if (!(fmaf(xc.w, bo.k.w, bo.beta.w) > 0.f)) g.w = 0.f;
                    }
                    g.x = bo.k.x * (g.x - m1.x - xc.x * bo.rstd.x * m2.x);
                    g.y = bo.k.y * (g.y - m1.y - xc.y * bo.rstd.y * m2.y);
                    g.z = bo.k.z * (g.z - m1.z - xc.z * bo.rstd.z * m2.z);
                    g.w = bo.k.w * (g.w - m1.w - xc.w * bo.rstd.w * m2.w);
                }
                db4.x += g.x; db4.y += g.y; db4.z += g.z; db4.w += g.w;
            }
            store_split2(sGh, sGl, tile_off(r, c_m, 128), sGmh, sGml, tile_off_mn(r, c_m, 128), g);
        }
        // ---- prologue B: the stage's forward input as the GEMM saw it, X' = act(bn_in(X))
#pragma unroll
        for (int i = 0; i < 128 / RPk; ++i) {
            const int r = r_k + RPk * i;
            const int64_t gr = row0 + r;
            float4 v = zero4();
            if (gr < a.N) {
                v = RING > 0 ? raw_chunk(slab + 2 * RAW_G, r, a.K, c_k) : load_chunk(a.X, gr, a.K, c_k, vecX);
                if (has_bn_in) v = bn_apply(v, bi);
                v.x = act_f(v.x, a.in_act, a.in_slope); v.y = act_f(v.y, a.in_act, a.in_slope);
                v.z = act_f(v.z, a.in_act, a.in_slope); v.w = act_f(v.w, a.in_act, a.in_slope);
            }
            store_split(sXh, sXl, tile_off_mn(r, c_k, 128), v, 0, 0);
        }
        fence_async_smem();
        __syncthreads();
        if (t == 0) {
            tc_fence_after();
            if (want_gx) {
                // data gradient: (128 x MP) x (MP x [KP hi | KP lo]); k-steps of 8 output channels
#pragma unroll
                for (int jj = 0; jj < KS_D; ++jj) {
                    const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u;
                    tc_mma_tf32(tmem, make_desc(sGl + aoff, 16, 1024), make_desc_mn(sWh + jj * 1024u, MP * 128u), IDESC_DATA, jj != 0 ? 1u : 0u);
                }
#pragma unroll
                for (int jj = 0; jj < KS_D; ++jj) {
                    const uint32_t aoff = (jj >> 2) * PANEL128 + (jj & 3) * 32u;
                    const int acc = jj / KPA_D;
                    tc_mma_tf32(tmem + acc * 2 * KP, make_desc(sGh + aoff, 16, 1024), make_desc_mn(sWh + jj * 1024u, MP * 128u), IDESC_DATA,
                                (acc == 0 || (jj % KPA_D) != 0) ? 1u : 0u);
                }
            }
            // weight gradient: ([MP hi ; MP lo ; ...] x 128 rows) x (128 rows x [KP hi | KP lo]); k-steps of 8 rows,
            // per tile into fresh accumulators (ACCW_SMEM) or on top of the previous tiles
#pragma unroll
            for (int jj = 0; jj < 16; ++jj)
                tc_mma_tf32(tmem + WBASE + (jj / KPA_W) * 2 * KP, make_desc_mn(sGmh + jj * 1024u, PANEL128),
                            make_desc_mn(sXh + jj * 1024u, PANEL128), IDESC_WGT,
                            ((jj % KPA_W) != 0 || (!ACCW_SMEM && !first)) ? 1u : 0u);
            tc_commit(bar);
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        __syncwarp();
        tc_fence_after();
        // ---- this tile's weight-gradient blocks += the CTA's shared-memory copy (thread = accumulator lane, its own
        // column of float4 slots: conflict-free, no race)
        if (ACCW_SMEM && w * 32 < 2 * MP) {
#pragma unroll
            for (int cb = 0; cb < 2 * PK; ++cb) {
                float v[32];
                tc_ld_sum<NACC_W>(tmem + (static_cast<uint32_t>(w * 32) << 16) + WBASE + cb * 32, 2 * KP, v);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint32_t slot = sAccW + static_cast<uint32_t>(((cb * 8 + q) * 2 * MP + t) * 16);
                    float4 o = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                    if (!first) {
                        const float4 p = lds128s(slot);
                        o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
                    }
                    sts128(slot, o);
                }
            }
        }
        first = false;
        if (want_gx) {
#pragma unroll
            for (int cb = 0; cb < (w < 4 ? PK : 0); ++cb) {
                float v[32];
                tc_ld_sum<2 * NACC_D>(tmem + (static_cast<uint32_t>(w * 32) << 16) + cb * 32, KP, v);
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    sts128(sStage + tile_off(t, cb * 8 + q, 128), make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]));
            }
            tc_fence_before();
            __syncthreads();
            // ---- cooperative epilogue: activation mask of the previous stage + its BatchNorm-backward sums
#pragma unroll
            for (int i = 0; i < 128 / RPk; ++i) {
                const int r = r_k + RPk * i;
                const int64_t gr = row0 + r;
                if (gr < a.N) {
                    float4 g = lds128s(sStage + tile_off(r, c_k, 128));
                    if (a.in_act != DN4GL_ACT_NONE || has_bn_in) {
                        const float4 x = RING > 0 ? raw_chunk(slab + 2 * RAW_G, r, a.K, c_k) : load_chunk(a.X, gr, a.K, c_k, vecX);
                        if (has_bn_in) {
                            const float4 xc = make_float4(x.x - bi.mean.x, x.y - bi.mean.y, x.z - bi.mean.z, x.w - bi.mean.w);
                            g.x *= dact_f(fmaf(xc.x, bi.k.x, bi.beta.x), a.in_act, a.in_slope);
                            g.y *= dact_f(fmaf(xc.y, bi.k.y, bi.beta.y), a.in_act, a.in_slope);
                            g.z *= dact_f(fmaf(xc.z, bi.k.z, bi.beta.z), a.in_act, a.in_slope);
                            g.w *= dact_f(fmaf(xc.w, bi.k.w, bi.beta.w), a.in_act, a.in_slope);
                            sp1.x += g.x; sp1.y += g.y; sp1.z += g.z; sp1.w += g.w;
                            sp2.x = fmaf(g.x, xc.x * bi.rstd.x, sp2.x); sp2.y = fmaf(g.y, xc.y * bi.rstd.y, sp2.y);
                            sp2.z = fmaf(g.z, xc.z * bi.rstd.z, sp2.z); sp2.w = fmaf(g.w, xc.w * bi.rstd.w, sp2.w);
                        } else {
                            g.x *= dact_f(x.x, a.in_act, a.in_slope); g.y *= dact_f(x.y, a.in_act, a.in_slope);
                            g.z *= dact_f(x.z, a.in_act, a.in_slope); g.w *= dact_f(x.w, a.in_act, a.in_slope);
                        }
                    }
                    store_chunk(a.GX, gr, a.K, c_k, g, vecGX);
                }
            }
        }
        __syncthreads();   // staging aliases the K-major gY copy; the ring slot of this tile is refilled next iteration
    }

    // ---- per-CTA partials: dW blocks (2 MP x 2 KP), db (MP), previous-stage sums (2 KP)
    if (w * 32 < 2 * MP) {
#pragma unroll
        for (int cb = 0; cb < 2 * PK; ++cb) {
            float4 *dst = reinterpret_cast<float4 *>(part + t * (2 * KP) + cb * 32);
            if (ACCW_SMEM) {
#pragma unroll
                for (int q = 0; q < 8; ++q) dst[q] = lds128s(sAccW + static_cast<uint32_t>(((cb * 8 + q) * 2 * MP + t) * 16));
            } else {
                float v[32];
                tc_ld_sum<NACC_W>(tmem + (static_cast<uint32_t>(w * 32) << 16) + WBASE + cb * 32, 2 * KP, v);
#pragma unroll
                for (int q = 0; q < 8; ++q) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            }
        }
    }
    __syncthreads();
    chunk_allreduce<CHm>(db4);
    chunk_allreduce<CHk>(sp1);
    chunk_allreduce<CHk>(sp2);
    if (lane < (CHm < 32 ? CHm : 32)) {
        const int c0 = 4 * c_m;
        red[w][c0] = db4.x; red[w][c0 + 1] = db4.y; red[w][c0 + 2] = db4.z; red[w][c0 + 3] = db4.w;
    }
    if (lane < (CHk < 32 ? CHk : 32)) {
        const int c0 = MP + 4 * c_k;
        red[w][c0] = sp1.x; red[w][c0 + 1] = sp1.y; red[w][c0 + 2] = sp1.z; red[w][c0 + 3] = sp1.w;
        red[w][KP + c0] = sp2.x; red[w][KP + c0 + 1] = sp2.y; red[w][KP + c0 + 2] = sp2.z; red[w][KP + c0 + 3] = sp2.w;
    }
    __syncthreads();
    for (int i = t; i < MP + 2 * KP; i += NT) {
        float sum = 0.f;
#pragma unroll
        for (int ww = 0; ww < NT / 32; ++ww) sum += red[ww][i];
        part[4 * MP * KP + i] = sum;
    }
    tc_fence_before();
    __syncthreads();
    if (w == 0) tc_dealloc(tmem, TCOLS);
}

// Fixed-order sums of per-CTA partials.  A block is 32 output elements x 32 partial groups: thread (lane, g) adds
// partials g, g+32, ... in double.  ALL loads of a thread (up to 8 partials x NCOL columns) are issued before the first
// add: the r1d profile showed these few-CTA kernels spending 14-15 us on 5-10 dependent L2/DRAM round trips
// (long_scoreboard 13-27 per issue) for 2.5 MB of data.  The add order stays fixed (p ascending, columns in order).
template <int NCOL, int UNR = 8>
__device__ __forceinline__ double partial_columns_sum(const float *__restrict__ part, int nparts, int stride,
                                                      const int (&e)[NCOL], int g) {
    double s = 0.0;
    for (int p0 = g; p0 < nparts; p0 += 32 * UNR) {
        float v[UNR][NCOL];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int p = p0 + 32 * u;
#pragma unroll
            for (int c = 0; c < NCOL; ++c) v[u][c] = (p < nparts) ? __ldcg(part + static_cast<size_t>(p) * stride + e[c]) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
#pragma unroll
            for (int c = 0; c < NCOL; ++c) s += static_cast<double>(v[u][c]);
        }
    }
    return s;
}
// sm[g][lane] = s for all 32 x 32 threads; warp w then owns element w: it reads the 32 group values of that element and
// combines them with a fixed xor-butterfly.  Returns the total of element `g` (valid in every lane of warp g).
__device__ __forceinline__ double group_sum(double (*sm)[33], int lane, int g, double s) {
    sm[g][lane] = s;
    __syncthreads();
    double t = sm[lane][g];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    __syncthreads();
    return t;
}

// dW / db / previous-stage sums.  dW[m][k] is the sum of the four hi/lo blocks of the weight accumulator.
__global__ void __launch_bounds__(1024)
lin_bwd_reduce_kernel(const float *__restrict__ part, int nparts, int MP, int KP, int M, int K,
                      float *__restrict__ dW, float *__restrict__ db, float *__restrict__ sums_prev) {
    __shared__ double sm[32][33];
    __shared__ float *sm_dst[32];
    const int stride = bwd_part_floats(KP, MP);
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    const int e = blockIdx.x * 32 + lane;                 // logical element: [MP*KP dW | MP db | 2 KP sums]
    float *dst = nullptr;
    double s = 0.0;
    if (e < MP * KP) {
        const int m = e / KP, k = e % KP;
        if (m < M && k < K && dW) {
            dst = dW + m * K + k;
            const int cols[4] = {m * 2 * KP + k, m * 2 * KP + KP + k, (MP + m) * 2 * KP + k, (MP + m) * 2 * KP + KP + k};
            s = partial_columns_sum<4, 5>(part, nparts, stride, cols, g);   // 148 partials: one pass of 5 x 4 loads
        }
    } else if (e < MP * KP + MP) {
        const int m = e - MP * KP;
        if (m < M && db) {
            dst = db + m;
            const int cols[1] = {4 * MP * KP + m};
            s = partial_columns_sum<1>(part, nparts, stride, cols, g);
        }
    } else if (e < MP * KP + MP + 2 * KP) {
        const int i = e - MP * KP - MP, which = i / KP, k = i % KP;
        if (k < K && sums_prev) {
            dst = sums_prev + which * K + k;
            const int cols[1] = {4 * MP * KP + MP + i};
            s = partial_columns_sum<1>(part, nparts, stride, cols, g);
        }
    }
    if (g == 0) sm_dst[lane] = dst;
    const double tot = group_sum(sm, lane, g, s);        // total of element blockIdx.x * 32 + g
    if (lane == 0 && sm_dst[g] != nullptr) *sm_dst[g] = static_cast<float>(tot);
}

// BatchNorm record from the per-CTA (n, shift, S1, S2) partials of lin_fwd_kernel: every partial is re-centred on the
// mean of CTA 0 (exact in double), so the merge is a plain fixed-order sum and cancellation-free.
__global__ void __launch_bounds__(1024)
bn_finalize_kernel(const float4 *__restrict__ part, int nparts, int MP, int M, int64_t N,
                   const float *__restrict__ gamma, const float *__restrict__ beta, float eps, float momentum,
                   float *__restrict__ bn_out, float *__restrict__ run_mean, float *__restrict__ run_var, long long *nbt) {
    __shared__ double sm[32][33];
    __shared__ double sm_kstar[32];
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + lane;     // < MP (MP is a multiple of 32)
    const float4 p0 = __ldcg(part + c);
    double A1 = 0.0, A2 = 0.0;
    double kstar = 0.0;
    bool have_k = false;
    constexpr int UNR = 5;                                 // 296 partials: two passes of 5 loads
    for (int q0 = g; q0 < nparts; q0 += 32 * UNR) {        // all loads of the chunk first, then the double arithmetic
        float4 v[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int p = q0 + 32 * u;
            v[u] = (p < nparts) ? __ldcg(part + static_cast<size_t>(p) * MP + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (!have_k) {
            kstar = static_cast<double>(p0.y) + static_cast<double>(p0.z) / static_cast<double>(p0.x);
            have_k = true;
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const double n = v[u].x;
            if (n > 0.0) {
                const double s1 = v[u].z, s2 = v[u].w;
                const double r = s1 / n;
                const double mean_i = static_cast<double>(v[u].y) + r, m2_i = s2 - s1 * r;
                const double d = mean_i - kstar;
                A1 += n * d;
                A2 += (m2_i > 0.0 ? m2_i : 0.0) + n * d * d;
            }
        }
    }
    if (!have_k) kstar = static_cast<double>(p0.y) + static_cast<double>(p0.z) / static_cast<double>(p0.x);
    if (g == 0) sm_kstar[lane] = kstar;
    const double a1 = group_sum(sm, lane, g, A1);          // totals of channel blockIdx.x * 32 + g
    const double a2 = group_sum(sm, lane, g, A2);
    const int cc = blockIdx.x * 32 + g;
    if (lane == 0 && cc < M) {
        const double ks = sm_kstar[g];
        const double Nd = static_cast<double>(N);
        const double mean = ks + a1 / Nd;
        double m2 = a2 - a1 * a1 / Nd;
        if (m2 < 0.0) m2 = 0.0;
        const double var = m2 / Nd;
        const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
        const float gam = gamma ? gamma[cc] : 1.f, bet = beta ? beta[cc] : 0.f;
        bn_out[cc] = static_cast<float>(mean);
        bn_out[M + cc] = rstd;
        bn_out[2 * M + cc] = gam * rstd;
        bn_out[3 * M + cc] = bet;
        if (run_mean) run_mean[cc] = (1.f - momentum) * run_mean[cc] + momentum * static_cast<float>(mean);
        if (run_var) {
            const double unb = N > 1 ? m2 / (Nd - 1.0) : var;
            run_var[cc] = (1.f - momentum) * run_var[cc] + momentum * static_cast<float>(unb);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && nbt) *nbt += 1;
}

// ------------------------------------------------------------------------------------------------------------------
// elementwise companions
// ------------------------------------------------------------------------------------------------------------------
// out = act(bn(Y))  (the activation a stage hands to a non-MLP consumer: aggregation, readout)
__global__ void bn_act_kernel(const float *__restrict__ Y, int64_t N, int M, const float *__restrict__ bn, int act, float slope,
                              float *__restrict__ out) {
    const int CH = (M + 3) / 4;
    const bool vec = (M % 4 == 0) && aligned16_dev(Y) && aligned16_dev(out);
    const int64_t total = N * CH;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t r = i / CH;
        const int c = static_cast<int>(i % CH);
        const Bn4 b = load_bn4(bn, M, c);
        float4 v = load_chunk(Y, r, M, c, vec);
        if (bn) v = bn_apply(v, b);
        v.x = act_f(v.x, act, slope); v.y = act_f(v.y, act, slope); v.z = act_f(v.z, act, slope); v.w = act_f(v.w, act, slope);
        store_chunk(out, r, M, c, v, vec);
    }
}

// out = act(bn(Y)) AND the per-graph readout of out in the same pass (global_add_pool / global_mean_pool over contiguous
// row segments, gconv.py:175-178,213): one CTA per graph, thread = fixed 4 channels x strided rows, fixed-order combine.
template <int CHP>
__global__ void __launch_bounds__(256) bn_act_pool_kernel(const float *__restrict__ Y, int M, const float *__restrict__ bn, int act,
                                                          float slope, float *__restrict__ out, const int32_t *__restrict__ seg_ptr,
                                                          int B, int mode, float *__restrict__ pooled) {
    constexpr int RP = 256 / CHP;
    __shared__ float red[8][4 * CHP];
    const int t = threadIdx.x, w = t >> 5, lane = t & 31, c = t % CHP, r0 = t / CHP;
    const bool vec = (M % 4 == 0) && aligned16_dev(Y) && aligned16_dev(out);
    const Bn4 b = load_bn4(bn, M, c);
    for (int g = blockIdx.x; g < B; g += gridDim.x) {
        const int beg = __ldg(seg_ptr + g), end = __ldg(seg_ptr + g + 1);
        float4 acc = zero4();
        if (4 * c < M) {
            // four rows per thread in flight: with one load per iteration the 1 000-row graphs of the C2 batch made their
            // CTA walk 34 dependent DRAM round trips (23 us for a 6 us traffic problem, profiles/r1d); same add order
            int r = beg + r0;
            for (; r + 3 * RP < end; r += 4 * RP) {
                float4 v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = load_chunk(Y, r + u * RP, M, c, vec);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (bn) v[u] = bn_apply(v[u], b);
                    v[u].x = act_f(v[u].x, act, slope); v[u].y = act_f(v[u].y, act, slope);
                    v[u].z = act_f(v[u].z, act, slope); v[u].w = act_f(v[u].w, act, slope);
                    store_chunk(out, r + u * RP, M, c, v[u], vec);
                    acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
                }
            }
            for (; r < end; r += RP) {
                float4 v = load_chunk(Y, r, M, c, vec);
                if (bn) v = bn_apply(v, b);
                v.x = act_f(v.x, act, slope); v.y = act_f(v.y, act, slope); v.z = act_f(v.z, act, slope); v.w = act_f(v.w, act, slope);
                store_chunk(out, r, M, c, v, vec);
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
        }
        chunk_allreduce<CHP>(acc);
        if (lane < CHP) {
            const int c0 = 4 * c;
            red[w][c0] = acc.x; red[w][c0 + 1] = acc.y; red[w][c0 + 2] = acc.z; red[w][c0 + 3] = acc.w;
        }
        __syncthreads();
        if (t < M) {
            // CHP >= 32 never occurs with 8-lane groups sharing a warp only when CHP < 32; for CHP == 32 every warp holds
            // distinct rows of all chunks, so the sum over warps is still the right combine
            float sum = 0.f;
#pragma unroll
            for (int ww = 0; ww < 8; ++ww) sum += red[ww][t];
            if (mode == 1) sum *= 1.f / static_cast<float>(max(end - beg, 1));
            pooled[static_cast<int64_t>(g) * M + t] = sum;
        }
        __syncthreads();
    }
}

// row -> segment index for contiguous segments (the `batch` vector of a PyG batch, as int32)
__global__ void segment_ids_kernel(const int32_t *__restrict__ seg_ptr, int B, int64_t N, int32_t *__restrict__ out) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < N) out[i] = segment_of(seg_ptr, B, i);
}

// BatchNorm-backward batch sums of a stage whose gradient arrives from outside the MLP:
// s1[c] = sum_r gm, s2[c] = sum_r gm * xhat, gm = G * act'(bn(Y)), xhat = (Y - mean) * rstd.  Per-CTA partials.
template <int CHP>   // chunks per row rounded up to a power of two (<= 32)
__global__ void __launch_bounds__(256) bn_bwd_sums_kernel(const float *__restrict__ G, const float *__restrict__ Gseg,
                                                          const int32_t *__restrict__ row2seg, const float *__restrict__ Y,
                                                          int64_t N, int M, const float *__restrict__ bn, int act, float slope,
                                                          float *__restrict__ part /* [grid][2*4*CHP] */, float *__restrict__ sums,
                                                          int *__restrict__ counters) {
    constexpr int RP = 256 / CHP;
    __shared__ float red[8][8 * CHP];
    __shared__ double dred[256];
    const int t = threadIdx.x, w = t >> 5, lane = t & 31, c = t % CHP, r0 = t / CHP;
    const bool vec = (M % 4 == 0) && aligned16_dev(G) && aligned16_dev(Y) && aligned16_dev(Gseg);
    const Bn4 b = load_bn4(bn, M, c);
    float4 s1 = zero4(), s2 = zero4();
    if (4 * c < M) {
        // several rows per thread in flight (all loads first, then the arithmetic in row order: same sums as one at a time)
        const int64_t stride = static_cast<int64_t>(gridDim.x) * RP;
        auto accumulate = [&](float4 g, const float4 &y) {
            const float4 xc = make_float4(y.x - b.mean.x, y.y - b.mean.y, y.z - b.mean.z, y.w - b.mean.w);
            g.x *= dact_f(fmaf(xc.x, b.k.x, b.beta.x), act, slope); g.y *= dact_f(fmaf(xc.y, b.k.y, b.beta.y), act, slope);
            g.z *= dact_f(fmaf(xc.z, b.k.z, b.beta.z), act, slope); g.w *= dact_f(fmaf(xc.w, b.k.w, b.beta.w), act, slope);
            s1.x += g.x; s1.y += g.y; s1.z += g.z; s1.w += g.w;
            s2.x = fmaf(g.x, xc.x * b.rstd.x, s2.x); s2.y = fmaf(g.y, xc.y * b.rstd.y, s2.y);
            s2.z = fmaf(g.z, xc.z * b.rstd.z, s2.z); s2.w = fmaf(g.w, xc.w * b.rstd.w, s2.w);
        };
        int64_t r = static_cast<int64_t>(blockIdx.x) * RP + r0;
        constexpr int UR = 2;   // rows in flight per thread (4 needed 90 registers and halved the occupancy)
        for (; r + (UR - 1) * stride < N; r += UR * stride) {
            float4 g[UR], y[UR];
            int seg[UR];
#pragma unroll
            for (int u = 0; u < UR; ++u) {
                g[u] = G != nullptr ? load_chunk(G, r + u * stride, M, c, vec) : zero4();
                seg[u] = Gseg != nullptr ? __ldg(row2seg + r + u * stride) : 0;
                y[u] = load_chunk(Y, r + u * stride, M, c, vec);
            }
            if (Gseg != nullptr) {
#pragma unroll
                for (int u = 0; u < UR; ++u) {
                    const float4 gs = load_chunk(Gseg, seg[u], M, c, vec);
                    g[u].x += gs.x; g[u].y += gs.y; g[u].z += gs.z; g[u].w += gs.w;
                }
            }
#pragma unroll
            for (int u = 0; u < UR; ++u) accumulate(g[u], y[u]);
        }
        for (; r < N; r += stride) {
            float4 g = G != nullptr ? load_chunk(G, r, M, c, vec) : zero4();
            if (Gseg != nullptr) {
                const float4 gs = load_chunk(Gseg, __ldg(row2seg + r), M, c, vec);
                g.x += gs.x; g.y += gs.y; g.z += gs.z; g.w += gs.w;
            }
            accumulate(g, load_chunk(Y, r, M, c, vec));
        }
    }
    chunk_allreduce<CHP>(s1);
    chunk_allreduce<CHP>(s2);
    if (lane < CHP) {
        const int c0 = 4 * c;
        red[w][c0] = s1.x; red[w][c0 + 1] = s1.y; red[w][c0 + 2] = s1.z; red[w][c0 + 3] = s1.w;
        red[w][4 * CHP + c0] = s2.x; red[w][4 * CHP + c0 + 1] = s2.y; red[w][4 * CHP + c0 + 2] = s2.z; red[w][4 * CHP + c0 + 3] = s2.w;
    }
    __syncthreads();
    for (int i = t; i < 8 * CHP; i += 256) {
        float s = 0.f;
#pragma unroll
        for (int ww = 0; ww < 8; ++ww) s += red[ww][i];
        part[static_cast<size_t>(blockIdx.x) * 8 * CHP + i] = s;
    }
    // grid rendezvous (tc_common.cuh), then CTA e merges entry e of the per-CTA partials: thread q adds partials q,
    // q + 256, ... in that order (double), then a fixed tree over the threads.  This replaces the follow-up reduce kernel.
    constexpr int NE = 8 * CHP;
    const int Gc = static_cast<int>(gridDim.x);
    const bool merger = static_cast<int>(blockIdx.x) < NE;
    const int passed = grid_arrive(counters, counters + 1, Gc, merger);
    if (!merger) return;
    for (int e = static_cast<int>(blockIdx.x); e < NE; e += Gc) {
        double acc = 0.0;
        constexpr int UNR = 3;      // 3 x 256 threads >= 4 x 148 CTAs: one round of loads
        for (int q0 = 0; q0 < Gc; q0 += 256 * UNR) {
            float v[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int q = q0 + t + 256 * u;
                v[u] = (q < Gc) ? __ldcg(part + static_cast<size_t>(q) * NE + e) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) acc += static_cast<double>(v[u]);
        }
        acc = warp_sum_f64(acc);
        if (lane == 0) dred[w] = acc;
        __syncthreads();
        if (t == 0) {
            double tot = 0.0;
#pragma unroll
            for (int ww = 0; ww < 8; ++ww) tot += dred[ww];
            const int which = e / (4 * CHP), ch = e % (4 * CHP);
            if (ch < M) sums[which * M + ch] = static_cast<float>(tot);
        }
        __syncthreads();
    }
    grid_depart(counters, counters + 1, passed, Gc < NE ? Gc : NE);
}

// ---------------------------------------------------------------------------------------------------------------
// Stand-alone training-mode BatchNorm1d for widths the fused stages do not take (65 .. 128 columns: main.py:174's default
// hidden 128): batch statistics as per-CTA shifted sums {n, a, S1 = sum (y - a), S2 = sum (y - a)^2} merged by
// bn_finalize_kernel (the same fixed-order double-precision merge as the stage kernels' statistics), and the backward
// elementwise pass  gx = gamma rstd (gm - s1 / N - xhat s2 / N),  gm = g act'(bn(y)).  ATen's batch-norm backward
// reduces the 1.5e5 rows of a full PROTEINS batch in fp32 and lands 3e-4 from float64 on the BatchNorm parameter
// gradients (profiles/*parity_errors*.json, hid 128); these are at 1e-6.
template <int CHP>
__global__ void __launch_bounds__(256) bn_stats_partial_kernel(const float *__restrict__ Y, int64_t N, int M, int MP,
                                                               float4 *__restrict__ part /* [grid][MP] */) {
    constexpr int RP = 256 / CHP;
    __shared__ float red[8][8 * CHP];
    const int t = threadIdx.x, w = t >> 5, lane = t & 31, c = t % CHP, r0 = t / CHP;
    const bool vec = (M % 4 == 0) && aligned16_dev(Y);
    const int64_t first = static_cast<int64_t>(blockIdx.x) * RP;          // < N: the host sizes the grid by row groups
    float4 s1 = zero4(), s2 = zero4(), a4 = zero4();
    if (4 * c < M) {
        a4 = load_chunk(Y, first, M, c, vec);                               // the CTA's shift: its first row
        const int64_t stride = static_cast<int64_t>(gridDim.x) * RP;
        auto accumulate = [&](const float4 &y) {
            const float dx = y.x - a4.x, dy = y.y - a4.y, dz = y.z - a4.z, dw = y.w - a4.w;
            s1.x += dx; s1.y += dy; s1.z += dz; s1.w += dw;
            s2.x = fmaf(dx, dx, s2.x); s2.y = fmaf(dy, dy, s2.y); s2.z = fmaf(dz, dz, s2.z); s2.w = fmaf(dw, dw, s2.w);
        };
        int64_t r = first + r0;
        for (; r + 3 * stride < N; r += 4 * stride) {
            float4 y[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) y[u] = load_chunk(Y, r + u * stride, M, c, vec);
#pragma unroll
            for (int u = 0; u < 4; ++u) accumulate(y[u]);
        }
        for (; r < N; r += stride) accumulate(load_chunk(Y, r, M, c, vec));
    }
    chunk_allreduce<CHP>(s1);
    chunk_allreduce<CHP>(s2);
    if (lane < CHP) {
        const int c0 = 4 * c;
        red[w][c0] = s1.x; red[w][c0 + 1] = s1.y; red[w][c0 + 2] = s1.z; red[w][c0 + 3] = s1.w;
        red[w][4 * CHP + c0] = s2.x; red[w][4 * CHP + c0 + 1] = s2.y; red[w][4 * CHP + c0 + 2] = s2.z; red[w][4 * CHP + c0 + 3] = s2.w;
    }
    __shared__ float shift_s[4 * CHP];
    if (r0 == 0) { shift_s[4 * c] = a4.x; shift_s[4 * c + 1] = a4.y; shift_s[4 * c + 2] = a4.z; shift_s[4 * c + 3] = a4.w; }
    __syncthreads();
    // rows this CTA saw: its row groups are blockIdx.x, blockIdx.x + G, ...; only the last group of the matrix may be short
    const int64_t groups = (N + RP - 1) / RP, G = gridDim.x;
    const int64_t mine = (groups - 1 - blockIdx.x) / G + 1;
    int64_t n_rows = mine * RP;
    if ((groups - 1) % G == blockIdx.x) n_rows -= groups * RP - N;
    for (int i = t; i < MP; i += 256) {
        float S1 = 0.f, S2 = 0.f;
        if (i < 4 * CHP && i < M) {
#pragma unroll
            for (int ww = 0; ww < 8; ++ww) { S1 += red[ww][i]; S2 += red[ww][4 * CHP + i]; }
            part[static_cast<size_t>(blockIdx.x) * MP + i] = make_float4(static_cast<float>(n_rows), shift_s[i], S1, S2);
        } else {
            part[static_cast<size_t>(blockIdx.x) * MP + i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

template <int CHP>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const float *__restrict__ G, const float *__restrict__ Y, int64_t N, int M,
                                                           const float *__restrict__ bn, const float *__restrict__ sums, int act,
                                                           float slope, float *__restrict__ GX) {
    constexpr int RP = 256 / CHP;
    const int t = threadIdx.x, c = t % CHP, r0 = t / CHP;
    if (4 * c >= M) return;
    const bool vec = (M % 4 == 0) && aligned16_dev(G) && aligned16_dev(Y) && aligned16_dev(GX);
    const Bn4 b = load_bn4(bn, M, c);
    const float invN = 1.f / static_cast<float>(N);
    const float4 s1 = load_vec4(sums, M, c), s2 = load_vec4(sums + M, M, c);
    const float4 m1 = make_float4(s1.x * invN, s1.y * invN, s1.z * invN, s1.w * invN);
    const float4 m2 = make_float4(s2.x * invN, s2.y * invN, s2.z * invN, s2.w * invN);
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * RP + r0; r < N; r += static_cast<int64_t>(gridDim.x) * RP) {
        float4 g = load_chunk(G, r, M, c, vec);
        const float4 y = load_chunk(Y, r, M, c, vec);
        const float4 xc = make_float4(y.x - b.mean.x, y.y - b.mean.y, y.z - b.mean.z, y.w - b.mean.w);
        g.x *= dact_f(fmaf(xc.x, b.k.x, b.beta.x), act, slope); g.y *= dact_f(fmaf(xc.y, b.k.y, b.beta.y), act, slope);
        g.z *= dact_f(fmaf(xc.z, b.k.z, b.beta.z), act, slope); g.w *= dact_f(fmaf(xc.w, b.k.w, b.beta.w), act, slope);
        float4 o;
        o.x = b.k.x * (g.x - m1.x - xc.x * b.rstd.x * m2.x); o.y = b.k.y * (g.y - m1.y - xc.y * b.rstd.y * m2.y);
        o.z = b.k.z * (g.z - m1.z - xc.z * b.rstd.z * m2.z); o.w = b.k.w * (g.w - m1.w - xc.w * b.rstd.w * m2.w);
        store_chunk(GX, r, M, c, o, vec);
    }
}

// fixed-order dot product: per-CTA partial (tree in shared memory), the last CTA adds the partials in index order
__global__ void __launch_bounds__(256) dot_kernel(const float *__restrict__ a, const float *__restrict__ b, int64_t n,
                                                  float *__restrict__ out, float *__restrict__ part, int *counter) {
    __shared__ float red[256];
    __shared__ int is_last;
    const int t = threadIdx.x;
    const bool vec = aligned16_dev(a) && aligned16_dev(b);
    float s = 0.f;
    if (vec) {
        const int64_t n4 = n / 4;
        const float4 *a4 = reinterpret_cast<const float4 *>(a), *b4 = reinterpret_cast<const float4 *>(b);
        const int64_t stride = gridDim.x * 256ll;
        int64_t i = blockIdx.x * 256ll + t;
        for (; i + 3 * stride < n4; i += 4 * stride) {      // eight independent 128-bit loads in flight, same add order
            float4 u[4], v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) { u[k] = __ldg(a4 + i + k * stride); v[k] = __ldg(b4 + i + k * stride); }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                s = fmaf(u[k].x, v[k].x, s); s = fmaf(u[k].y, v[k].y, s); s = fmaf(u[k].z, v[k].z, s); s = fmaf(u[k].w, v[k].w, s);
            }
        }
        for (; i < n4; i += stride) {
            const float4 u = __ldg(a4 + i), v = __ldg(b4 + i);
            s = fmaf(u.x, v.x, s); s = fmaf(u.y, v.y, s); s = fmaf(u.z, v.z, s); s = fmaf(u.w, v.w, s);
        }
        for (int64_t i = n4 * 4 + blockIdx.x * 256ll + t; i < n; i += gridDim.x * 256ll) s = fmaf(__ldg(a + i), __ldg(b + i), s);
    } else {
        for (int64_t i = blockIdx.x * 256ll + t; i < n; i += gridDim.x * 256ll) s = fmaf(__ldg(a + i), __ldg(b + i), s);
    }
    red[t] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (t < o) red[t] += red[t + o];
        __syncthreads();
    }
    if (t == 0) {
        part[blockIdx.x] = red[0];
        __threadfence();
        is_last = (atomicAdd(counter, 1) == static_cast<int>(gridDim.x) - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        __shared__ double dred[256];
        double tot = 0.0;
        for (int i = t; i < static_cast<int>(gridDim.x); i += 256) tot += static_cast<double>(__ldcg(part + i));
        dred[t] = tot;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (t < o) dred[t] += dred[t + o];
            __syncthreads();
        }
        if (t == 0) {
            out[0] = static_cast<float>(dred[0]);
            *counter = 0;
        }
    }
}

constexpr int pad32(int x) { return x <= 32 ? 32 : (x <= 64 ? 64 : 128); }   // padded channel counts: whole power-of-two panels

constexpr int RING_FWD = 3, RING_BWD = 2;
constexpr size_t fwd_smem_c(int KP, int MP, int ring) {
    return 1024 + 2 * (KP / 32) * 16384 + 2 * (KP / 32) * MP * 128 + static_cast<size_t>(ring) * 128 * KP * 4;
}
constexpr size_t bwd_smem_c(int KP, int MP, int ring) {
    return 1024 + 4 * (MP / 32) * 16384 + 2 * (KP / 32) * 16384 + 2 * (KP / 32) * MP * 128 + static_cast<size_t>(ring) * 128 * (2 * MP + KP) * 4 +
           (KP * MP <= 32 * 64 ? 16u * MP * KP : 0u);
}
constexpr size_t SMEM_CAP = 227 * 1024 - 4096;     // dynamic shared memory a CTA may ask for (static part + slack kept back)
size_t fwd_smem(int KP, int MP, int ring) {
    return 1024 + 2 * (KP / 32) * PANEL128 + 2 * (KP / 32) * MP * 128 + static_cast<size_t>(ring) * 128 * KP * 4;
}
size_t bwd_smem(int KP, int MP, int ring) {
    return 1024 + 4 * (MP / 32) * PANEL128 + 2 * (KP / 32) * PANEL128 + 2 * (KP / 32) * MP * 128 +
           static_cast<size_t>(ring) * 128 * (2 * MP + KP) * 4 + (bwd_accw_smem(KP, MP) ? 16u * MP * KP : 0u);
}
int ctas_per_sm(size_t smem, int tmem_cols, int threads) {
    int n = static_cast<int>((227 * 1024) / (smem + 2048));
    const int by_tmem = 512 / tmem_cols, by_threads = 1024 / threads;
    if (n > by_tmem) n = by_tmem;
    if (n > by_threads) n = by_threads;
    return n < 1 ? 1 : (n > 4 ? 4 : n);
}
int tc_grid(int64_t N, size_t smem, int tmem_cols, int threads) {
    const int64_t tiles = ceil_div64(N, 128);
    const int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * ctas_per_sm(smem, tmem_cols, threads);
    return static_cast<int>(tiles < cap ? tiles : cap);
}

constexpr int NT_FWD = 256, NT_BWD = 512;
template <int KP, int MP, int RING>
int launch_fwd(const LinFwdArgs &a, int *grid_out, cudaStream_t s) {
    const size_t smem = fwd_smem(KP, MP, RING);
    const int grid = tc_grid(a.N, smem, (TC_SPLIT_ACC < KP / 16 ? TC_SPLIT_ACC : KP / 16) * 2 * MP, NT_FWD);
    DN_CUDA(cudaFuncSetAttribute(lin_fwd_kernel<KP, MP, RING, NT_FWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    lin_fwd_kernel<KP, MP, RING, NT_FWD><<<grid, NT_FWD, smem, s>>>(a);
    *grid_out = grid;
    return 0;
}
template <int KP, int MP, int RING>
int launch_bwd(const LinBwdArgs &a, int *grid_out, cudaStream_t s) {
    const size_t smem = bwd_smem(KP, MP, RING);
    constexpr int nacc_d = (MP >= 64 && TC_SPLIT_ACC < 2) ? 2 : TC_SPLIT_ACC;
    constexpr int cols = (nacc_d + TC_SPLIT_ACC) * 2 * KP;
    const int grid = tc_grid(a.N, smem, cols <= 128 ? 128 : (cols <= 256 ? 256 : 512), NT_BWD);
    DN_CUDA(cudaFuncSetAttribute(lin_bwd_kernel<KP, MP, RING, NT_BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    lin_bwd_kernel<KP, MP, RING, NT_BWD><<<grid, NT_BWD, smem, s>>>(a);
    *grid_out = grid;
    return 0;
}
// the raw ring needs 16-byte slabs (row length a multiple of 4 floats, aligned bases) and room in shared memory
template <int KP, int MP>
int dispatch_fwd(const LinFwdArgs &a, bool ring_ok, int *grid_out, cudaStream_t s) {
    if constexpr (fwd_smem_c(KP, MP, RING_FWD) <= SMEM_CAP) {
        if (ring_ok) return launch_fwd<KP, MP, RING_FWD>(a, grid_out, s);
    }
    return launch_fwd<KP, MP, 0>(a, grid_out, s);
}
template <int KP, int MP>
int dispatch_bwd(const LinBwdArgs &a, bool ring_ok, int *grid_out, cudaStream_t s) {
    if constexpr (bwd_smem_c(KP, MP, RING_BWD) <= SMEM_CAP) {
        if (ring_ok) return launch_bwd<KP, MP, RING_BWD>(a, grid_out, s);
    }
    return launch_bwd<KP, MP, 0>(a, grid_out, s);
}

}  // namespace

extern "C" {

int32_t dn4gl_lin_supported(int32_t K, int32_t M) { return (K >= 1 && M >= 1 && K <= 64 && M <= 64) ? 1 : 0; }

size_t dn4gl_lin_workspace_bytes(int64_t N, int32_t K, int32_t M) {
    if (!dn4gl_lin_supported(K, M)) return 0;
    const int KP = pad32(K), MP = pad32(M);
    const size_t ctas = static_cast<size_t>(dn4gl_num_sms()) * 4;
    const size_t fwd = ctas * MP * 4 * sizeof(float);
    const size_t bwd = ctas * static_cast<size_t>(bwd_part_floats(KP, MP)) * sizeof(float);
    (void)N;
    const size_t pipe = dn4gl_pipe_lin_bwd_ws_bytes(K, M);
    const size_t m = fwd > bwd ? fwd : bwd;
    return align_up(m > pipe ? m : pipe, 256);
}

int dn4gl_lin_fwd_f32(const float *X, int64_t N, int32_t K, const float *in_bn, int32_t in_act, float in_slope,
                      const float *W, const float *bias, int32_t M, float *Y,
                      const float *gamma, const float *beta, float eps, float momentum, float *bn_out,
                      float *running_mean, float *running_var, int64_t *num_batches_tracked,
                      void *ws, size_t ws_bytes, int32_t *counters, void *stream) {
    DN_ARG(N >= 0 && X != nullptr && W != nullptr && Y != nullptr);
    DN_ARG(dn4gl_lin_supported(K, M));
    DN_ARG(in_act >= DN4GL_ACT_NONE && in_act <= DN4GL_ACT_LEAKY_RELU);
    DN_ARG(bn_out == nullptr || (ws != nullptr && ws_bytes >= dn4gl_lin_workspace_bytes(N, K, M)));
    if (N == 0) return DN4GL_OK;
    DN_ARG(N < (static_cast<int64_t>(1) << 31) * 128);
    const int KP = pad32(K), MP = pad32(M);
    LinFwdArgs a;
    a.X = X; a.N = N; a.K = K; a.in_bn = in_bn; a.in_act = in_act; a.in_slope = in_slope;
    a.W = W; a.bias = bias; a.M = M; a.Y = Y;
    a.stats = bn_out != nullptr ? 1 : 0;
    a.part = static_cast<float *>(ws);
    a.num_tiles = static_cast<int>(ceil_div64(N, 128));
    cudaStream_t s = as_stream(stream);
    const bool ring_ok = (K % 4 == 0) && aligned16(X);
    int rc = 0, grid = 0;
    // warp-specialised pipeline (mlp_pipe.cu) whenever the slabs are 16-byte granular; it also merges the batch statistics
    // after a grid rendezvous (no bn_finalize launch)
    if ((M % 4 == 0) && aligned16(Y) && (bn_out == nullptr || counters != nullptr)) {
        a.x_direct = (ring_ok && aligned16(W)) ? 0 : 1;     // e.g. the 2-feature first layer: X / W through bounds-checked loads
        BnFinalArgs f;
        f.gamma = gamma; f.beta = beta; f.eps = eps; f.momentum = momentum; f.bn_out = bn_out;
        f.run_mean = running_mean; f.run_var = running_var; f.nbt = reinterpret_cast<long long *>(num_batches_tracked);
        const int g = dn4gl_pipe_lin_fwd(a, f, counters, s);
        if (g < 0) { dn4gl_set_error("dn4gl_lin_fwd_f32: launch configuration of the pipelined kernel failed"); return DN4GL_ECUDA; }
        if (g > 0) { DN_LAUNCHED(); return DN4GL_OK; }
    }
#define DN_FWD_CASE(kp, mp) if (KP == kp && MP == mp) rc = dispatch_fwd<kp, mp>(a, ring_ok, &grid, s); else
    DN_FWD_CASE(32, 32) DN_FWD_CASE(32, 64) DN_FWD_CASE(64, 32) DN_FWD_CASE(64, 64)
    { dn4gl_set_error("dn4gl_lin_fwd_f32: no instantiation for K=%d M=%d", K, M); return DN4GL_EINVAL; }
#undef DN_FWD_CASE
    if (rc) return rc;
    if (bn_out != nullptr) {
        bn_finalize_kernel<<<MP / 32, 1024, 0, s>>>(reinterpret_cast<const float4 *>(a.part), grid, MP, M, N, gamma, beta, eps,
                                                    momentum, bn_out, running_mean, running_var,
                                                    reinterpret_cast<long long *>(num_batches_tracked));
        DN_LAUNCHED_N(2);
    } else {
        DN_LAUNCHED();
    }
    return DN4GL_OK;
}

int dn4gl_lin_bwd_f32(const float *G, const float *Gseg, const int32_t *row2seg, const float *Yout, int64_t N, int32_t M,
                      const float *bn, const float *sums, int32_t g_masked,
                      const float *W, int32_t K,
                      const float *X, const float *in_bn, int32_t in_act, float in_slope,
                      float *GX, float *sums_prev, float *dW, float *db,
                      void *ws, size_t ws_bytes, int32_t *counters, void *stream) {
    DN_ARG(N >= 0 && (G != nullptr || Gseg != nullptr) && W != nullptr && X != nullptr && ws != nullptr);
    DN_ARG((Gseg == nullptr) == (row2seg == nullptr));
    DN_ARG(dn4gl_lin_supported(K, M));
    DN_ARG(bn == nullptr || (Yout != nullptr && sums != nullptr));
    DN_ARG(sums_prev == nullptr || in_bn != nullptr);
    DN_ARG(in_act >= DN4GL_ACT_NONE && in_act <= DN4GL_ACT_LEAKY_RELU);
    DN_ARG(ws_bytes >= dn4gl_lin_workspace_bytes(N, K, M));
    const int KP = pad32(K), MP = pad32(M);
    // the canonical layouts used here need MP and KP to be whole 32-float panels and tcgen05 needs N % 16 == 0
    cudaStream_t s = as_stream(stream);
    if (N == 0) {
        if (dW) DN_CUDA(cudaMemsetAsync(dW, 0, sizeof(float) * M * K, s));
        if (db) DN_CUDA(cudaMemsetAsync(db, 0, sizeof(float) * M, s));
        if (sums_prev) DN_CUDA(cudaMemsetAsync(sums_prev, 0, sizeof(float) * 2 * K, s));
        return DN4GL_OK;
    }
    LinBwdArgs a;
    a.G = G; a.Gseg = Gseg; a.row2seg = row2seg; a.Yo = Yout; a.N = N; a.M = M; a.bn = bn; a.sums = sums; a.g_masked = g_masked;
    a.W = W; a.K = K; a.X = X; a.in_bn = in_bn; a.in_act = in_act; a.in_slope = in_slope;
    a.GX = GX; a.part = static_cast<float *>(ws);
    a.num_tiles = static_cast<int>(ceil_div64(N, 128));
    const bool ring_ok = (K % 4 == 0) && (M % 4 == 0) && aligned16(X) && (G == nullptr || aligned16(G)) && (Yout == nullptr || aligned16(Yout));
    int rc = 0, grid = 0;
    // warp-specialised pipeline, partials merged after a grid rendezvous (mlp_pipe.cu): no lin_bwd_reduce launch
    const bool gy_ok = (M % 4 == 0) && (G == nullptr || aligned16(G)) && (Yout == nullptr || aligned16(Yout));
    const bool x_ok = (K % 4 == 0) && aligned16(X) && aligned16(W);
    if (gy_ok && counters != nullptr && (x_ok || GX == nullptr) && (GX == nullptr || aligned16(GX)) &&
        (Gseg == nullptr || (aligned16(Gseg) && aligned16(row2seg)))) {
        a.x_direct = x_ok ? 0 : 1;
        const int g = dn4gl_pipe_lin_bwd(a, dW, db, sums_prev, ws, counters, s);
        if (g < 0) { dn4gl_set_error("dn4gl_lin_bwd_f32: launch configuration of the pipelined kernel failed"); return DN4GL_ECUDA; }
        if (g > 0) { DN_LAUNCHED(); return DN4GL_OK; }
    }
#define DN_BWD_CASE(kp, mp) if (KP == kp && MP == mp) rc = dispatch_bwd<kp, mp>(a, ring_ok, &grid, s); else
    DN_BWD_CASE(32, 32) DN_BWD_CASE(32, 64) DN_BWD_CASE(64, 32) DN_BWD_CASE(64, 64)
    { dn4gl_set_error("dn4gl_lin_bwd_f32: no instantiation for K=%d M=%d", K, M); return DN4GL_EINVAL; }
#undef DN_BWD_CASE
    if (rc) return rc;
    const int elems = MP * KP + MP + 2 * KP;
    lin_bwd_reduce_kernel<<<(elems + 31) / 32, 1024, 0, s>>>(a.part, grid, MP, KP, M, K, dW, db, sums_prev);
    DN_LAUNCHED_N(2);
    return DN4GL_OK;
}

int dn4gl_bn_act_f32(const float *Y, int64_t N, int32_t M, const float *bn, int32_t act, float slope, float *out,
                     void *stream) {
    DN_ARG(N >= 0 && M >= 1 && Y != nullptr && out != nullptr);
    DN_ARG(act >= DN4GL_ACT_NONE && act <= DN4GL_ACT_LEAKY_RELU);
    if (N == 0) return DN4GL_OK;
    const int64_t total = N * ((M + 3) / 4);
    const int64_t want = ceil_div64(total, 256 * 4);
    const int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * 8;
    bn_act_kernel<<<static_cast<int>(want < cap ? want : cap), 256, 0, as_stream(stream)>>>(Y, N, M, bn, act, slope, out);
    DN_LAUNCHED();
    return DN4GL_OK;
}

int dn4gl_bn_act_pool_f32(const float *Y, int64_t N, int32_t M, const float *bn, int32_t act, float slope, float *out,
                          const int32_t *seg_ptr, int32_t B, int32_t mode, float *pooled, void *stream) {
    DN_ARG(N >= 0 && M >= 1 && M <= 128 && B >= 0 && (mode == 0 || mode == 1));
    DN_ARG(act >= DN4GL_ACT_NONE && act <= DN4GL_ACT_LEAKY_RELU);
    if (B == 0) return DN4GL_OK;
    DN_ARG(Y != nullptr && out != nullptr && seg_ptr != nullptr && pooled != nullptr);
    const int CH = (M + 3) / 4;
    int CHP = 1;
    while (CHP < CH) CHP <<= 1;
    const int cap = dn4gl_num_sms() * 8;
    const int grid = B < cap ? B : cap;
    cudaStream_t s = as_stream(stream);
    switch (CHP) {
    case 1: bn_act_pool_kernel<1><<<grid, 256, 0, s>>>(Y, M, bn, act, slope, out, seg_ptr, B, mode, pooled); break;
    case 2: bn_act_pool_kernel<2><<<grid, 256, 0, s>>>(Y, M, bn, act, slope, out, seg_ptr, B, mode, pooled); break;
    case 4: bn_act_pool_kernel<4><<<grid, 256, 0, s>>>(Y, M, bn, act, slope, out, seg_ptr, B, mode, pooled); break;
    case 8: bn_act_pool_kernel<8><<<grid, 256, 0, s>>>(Y, M, bn, act, slope, out, seg_ptr, B, mode, pooled); break;
    case 16: bn_act_pool_kernel<16><<<grid, 256, 0, s>>>(Y, M, bn, act, slope, out, seg_ptr, B, mode, pooled); break;
    default: bn_act_pool_kernel<32><<<grid, 256, 0, s>>>(Y, M, bn, act, slope, out, seg_ptr, B, mode, pooled); break;
    }
    DN_LAUNCHED();
    return DN4GL_OK;
}

int dn4gl_segment_ids_i32(const int32_t *seg_ptr, int32_t B, int64_t N, int32_t *out, void *stream) {
    DN_ARG(B >= 0 && N >= 0);
    if (N == 0) return DN4GL_OK;
    DN_ARG(seg_ptr != nullptr && out != nullptr && B >= 1);
    segment_ids_kernel<<<static_cast<unsigned>(ceil_div64(N, 256)), 256, 0, as_stream(stream)>>>(seg_ptr, B, N, out);
    DN_LAUNCHED();
    return DN4GL_OK;
}

size_t dn4gl_dot_workspace_bytes(int64_t n) {
    (void)n;
    return static_cast<size_t>(dn4gl_num_sms()) * 4 * sizeof(float);
}

int dn4gl_dot_f32(const float *a, const float *b, int64_t n, float *out, void *ws, size_t ws_bytes, int32_t *counter,
                  void *stream) {
    DN_ARG(n >= 0 && a != nullptr && b != nullptr && out != nullptr && ws != nullptr && counter != nullptr);
    DN_ARG(ws_bytes >= dn4gl_dot_workspace_bytes(n));
    const int64_t want = ceil_div64(n > 0 ? n : 1, 256 * 16);
    const int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * 4;
    dot_kernel<<<static_cast<int>(want < cap ? want : cap), 256, 0, as_stream(stream)>>>(a, b, n, out, static_cast<float *>(ws), counter);
    DN_LAUNCHED();
    return DN4GL_OK;
}

size_t dn4gl_bn_bwd_sums_workspace_bytes(int64_t N, int32_t M) {
    (void)N;
    (void)M;
    return static_cast<size_t>(dn4gl_num_sms()) * 4 * 8 * 32 * sizeof(float);
}

int dn4gl_bn_bwd_sums_f32(const float *G, const float *Gseg, const int32_t *row2seg, const float *Y, int64_t N, int32_t M,
                          const float *bn, int32_t act, float slope, float *sums, void *ws, size_t ws_bytes, int32_t *counters,
                          void *stream) {
    DN_ARG(N >= 0 && M >= 1 && M <= 128 && (G != nullptr || Gseg != nullptr) && Y != nullptr && bn != nullptr && sums != nullptr && ws != nullptr);
    DN_ARG((Gseg == nullptr) == (row2seg == nullptr) && counters != nullptr);
    DN_ARG(ws_bytes >= dn4gl_bn_bwd_sums_workspace_bytes(N, M));
    cudaStream_t s = as_stream(stream);
    if (N == 0) { DN_CUDA(cudaMemsetAsync(sums, 0, sizeof(float) * 2 * M, s)); return DN4GL_OK; }
    const int CH = (M + 3) / 4;
    int CHP = 1;
    while (CHP < CH) CHP <<= 1;
    const int RP = 256 / CHP;
    const int64_t want = ceil_div64(N, static_cast<int64_t>(RP) * 8);
    int occ = 0;        // resident CTAs per SM of this instantiation (the cooperative launch refuses a larger grid)
    switch (CHP) {
    case 1: DN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bn_bwd_sums_kernel<1>, 256, 0)); break;
    case 2: DN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bn_bwd_sums_kernel<2>, 256, 0)); break;
    case 4: DN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bn_bwd_sums_kernel<4>, 256, 0)); break;
    case 8: DN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bn_bwd_sums_kernel<8>, 256, 0)); break;
    case 16: DN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bn_bwd_sums_kernel<16>, 256, 0)); break;
    default: DN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bn_bwd_sums_kernel<32>, 256, 0)); break;
    }
    const int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * (occ < 1 ? 1 : (occ > 4 ? 4 : occ));
    const int grid = static_cast<int>(want < cap ? (want < 1 ? 1 : want) : cap);
    float *part = static_cast<float *>(ws);
    // cooperative: the merge of the per-CTA partials rendezvouses the grid (4 CTAs of 256 threads per SM are resident)
    cudaError_t rc;
    switch (CHP) {
    case 1: rc = launch_coop(bn_bwd_sums_kernel<1>, grid, 256, 0, s, G, Gseg, row2seg, Y, N, M, bn, act, slope, part, sums, counters); break;
    case 2: rc = launch_coop(bn_bwd_sums_kernel<2>, grid, 256, 0, s, G, Gseg, row2seg, Y, N, M, bn, act, slope, part, sums, counters); break;
    case 4: rc = launch_coop(bn_bwd_sums_kernel<4>, grid, 256, 0, s, G, Gseg, row2seg, Y, N, M, bn, act, slope, part, sums, counters); break;
    case 8: rc = launch_coop(bn_bwd_sums_kernel<8>, grid, 256, 0, s, G, Gseg, row2seg, Y, N, M, bn, act, slope, part, sums, counters); break;
    case 16: rc = launch_coop(bn_bwd_sums_kernel<16>, grid, 256, 0, s, G, Gseg, row2seg, Y, N, M, bn, act, slope, part, sums, counters); break;
    default: rc = launch_coop(bn_bwd_sums_kernel<32>, grid, 256, 0, s, G, Gseg, row2seg, Y, N, M, bn, act, slope, part, sums, counters); break;
    }
    DN_CUDA(rc);
    DN_LAUNCHED();
    return DN4GL_OK;
}

static int bn_chp(int M) {
    const int CH = (M + 3) / 4;
    int CHP = 1;
    while (CHP < CH) CHP <<= 1;
    return CHP;
}

size_t dn4gl_bn_stats_workspace_bytes(int64_t N, int32_t M) {
    (void)N;
    const size_t MP = (static_cast<size_t>(M) + 31) / 32 * 32;
    return static_cast<size_t>(dn4gl_num_sms()) * 4 * MP * sizeof(float4);
}

int dn4gl_bn_stats_f32(const float *Y, int64_t N, int32_t M, const float *gamma, const float *beta, float eps, float momentum,
                       float *running_mean, float *running_var, int64_t *num_batches_tracked, float *bn_out, void *ws,
                       size_t ws_bytes, void *stream) {
    DN_ARG(N >= 1 && M >= 1 && M <= 128 && Y != nullptr && bn_out != nullptr && ws != nullptr);
    DN_ARG(ws_bytes >= dn4gl_bn_stats_workspace_bytes(N, M));
    cudaStream_t s = as_stream(stream);
    const int CHP = bn_chp(M), RP = 256 / CHP, MP = (M + 31) / 32 * 32;
    const int64_t groups = ceil_div64(N, RP), want = ceil_div64(groups, 8), cap = static_cast<int64_t>(dn4gl_num_sms()) * 4;
    const int grid = static_cast<int>(want < cap ? (want < 1 ? 1 : want) : cap);       // <= groups: every CTA has a first row
    float4 *part = static_cast<float4 *>(ws);
    switch (CHP) {
    case 1: bn_stats_partial_kernel<1><<<grid, 256, 0, s>>>(Y, N, M, MP, part); break;
    case 2: bn_stats_partial_kernel<2><<<grid, 256, 0, s>>>(Y, N, M, MP, part); break;
    case 4: bn_stats_partial_kernel<4><<<grid, 256, 0, s>>>(Y, N, M, MP, part); break;
    case 8: bn_stats_partial_kernel<8><<<grid, 256, 0, s>>>(Y, N, M, MP, part); break;
    case 16: bn_stats_partial_kernel<16><<<grid, 256, 0, s>>>(Y, N, M, MP, part); break;
    default: bn_stats_partial_kernel<32><<<grid, 256, 0, s>>>(Y, N, M, MP, part); break;
    }
    bn_finalize_kernel<<<MP / 32, 1024, 0, s>>>(reinterpret_cast<const float4 *>(part), grid, MP, M, N, gamma, beta, eps, momentum,
                                                bn_out, running_mean, running_var, reinterpret_cast<long long *>(num_batches_tracked));
    DN_LAUNCHED_N(2);
    return DN4GL_OK;
}

int dn4gl_bn_bwd_apply_f32(const float *G, const float *Y, int64_t N, int32_t M, const float *bn, const float *sums, int32_t act,
                           float slope, float *GX, void *stream) {
    DN_ARG(N >= 0 && M >= 1 && M <= 128);
    if (N == 0) return DN4GL_OK;
    DN_ARG(G != nullptr && Y != nullptr && bn != nullptr && sums != nullptr && GX != nullptr);
    cudaStream_t s = as_stream(stream);
    const int CHP = bn_chp(M), RP = 256 / CHP;
    const int64_t want = ceil_div64(N, static_cast<int64_t>(RP) * 4), cap = static_cast<int64_t>(dn4gl_num_sms()) * 8;
    const int grid = static_cast<int>(want < cap ? (want < 1 ? 1 : want) : cap);
    switch (CHP) {
    case 1: bn_bwd_apply_kernel<1><<<grid, 256, 0, s>>>(G, Y, N, M, bn, sums, act, slope, GX); break;
    case 2: bn_bwd_apply_kernel<2><<<grid, 256, 0, s>>>(G, Y, N, M, bn, sums, act, slope, GX); break;
    case 4: bn_bwd_apply_kernel<4><<<grid, 256, 0, s>>>(G, Y, N, M, bn, sums, act, slope, GX); break;
    case 8: bn_bwd_apply_kernel<8><<<grid, 256, 0, s>>>(G, Y, N, M, bn, sums, act, slope, GX); break;
    case 16: bn_bwd_apply_kernel<16><<<grid, 256, 0, s>>>(G, Y, N, M, bn, sums, act, slope, GX); break;
    default: bn_bwd_apply_kernel<32><<<grid, 256, 0, s>>>(G, Y, N, M, bn, sums, act, slope, GX); break;
    }
    DN_LAUNCHED();
    return DN4GL_OK;
}

}  // extern "C"
