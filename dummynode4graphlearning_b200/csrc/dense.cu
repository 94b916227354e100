// libdn4gl.so -- dense helpers of the per-node / per-edge MLPs.
//
// dn4gl_atb_f32:  C (Ka x Kb) = A^T B  with A (N x Ka), B (N x Kb), N = number of nodes / edges (1e4..1e7),
//                 ceil(Ka/4)*ceil(Kb/4) <= 256 (e.g. 64 x 64, 32 x 128); optionally colsum(A) (Ka).  This is the weight-gradient of every Linear
//                 (dW = G^T X, db = colsum G) and raw-parameter matmul (dW = X^T G) on the path.  Library SGEMMs
//                 treat it as a "large-K" GEMM with a tiny output and run at a few % of HBM bandwidth
//                 (profiles/r1a: sgemm_largek_lds64, 453 us for 40 MB); it is a REDUCTION over rows, so it is
//                 written as one: every CTA streams a contiguous slab of rows once (128-bit loads staged through
//                 shared memory), keeps its Ka x Kb partial in registers, and a second kernel adds the per-CTA
//                 partials in a fixed order (deterministic, no atomics).  fp32 FMA throughout: HBM-bound for
//                 Ka*Kb <= 64*64 (2*Ka*Kb / (4*(Ka+Kb)) flop/B <= 16).
#include "common.cuh"

constexpr int ATB_THREADS = 256;
constexpr int ATB_ROWS = 32;      // rows staged per iteration
constexpr int ATB_MAX_TILES = 256;  // (Ka/4) * (Kb/4) register tiles of 4 x 4 must fit one CTA

// Thread layout: GA x GB register tiles of 4 x 4 outputs, replicated over RS = 256 / (GA*GB) row slices; slice s
// accumulates staged rows r = s, s+RS, ...; the slices are summed through shared memory at the end (fixed order).
// Per staged row a thread issues two 128-bit shared loads for 16 FMAs.
__global__ void __launch_bounds__(ATB_THREADS)
atb_partial_kernel(const float *__restrict__ A, const float *__restrict__ B, int64_t N, int Ka, int Kb, int GA, int GB,
                   int64_t rows_per_cta, float *__restrict__ partial /* [grid][Ka*Kb + Ka] */) {
    extern __shared__ __align__(16) float smem[];
    const int PA = 4 * GA, PB = 4 * GB;
    float *sA = smem;                      // [ATB_ROWS][PA]
    float *sB = smem + ATB_ROWS * PA;      // [ATB_ROWS][PB]
    const int tiles = GA * GB, RS = ATB_THREADS / tiles;
    const int slice = threadIdx.x / tiles, t = threadIdx.x % tiles;
    const int ga = t / GB, gb = t % GB;
    const bool active = slice < RS;
    float acc[4][4];
    float colsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int64_t r_begin = static_cast<int64_t>(blockIdx.x) * rows_per_cta;
    const int64_t r_end = min(N, r_begin + rows_per_cta);
    const bool vecA = (Ka % 4 == 0), vecB = (Kb % 4 == 0);
    for (int64_t r0 = r_begin; r0 < r_end; r0 += ATB_ROWS) {
        const int64_t rem = r_end - r0;
        const int nr = rem < ATB_ROWS ? static_cast<int>(rem) : ATB_ROWS;
        // ---- stage rows (zero-padded to PA / PB columns and ATB_ROWS rows); 128-bit global loads when possible
        if (vecA) {
            for (int i = threadIdx.x; i < ATB_ROWS * GA; i += ATB_THREADS) {
                int r = i / GA, c = i % GA;
                float4 v = zero4();
                if (r < nr && 4 * c < Ka) v = ldg4(reinterpret_cast<const float4 *>(A + (r0 + r) * Ka) + c);
                reinterpret_cast<float4 *>(sA + r * PA)[c] = v;
            }
        } else {
            for (int i = threadIdx.x; i < ATB_ROWS * PA; i += ATB_THREADS) {
                int r = i / PA, c = i % PA;
                sA[r * PA + c] = (r < nr && c < Ka) ? __ldg(A + (r0 + r) * Ka + c) : 0.f;
            }
        }
        if (vecB) {
            for (int i = threadIdx.x; i < ATB_ROWS * GB; i += ATB_THREADS) {
                int r = i / GB, c = i % GB;
                float4 v = zero4();
                if (r < nr && 4 * c < Kb) v = ldg4(reinterpret_cast<const float4 *>(B + (r0 + r) * Kb) + c);
                reinterpret_cast<float4 *>(sB + r * PB)[c] = v;
            }
        } else {
            for (int i = threadIdx.x; i < ATB_ROWS * PB; i += ATB_THREADS) {
                int r = i / PB, c = i % PB;
                sB[r * PB + c] = (r < nr && c < Kb) ? __ldg(B + (r0 + r) * Kb + c) : 0.f;
            }
        }
        __syncthreads();
        if (active) {
            for (int r = slice; r < ATB_ROWS; r += RS) {
                const float4 a4 = reinterpret_cast<const float4 *>(sA + r * PA)[ga];
                const float4 b4 = reinterpret_cast<const float4 *>(sB + r * PB)[gb];
                const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    colsum[i] += a[i];
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
                }
            }
        }
        __syncthreads();
    }
    // ---- combine the RS slices in shared memory (ascending slice order), then write this CTA's partial
    float *red = smem;  // reuse: [RS][tiles][20]
    if (active) {
        float *mine = red + (static_cast<size_t>(slice) * tiles + t) * 20;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int j = 0; j < 4; ++j) mine[i * 4 + j] = acc[i][j];
            mine[16 + i] = colsum[i];
        }
    }
    __syncthreads();
    float *out = partial + static_cast<int64_t>(blockIdx.x) * (static_cast<int64_t>(Ka) * Kb + Ka);
    for (int idx = threadIdx.x; idx < tiles * 20; idx += ATB_THREADS) {
        int tt = idx / 20, e = idx % 20;
        float s = 0.f;
        for (int sl = 0; sl < RS; ++sl) s += red[(static_cast<size_t>(sl) * tiles + tt) * 20 + e];
        int tga = tt / GB, tgb = tt % GB;
        if (e < 16) {
            int ra = 4 * tga + e / 4, cb = 4 * tgb + e % 4;
            if (ra < Ka && cb < Kb) out[ra * Kb + cb] = s;
        } else if (tgb == 0) {
            int ra = 4 * tga + (e - 16);
            if (ra < Ka) out[static_cast<int64_t>(Ka) * Kb + ra] = s;
        }
    }
}

// C[i] = sum_p partial[p][i]: a CTA owns 32 outputs; its 8 warps stride the partials (coalesced 128-byte rows), each
// with 4 independent chains, and the 8 x 4 partial sums are combined in a fixed order (deterministic, no atomics)
__global__ void __launch_bounds__(256)
atb_reduce_kernel(const float *__restrict__ partial, int P, int KaKb, int Ka, float *__restrict__ C,
                  float *__restrict__ colsum) {
    __shared__ float red[8][33];
    const int o = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + o;
    const int total = KaKb + Ka;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (i < total) {
        int p = w;
        for (; p + 24 < P; p += 32) {
            s0 += partial[static_cast<int64_t>(p) * total + i];
            s1 += partial[static_cast<int64_t>(p + 8) * total + i];
            s2 += partial[static_cast<int64_t>(p + 16) * total + i];
            s3 += partial[static_cast<int64_t>(p + 24) * total + i];
        }
        for (; p < P; p += 8) s0 += partial[static_cast<int64_t>(p) * total + i];
    }
    red[w][o] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (w == 0 && i < total) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][o];
        if (i < KaKb) C[i] = s;
        else if (colsum) colsum[i - KaKb] = s;
    }
}

static int atb_grid(int64_t N) {
    int64_t want = ceil_div64(N, 4 * ATB_ROWS);  // at least 128 rows per CTA
    int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * 2;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return static_cast<int>(want);
}

extern "C" size_t dn4gl_atb_workspace_bytes(int64_t N, int32_t Ka, int32_t Kb) {
    return align_up(static_cast<size_t>(atb_grid(N)) * (static_cast<size_t>(Ka) * Kb + Ka) * sizeof(float), 256);
}

extern "C" int dn4gl_atb_f32(const float *A, const float *B, float *C, float *colsum_A, int64_t N, int32_t Ka,
                             int32_t Kb, void *ws, size_t ws_bytes, void *stream) {
    DN_ARG(N >= 0 && Ka > 0 && Kb > 0 && C != nullptr);
    DN_ARG(((Ka + 3) / 4) * ((Kb + 3) / 4) <= ATB_MAX_TILES);   // e.g. up to 64 x 64; larger shapes stay on the library GEMM
    DN_ARG(N == 0 || (A && B && aligned16(A) && aligned16(B)));
    cudaStream_t st = as_stream(stream);
    if (N == 0) {
        DN_CUDA(cudaMemsetAsync(C, 0, sizeof(float) * Ka * Kb, st));
        if (colsum_A) DN_CUDA(cudaMemsetAsync(colsum_A, 0, sizeof(float) * Ka, st));
        return DN4GL_OK;
    }
    if (ws == nullptr || ws_bytes < dn4gl_atb_workspace_bytes(N, Ka, Kb)) {
        dn4gl_set_error("dn4gl_atb_f32: workspace too small");
        return DN4GL_EWORKSPACE;
    }
    const int grid = atb_grid(N);
    const int64_t rows_per_cta = ceil_div64(ceil_div64(N, grid), ATB_ROWS) * ATB_ROWS;
    float *partial = static_cast<float *>(ws);
    const int GA = (Ka + 3) / 4, GB = (Kb + 3) / 4;
    const int RS = ATB_THREADS / (GA * GB);
    size_t smem = sizeof(float) * static_cast<size_t>(ATB_ROWS) * 4 * (GA + GB);
    const size_t red = sizeof(float) * static_cast<size_t>(RS) * GA * GB * 20;
    if (red > smem) smem = red;
    atb_partial_kernel<<<grid, ATB_THREADS, smem, st>>>(A, B, N, Ka, Kb, GA, GB, rows_per_cta, partial);
    const int total = Ka * Kb + Ka;
    atb_reduce_kernel<<<(total + 31) / 32, 256, 0, st>>>(partial, grid, Ka * Kb, Ka, C, colsum_A);
    DN_LAUNCHED_N(2);
    return DN4GL_OK;
}
