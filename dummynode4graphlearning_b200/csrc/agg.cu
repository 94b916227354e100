// libdn4gl.so -- K1 sum aggregation (CSR gather-sum), K3 segment readout / padding, label filter.
//
// Memory-bound kernels: every feature row moves as 128-bit (float4) accesses, a sub-group of
// LANES = min(32, D/4) lanes owns one output row so a warp covers 32/LANES rows with fully
// coalesced row segments; neighbour indices are broadcast loads; U independent row loads are
// issued before they are consumed (memory-level parallelism) but are ACCUMULATED IN CSR ORDER with
// separately rounded adds, so the result is bit-identical to a sequential scatter_add in edge-id
// order (the oracle) for every row handled by the per-row path.  Rows above the heavy threshold
// (dummy nodes: degree = graph size) are reduced by a whole CTA with a fixed-shape tree.
#include "common.cuh"

// -------------------------------------------------------------------------------------------
template <int LANES, int VEC>
__global__ void __launch_bounds__(256)
spmm_rows_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col, const float4 *__restrict__ x,
                 float4 *__restrict__ out, int64_t N, float self_scale, const float *__restrict__ eps_dev, int heavy_thr) {
    if (eps_dev != nullptr) self_scale = 1.f + __ldg(eps_dev);
    constexpr int ROWS = 256 / LANES;
    constexpr int U = (VEC == 1) ? 8 : (VEC == 2 ? 4 : 2);
    constexpr int DV = LANES * VEC;  // float4 per row
    const int64_t row = static_cast<int64_t>(blockIdx.x) * ROWS + threadIdx.x / LANES;
    const int lane = threadIdx.x % LANES;
    if (row >= N) return;
    const int beg = __ldg(row_ptr + row), end = __ldg(row_ptr + row + 1);
    if (heavy_thr > 0 && end - beg > heavy_thr) return;  // CTA-per-row kernel owns it
    float4 acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = zero4();
    int p = beg;
    for (; p + U <= end; p += U) {
        int c[U];
#pragma unroll
        for (int u = 0; u < U; ++u) c[u] = __ldg(col + p + u);
        float4 v[U][VEC];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < VEC; ++k) v[u][k] = ldg4(x + static_cast<int64_t>(c[u]) * DV + lane + k * LANES);
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < VEC; ++k) add4(acc[k], v[u][k]);
    }
    if (p < end) {  // tail: same shape, predicated
        int c[U];
        float4 v[U][VEC];
#pragma unroll
        for (int u = 0; u < U; ++u) c[u] = (p + u < end) ? __ldg(col + p + u) : -1;
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < VEC; ++k)
                if (c[u] >= 0) v[u][k] = ldg4(x + static_cast<int64_t>(c[u]) * DV + lane + k * LANES);
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < VEC; ++k)
                if (c[u] >= 0) add4(acc[k], v[u][k]);
    }
    if (self_scale != 0.f) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) axpy4_rn(acc[k], self_scale, ldg4(x + row * DV + lane + k * LANES));
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) out[row * DV + lane + k * LANES] = acc[k];
}

// one CTA (256 threads = SUBS sub-groups of LANES lanes) per heavy row; sub-group g takes items
// beg+g, beg+g+SUBS, ...; partials are combined in shared memory by a fixed binary tree.
template <int LANES, int VEC>
__global__ void __launch_bounds__(256)
spmm_heavy_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col, const float4 *__restrict__ x,
                  float4 *__restrict__ out, float self_scale, const float *__restrict__ eps_dev,
                  const int32_t *__restrict__ heavy_rows, const int32_t *__restrict__ heavy_count) {
    if (eps_dev != nullptr) self_scale = 1.f + __ldg(eps_dev);
    constexpr int SUBS = 256 / LANES;
    constexpr int DV = LANES * VEC;
    __shared__ float4 part[256 * VEC];
    const int sub = threadIdx.x / LANES, lane = threadIdx.x % LANES;
    const int n_heavy = *heavy_count;
    for (int h = blockIdx.x; h < n_heavy; h += gridDim.x) {
        const int64_t row = heavy_rows[h];
        const int beg = row_ptr[row], end = row_ptr[row + 1];
        float4 acc[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = zero4();
        int p = beg + sub;
        for (; p + 3 * SUBS < end; p += 4 * SUBS) {
            int c0 = __ldg(col + p), c1 = __ldg(col + p + SUBS), c2 = __ldg(col + p + 2 * SUBS),
                c3 = __ldg(col + p + 3 * SUBS);
            float4 v0[VEC], v1[VEC], v2[VEC], v3[VEC];
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                v0[k] = ldg4(x + static_cast<int64_t>(c0) * DV + lane + k * LANES);
                v1[k] = ldg4(x + static_cast<int64_t>(c1) * DV + lane + k * LANES);
                v2[k] = ldg4(x + static_cast<int64_t>(c2) * DV + lane + k * LANES);
                v3[k] = ldg4(x + static_cast<int64_t>(c3) * DV + lane + k * LANES);
            }
#pragma unroll
            for (int k = 0; k < VEC; ++k) { add4(acc[k], v0[k]); add4(acc[k], v1[k]); add4(acc[k], v2[k]); add4(acc[k], v3[k]); }
        }
        for (; p < end; p += SUBS) {
            int c0 = __ldg(col + p);
#pragma unroll
            for (int k = 0; k < VEC; ++k) add4(acc[k], ldg4(x + static_cast<int64_t>(c0) * DV + lane + k * LANES));
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) part[(sub * VEC + k) * LANES + lane] = acc[k];
        __syncthreads();
#pragma unroll
        for (int s = SUBS / 2; s >= 1; s >>= 1) {
            if (sub < s) {
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    float4 a = part[(sub * VEC + k) * LANES + lane];
                    add4(a, part[((sub + s) * VEC + k) * LANES + lane]);
                    part[(sub * VEC + k) * LANES + lane] = a;
                }
            }
            __syncthreads();
        }
        if (sub == 0) {
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                float4 a = part[k * LANES + lane];
                if (self_scale != 0.f) axpy4_rn(a, self_scale, ldg4(x + row * DV + lane + k * LANES));
                out[row * DV + lane + k * LANES] = a;
            }
        }
        __syncthreads();
    }
}

template <int LANES, int VEC>
static int launch_spmm(const int32_t *row_ptr, const int32_t *col, const float *x, float *out, int64_t N,
                       float self_scale, const float *eps_dev, const int32_t *heavy_rows, const int32_t *heavy_count,
                       int heavy_thr, cudaStream_t st) {
    constexpr int ROWS = 256 / LANES;
    const bool heavy = heavy_rows != nullptr && heavy_count != nullptr && heavy_thr > 0;
    spmm_rows_kernel<LANES, VEC><<<static_cast<unsigned>(ceil_div64(N, ROWS)), 256, 0, st>>>(
        row_ptr, col, reinterpret_cast<const float4 *>(x), reinterpret_cast<float4 *>(out), N, self_scale, eps_dev,
        heavy ? heavy_thr : 0);
    if (heavy) {
        spmm_heavy_kernel<LANES, VEC><<<dn4gl_num_sms() * 4, 256, 0, st>>>(
            row_ptr, col, reinterpret_cast<const float4 *>(x), reinterpret_cast<float4 *>(out), self_scale, eps_dev,
            heavy_rows, heavy_count);
    }
    return 0;
}

extern "C" int dn4gl_spmm_sum_f32(const int32_t *row_ptr, const int32_t *col, const float *x, float *out, int64_t N,
                                  int64_t n_src, int32_t D, float self_scale, const float *eps_dev, const int32_t *heavy_rows,
                                  const int32_t *heavy_count, int32_t heavy_threshold, void *stream) {
    DN_ARG(N >= 0 && n_src >= 0 && D > 0 && D % 4 == 0);
    if (N == 0) return DN4GL_OK;
    DN_ARG(row_ptr && x && out && aligned16(x) && aligned16(out));
    DN_ARG((self_scale == 0.f && eps_dev == nullptr) || n_src == N);
    cudaStream_t st = as_stream(stream);
    const int dv = D / 4;
#define SPMM_CASE(L, V)                                                                                       \
    launch_spmm<L, V>(row_ptr, col, x, out, N, self_scale, eps_dev, heavy_rows, heavy_count, heavy_threshold, st); \
    break
    switch (dv) {
        case 1: SPMM_CASE(1, 1);
        case 2: SPMM_CASE(2, 1);
        case 4: SPMM_CASE(4, 1);
        case 8: SPMM_CASE(8, 1);     // D = 32
        case 16: SPMM_CASE(16, 1);   // D = 64
        case 32: SPMM_CASE(32, 1);   // D = 128
        case 64: SPMM_CASE(32, 2);   // D = 256
        case 128: SPMM_CASE(32, 4);  // D = 512
        default:
            dn4gl_set_error("dn4gl_spmm_sum_f32: unsupported D=%d (supported: 4,8,16,32,64,128,256,512)", D);
            return DN4GL_EINVAL;
    }
#undef SPMM_CASE
    DN_LAUNCHED_N((heavy_rows != nullptr && heavy_count != nullptr && heavy_threshold > 0) ? 2 : 1);
    return DN4GL_OK;
}

// -------------------------------------------------------------------------------------------
// K3 segment readout: one CTA per segment, SUBS sub-groups stride the rows, tree-combine.
template <int LANES, int VEC>
__global__ void __launch_bounds__(256)
segment_sum_kernel(const int32_t *__restrict__ seg_ptr, const uint8_t *__restrict__ mask,
                   const float4 *__restrict__ x, float4 *__restrict__ out, int B, int mode) {
    constexpr int SUBS = 256 / LANES;
    constexpr int DV = LANES * VEC;
    __shared__ float4 part[256 * VEC];
    const int sub = threadIdx.x / LANES, lane = threadIdx.x % LANES;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const int beg = seg_ptr[b], end = seg_ptr[b + 1];
        float4 acc[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = zero4();
        for (int r = beg + sub; r < end; r += SUBS) {
            if (mask && mask[r]) continue;
#pragma unroll
            for (int k = 0; k < VEC; ++k) add4(acc[k], ldg4(x + static_cast<int64_t>(r) * DV + lane + k * LANES));
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) part[(sub * VEC + k) * LANES + lane] = acc[k];
        __syncthreads();
#pragma unroll
        for (int s = SUBS / 2; s >= 1; s >>= 1) {
            if (sub < s) {
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    float4 a = part[(sub * VEC + k) * LANES + lane];
                    add4(a, part[((sub + s) * VEC + k) * LANES + lane]);
                    part[(sub * VEC + k) * LANES + lane] = a;
                }
            }
            __syncthreads();
        }
        if (sub == 0) {
            float sc = 1.f;
            if (mode == 1) sc = 1.f / static_cast<float>(max(end - beg, 1));
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                float4 a = part[k * LANES + lane];
                if (mode == 1) { a.x *= sc; a.y *= sc; a.z *= sc; a.w *= sc; }
                out[static_cast<int64_t>(b) * DV + lane + k * LANES] = a;
            }
        }
        __syncthreads();
    }
}

// generic-width fallback (any D % 4 == 0, e.g. the 90/124-wide representation rows rounded up by
// the caller, or class-score widths): one warp per segment, lanes stride the float4 columns.
__global__ void __launch_bounds__(256)
segment_sum_generic(const int32_t *__restrict__ seg_ptr, const uint8_t *__restrict__ mask,
                    const float *__restrict__ x, float *__restrict__ out, int B, int D, int mode) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B) return;
    const int beg = seg_ptr[warp], end = seg_ptr[warp + 1];
    const float sc = (mode == 1) ? 1.f / static_cast<float>(max(end - beg, 1)) : 1.f;
    for (int c = lane; c < D; c += 32) {
        float acc = 0.f;
        for (int r = beg; r < end; ++r)
            if (!(mask && mask[r])) acc = __fadd_rn(acc, __ldg(x + static_cast<int64_t>(r) * D + c));
        out[static_cast<int64_t>(warp) * D + c] = (mode == 1) ? acc * sc : acc;
    }
}

// narrow rows (D <= 8, e.g. per-class scores pooled at gconv.py:210): one warp per segment, lanes stride the ROWS,
// every lane keeps all D column sums, fixed-shape shuffle tree at the end.
template <int DMAX>
__global__ void __launch_bounds__(256)
segment_sum_narrow(const int32_t *__restrict__ seg_ptr, const uint8_t *__restrict__ mask, const float *__restrict__ x,
                   float *__restrict__ out, int B, int D, int mode) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= B) return;
    const int beg = seg_ptr[warp], end = seg_ptr[warp + 1];
    float acc[DMAX];
#pragma unroll
    for (int c = 0; c < DMAX; ++c) acc[c] = 0.f;
    for (int r = beg + lane; r < end; r += 32) {
        if (mask && mask[r]) continue;
#pragma unroll
        for (int c = 0; c < DMAX; ++c)
            if (c < D) acc[c] = __fadd_rn(acc[c], __ldg(x + static_cast<int64_t>(r) * D + c));
    }
#pragma unroll
    for (int c = 0; c < DMAX; ++c)
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) acc[c] = __fadd_rn(acc[c], __shfl_xor_sync(0xffffffffu, acc[c], o));
    if (lane == 0) {
        const float sc = (mode == 1) ? 1.f / static_cast<float>(max(end - beg, 1)) : 1.f;
#pragma unroll
        for (int c = 0; c < DMAX; ++c)
            if (c < D) out[static_cast<int64_t>(warp) * D + c] = (mode == 1) ? acc[c] * sc : acc[c];
    }
}

extern "C" int dn4gl_segment_sum_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *x, float *out,
                                     int32_t B, int32_t D, int32_t mode, void *stream) {
    DN_ARG(B >= 0 && D > 0 && (mode == 0 || mode == 1));
    if (B == 0) return DN4GL_OK;
    DN_ARG(seg_ptr && x && out);
    cudaStream_t st = as_stream(stream);
    const unsigned grid = static_cast<unsigned>(B < dn4gl_num_sms() * 8 ? B : dn4gl_num_sms() * 8);
    const bool vec_ok = (D % 4 == 0) && aligned16(x) && aligned16(out);
    const int dv = vec_ok ? D / 4 : 0;
#define SEG_CASE(L, V)                                                                                       \
    segment_sum_kernel<L, V><<<grid, 256, 0, st>>>(seg_ptr, mask, reinterpret_cast<const float4 *>(x),       \
                                                   reinterpret_cast<float4 *>(out), B, mode);                \
    break
    switch (dv) {
        case 8: SEG_CASE(8, 1);
        case 16: SEG_CASE(16, 1);
        case 32: SEG_CASE(32, 1);
        case 64: SEG_CASE(32, 2);
        case 128: SEG_CASE(32, 4);
        default:
            if (D <= 8)
                segment_sum_narrow<8><<<static_cast<unsigned>(ceil_div64(static_cast<int64_t>(B) * 32, 256)), 256, 0, st>>>(
                    seg_ptr, mask, x, out, B, D, mode);
            else
                segment_sum_generic<<<static_cast<unsigned>(ceil_div64(static_cast<int64_t>(B) * 32, 256)), 256, 0, st>>>(
                    seg_ptr, mask, x, out, B, D, mode);
    }
#undef SEG_CASE
    DN_LAUNCHED();
    return DN4GL_OK;
}

__global__ void segment_bcast_kernel(const int32_t *__restrict__ seg_ptr, const uint8_t *__restrict__ mask,
                                     const float *__restrict__ g, float *__restrict__ gx, int B, int64_t N, int D,
                                     int mode) {
    int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= N * D) return;
    int64_t v = i / D;
    int c = static_cast<int>(i - v * D);
    if (mask && mask[v]) { gx[i] = 0.f; return; }
    int b = segment_of(seg_ptr, B, v);
    float val = __ldg(g + static_cast<int64_t>(b) * D + c);
    if (mode == 1) val *= 1.f / static_cast<float>(max(seg_ptr[b + 1] - seg_ptr[b], 1));
    gx[i] = val;
}

extern "C" int dn4gl_segment_bcast_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *g, float *gx,
                                       int32_t B, int64_t N, int32_t D, int32_t mode, void *stream) {
    DN_ARG(B >= 0 && N >= 0 && D > 0 && (mode == 0 || mode == 1));
    if (N == 0) return DN4GL_OK;
    DN_ARG(seg_ptr && g && gx);
    segment_bcast_kernel<<<static_cast<unsigned>(ceil_div64(N * D, 256)), 256, 0, as_stream(stream)>>>(
        seg_ptr, mask, g, gx, B, N, D, mode);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// -------------------------------------------------------------------------------------------
// left-padded batchify (utils/dl.py:51-81 with pre_pad=True) and its adjoint.
__global__ void pad_segments_kernel(const int32_t *__restrict__ seg_ptr, const uint8_t *__restrict__ mask,
                                    const float *__restrict__ x, float *__restrict__ out, int B, int Lmax, int D) {
    int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    int64_t total = static_cast<int64_t>(B) * Lmax * D;
    if (i >= total) return;
    int c = static_cast<int>(i % D);
    int64_t t = i / D;
    int l = static_cast<int>(t % Lmax);
    int b = static_cast<int>(t / Lmax);
    int beg = seg_ptr[b], len = seg_ptr[b + 1] - beg;
    int j = l - (Lmax - len);
    float v = 0.f;
    if (j >= 0) {
        int r = beg + j;
        if (!(mask && mask[r])) v = __ldg(x + static_cast<int64_t>(r) * D + c);
    }
    out[i] = v;
}

__global__ void unpad_segments_kernel(const int32_t *__restrict__ seg_ptr, const uint8_t *__restrict__ mask,
                                      const float *__restrict__ g, float *__restrict__ gx, int B, int Lmax, int D,
                                      int64_t N) {
    int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= N * D) return;
    int64_t r = i / D;
    int c = static_cast<int>(i - r * D);
    if (mask && mask[r]) { gx[i] = 0.f; return; }
    int b = segment_of(seg_ptr, B, r);
    int beg = seg_ptr[b], len = seg_ptr[b + 1] - beg;
    int l = (Lmax - len) + static_cast<int>(r - beg);
    gx[i] = __ldg(g + (static_cast<int64_t>(b) * Lmax + l) * D + c);
}

extern "C" int dn4gl_pad_segments_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *x, float *out,
                                      int32_t B, int32_t Lmax, int32_t D, void *stream) {
    DN_ARG(B >= 0 && Lmax >= 0 && D > 0);
    int64_t total = static_cast<int64_t>(B) * Lmax * D;
    if (total == 0) return DN4GL_OK;
    DN_ARG(seg_ptr && x && out);
    pad_segments_kernel<<<static_cast<unsigned>(ceil_div64(total, 256)), 256, 0, as_stream(stream)>>>(seg_ptr, mask, x,
                                                                                                      out, B, Lmax, D);
    DN_LAUNCHED();
    return DN4GL_OK;
}

extern "C" int dn4gl_unpad_segments_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *g, float *gx,
                                        int32_t B, int32_t Lmax, int32_t D, int64_t N, void *stream) {
    DN_ARG(B >= 0 && Lmax >= 0 && D > 0 && N >= 0);
    if (N == 0) return DN4GL_OK;
    DN_ARG(seg_ptr && g && gx);
    unpad_segments_kernel<<<static_cast<unsigned>(ceil_div64(N * D, 256)), 256, 0, as_stream(stream)>>>(
        seg_ptr, mask, g, gx, B, Lmax, D, N);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// -------------------------------------------------------------------------------------------
// ScalarFilter on left-padded label matrices (filter.py:10-16 via basemodel.py:830-847).
__global__ void label_filter_kernel(const int32_t *__restrict__ g_ptr, const int32_t *__restrict__ g_label,
                                    const int32_t *__restrict__ p_ptr, const int32_t *__restrict__ p_label, int B,
                                    int Lp_max, float *__restrict__ gate, int64_t Ng) {
    int64_t v = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (v >= Ng) return;
    int b = segment_of(g_ptr, B, v);
    int lab = g_label[v];
    int pb = p_ptr[b], pe = p_ptr[b + 1];
    bool hit = (pe - pb < Lp_max) && (lab == 0);  // zero padding of shorter patterns leaks into the match
    for (int j = pb; j < pe && !hit; ++j) hit = (p_label[j] == lab);
    gate[v] = hit ? 1.f : 0.f;
}

extern "C" int dn4gl_label_filter_gate(const int32_t *g_ptr, const int32_t *g_label, const int32_t *p_ptr,
                                       const int32_t *p_label, int32_t B, int32_t Lp_max, int64_t Ng, float *gate,
                                       void *stream) {
    DN_ARG(B >= 0 && Ng >= 0);
    if (Ng == 0) return DN4GL_OK;
    DN_ARG(g_ptr && g_label && p_ptr && p_label && gate);
    label_filter_kernel<<<static_cast<unsigned>(ceil_div64(Ng, 256)), 256, 0, as_stream(stream)>>>(
        g_ptr, g_label, p_ptr, p_label, B, Lp_max, gate, Ng);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Classification loss of the train step: F.nll_loss(log_probs, y) with the default mean reduction
// (graph_classification/graph_neural_networks/main.py:41).  The library kernels behind torch's nll_loss take 20 + 12 us
// for a 1113 x 2 input (profiles/r1f launch list); this is one CTA with a fixed reduction tree, and one elementwise kernel
// for the gradient  g_logp[b, c] = (c == y_b) ? -g / B : 0.
__global__ void __launch_bounds__(1024) nll_mean_fwd_kernel(const float *__restrict__ logp, const int64_t *__restrict__ y,
                                                           int B, int C, float *__restrict__ loss) {
    __shared__ float red[1024];
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += 1024) {
        const int64_t c = y[b];
        if (c >= 0 && c < C) s -= logp[static_cast<int64_t>(b) * C + c];
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) loss[0] = red[0] / static_cast<float>(B > 0 ? B : 1);
}

__global__ void nll_mean_bwd_kernel(const float *__restrict__ g, const int64_t *__restrict__ y, int B, int C,
                                    float *__restrict__ g_logp) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<int64_t>(B) * C) return;
    const int b = static_cast<int>(i / C), c = static_cast<int>(i - static_cast<int64_t>(b) * C);
    g_logp[i] = (y[b] == c) ? -g[0] / static_cast<float>(B) : 0.f;
}

extern "C" int dn4gl_nll_mean_f32(const float *logp, const int64_t *y, int32_t B, int32_t C, float *loss, void *stream) {
    DN_ARG(B >= 0 && C > 0 && loss != nullptr && (B == 0 || (logp != nullptr && y != nullptr)));
    nll_mean_fwd_kernel<<<1, 1024, 0, as_stream(stream)>>>(logp, y, B, C, loss);
    DN_LAUNCHED();
    return DN4GL_OK;
}

extern "C" int dn4gl_nll_mean_bwd_f32(const float *g, const int64_t *y, int32_t B, int32_t C, float *g_logp, void *stream) {
    DN_ARG(B >= 0 && C > 0);
    if (B == 0) return DN4GL_OK;
    DN_ARG(g != nullptr && y != nullptr && g_logp != nullptr);
    nll_mean_bwd_kernel<<<static_cast<unsigned>(ceil_div64(static_cast<int64_t>(B) * C, 256)), 256, 0, as_stream(stream)>>>(
        g, y, B, C, g_logp);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Jumping-knowledge class head of the GIN classifier (gconv.py:205-214): the scores are the sum over layers of
// Linear_l(pooled_l) followed by log_softmax.  As torch ops this was two concatenations, a stack, a small GEMM, five
// elementwise kernels and log_softmax forward, and the mirror image backward (slices of the concatenation gradient
// copied out one by one): ~25 launches of 2-3 us in a train step bound by launch count.  Here: one kernel each way.
//   score[b, c] = sum_l sum_d pooled_l[b, d] W_l[c, d] + n_b bias_0[c] + sum_{l >= 1} bias_l[c]
// n_b = rows of graph b when seg_ptr is given (sum pooling: the reference pools Linear_0(h), so bias_0 is counted once
// per pooled row), 1 otherwise.
constexpr int JK_MAX_LAYERS = 16;
struct JkHeadPtrs {
    const float *pooled[JK_MAX_LAYERS];
    const float *W[JK_MAX_LAYERS];
    const float *bias[JK_MAX_LAYERS];
    float *g_pooled[JK_MAX_LAYERS];
    float *dW[JK_MAX_LAYERS];
    float *db[JK_MAX_LAYERS];
};

// one warp per graph; lane c ends up with score[b, c] (C <= 32)
__global__ void __launch_bounds__(256) jk_head_fwd_kernel(JkHeadPtrs p, int L, int B, int D, int C,
                                                         const int32_t *__restrict__ seg_ptr, float *__restrict__ logp) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float mine = 0.f;
    for (int c = 0; c < C; ++c) {
        float s = 0.f;
        for (int l = 0; l < L; ++l) {
            const float *x = p.pooled[l] + static_cast<int64_t>(b) * D, *w = p.W[l] + static_cast<int64_t>(c) * D;
            for (int d = lane; d < D; d += 32) s = fmaf(__ldg(x + d), __ldg(w + d), s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == c) mine = s;
    }
    if (lane < C) {
        float rest = 0.f;
        for (int l = 1; l < L; ++l) rest += __ldg(p.bias[l] + lane);
        const float n = seg_ptr ? static_cast<float>(seg_ptr[b + 1] - seg_ptr[b]) : 1.f;
        mine += n * __ldg(p.bias[0] + lane) + rest;
    }
    float m = lane < C ? mine : -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float e = lane < C ? expf(mine - m) : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    if (lane < C) logp[static_cast<int64_t>(b) * C + lane] = mine - m - logf(e);
}

// Backward.  Each CTA owns a contiguous range of graphs and walks it JK_ROWS graphs at a time: the pooled rows and the
// score gradient gs = g - exp(logp) * rowsum(g) of those graphs are staged in shared memory (one round of independent
// loads), g_pooled_l = gs W_l is written, and the weight / bias gradients accumulate in shared memory (entry q of acc is
// owned by thread q mod 256: no atomics, fixed order).  The last CTA to finish (ticket) merges the per-CTA partials:
// one warp per entry, lanes over CTAs, butterfly sum -- a fixed tree.
constexpr int JK_ROWS = 8;
__global__ void __launch_bounds__(256) jk_head_bwd_kernel(JkHeadPtrs p, int L, int B, int D, int C,
                                                         const int32_t *__restrict__ seg_ptr, const float *__restrict__ g_logp,
                                                         const float *__restrict__ logp, float *__restrict__ part,
                                                         int *counter) {
    extern __shared__ float jk_smem[];
    __shared__ int is_last;
    const int LD = L * D, NW = C * LD, NACC = NW + 2 * C;      // acc: dW (l, c, d) | sum_b gs[b, c] | sum_b n_b gs[b, c]
    float *acc = jk_smem, *gs = jk_smem + NACC, *cnt = gs + JK_ROWS * C, *xs = cnt + JK_ROWS;   // xs: JK_ROWS x LD
    const int t = threadIdx.x;
    for (int q = t; q < NACC; q += 256) acc[q] = 0.f;
    const int per = (B + gridDim.x - 1) / gridDim.x;
    const int r_begin = blockIdx.x * per, r_end = min(B, r_begin + per);
    for (int r0 = r_begin; r0 < r_end; r0 += JK_ROWS) {
        const int rows = min(JK_ROWS, r_end - r0);
        __syncthreads();
        for (int q = t; q < rows * LD; q += 256) {
            const int r = q / LD, j = q - r * LD, l = j / D, d = j - l * D;
            xs[q] = __ldg(p.pooled[l] + static_cast<int64_t>(r0 + r) * D + d);
        }
        if (t < rows) {
            const float *g = g_logp + static_cast<int64_t>(r0 + t) * C, *lp = logp + static_cast<int64_t>(r0 + t) * C;
            float tot = 0.f;
            for (int c = 0; c < C; ++c) tot += g[c];
            for (int c = 0; c < C; ++c) gs[t * C + c] = g[c] - expf(lp[c]) * tot;
            cnt[t] = seg_ptr ? static_cast<float>(seg_ptr[r0 + t + 1] - seg_ptr[r0 + t]) : 1.f;
        }
        __syncthreads();
        for (int q = t; q < rows * LD; q += 256) {             // g_pooled_l[b, d] = sum_c gs[b, c] W_l[c, d]
            const int r = q / LD, j = q - r * LD, l = j / D, d = j - l * D;
            float s = 0.f;
            for (int c = 0; c < C; ++c) s = fmaf(gs[r * C + c], __ldg(p.W[l] + static_cast<int64_t>(c) * D + d), s);
            p.g_pooled[l][static_cast<int64_t>(r0 + r) * D + d] = s;
        }
        for (int q = t; q < NW; q += 256) {                    // dW_l[c, d] += sum_b gs[b, c] pooled_l[b, d]
            const int l = q / (C * D), rem = q - l * C * D, c = rem / D, d = rem - c * D;
            const float *x = xs + l * D + d;
            float s = acc[q];
            for (int r = 0; r < rows; ++r) s = fmaf(gs[r * C + c], x[r * LD], s);
            acc[q] = s;
        }
        if (t < 2 * C) {
            const int c = t < C ? t : t - C;
            float s = acc[NW + t];
            for (int r = 0; r < rows; ++r) s += (t < C ? 1.f : cnt[r]) * gs[r * C + c];
            acc[NW + t] = s;
        }
    }
    __syncthreads();
    float *mine = part + static_cast<int64_t>(blockIdx.x) * NACC;
    for (int q = t; q < NACC; q += 256) mine[q] = acc[q];
    __threadfence();
    __syncthreads();
    if (t == 0) is_last = (atomicAdd(counter, 1) == static_cast<int>(gridDim.x) - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    const int G = gridDim.x, lane = t & 31;
    for (int q = t >> 5; q < NACC; q += 8) {
        float s = 0.f;
        for (int k = lane; k < G; k += 32) s += __ldcg(part + static_cast<int64_t>(k) * NACC + q);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane != 0) continue;
        if (q < NW) {
            const int l = q / (C * D);
            p.dW[l][q - l * C * D] = s;
        } else {
            const int u = q - NW, c = u < C ? u : u - C;
            if (u < C) {                                       // plain sum: every layer but the first
                for (int l = 1; l < L; ++l) p.db[l][c] = s;
                if (!seg_ptr) p.db[0][c] = s;
            } else if (seg_ptr) {
                p.db[0][c] = s;
            }
        }
    }
    if (t == 0) *counter = 0;
}

static inline int jk_grid(int B) {
    const int want = (B + JK_ROWS - 1) / JK_ROWS;
    const int cap = dn4gl_num_sms();
    return want < 1 ? 1 : (want > cap ? cap : want);
}

static inline size_t jk_bwd_smem(int L, int D, int C) {
    return (static_cast<size_t>(C) * L * D + 2 * C + JK_ROWS * C + JK_ROWS + static_cast<size_t>(JK_ROWS) * L * D) * sizeof(float);
}

extern "C" size_t dn4gl_jk_head_workspace_bytes(int32_t L, int32_t B, int32_t D, int32_t C) {
    return static_cast<size_t>(jk_grid(B)) * (static_cast<size_t>(C) * L * D + 2 * C) * sizeof(float);
}

static bool jk_fill(JkHeadPtrs &p, int L, const float *const *pooled, const float *const *W, const float *const *bias) {
    for (int l = 0; l < L; ++l) {
        if (!pooled[l] || !W[l] || !bias[l]) return false;
        p.pooled[l] = pooled[l]; p.W[l] = W[l]; p.bias[l] = bias[l];
    }
    return true;
}

extern "C" int dn4gl_jk_head_fwd_f32(const float *const *pooled, const float *const *W, const float *const *bias, int32_t L,
                                     int32_t B, int32_t D, int32_t C, const int32_t *seg_ptr, float *logp, void *stream) {
    DN_ARG(L >= 1 && L <= JK_MAX_LAYERS && B >= 0 && D >= 1 && C >= 1 && C <= 32 && pooled && W && bias);
    if (B == 0) return DN4GL_OK;
    JkHeadPtrs p = {};
    DN_ARG(jk_fill(p, L, pooled, W, bias) && logp != nullptr);
    jk_head_fwd_kernel<<<(B + 7) / 8, 256, 0, as_stream(stream)>>>(p, L, B, D, C, seg_ptr, logp);
    DN_LAUNCHED();
    return DN4GL_OK;
}

extern "C" int dn4gl_jk_head_bwd_f32(const float *g_logp, const float *logp, const float *const *pooled, const float *const *W,
                                     int32_t L, int32_t B, int32_t D, int32_t C, const int32_t *seg_ptr,
                                     float *const *g_pooled, float *const *dW, float *const *db, void *ws, size_t ws_bytes,
                                     int32_t *counter, void *stream) {
    DN_ARG(L >= 1 && L <= JK_MAX_LAYERS && B >= 1 && D >= 1 && C >= 1 && C <= 32 && pooled && W && g_pooled && dW && db);
    DN_ARG(g_logp && logp && ws && counter && ws_bytes >= dn4gl_jk_head_workspace_bytes(L, B, D, C));
    const size_t smem = jk_bwd_smem(L, D, C);
    DN_ARG(smem <= 48 * 1024);
    JkHeadPtrs p = {};
    for (int l = 0; l < L; ++l) {
        DN_ARG(pooled[l] && W[l] && g_pooled[l] && dW[l] && db[l]);
        p.pooled[l] = pooled[l]; p.W[l] = W[l]; p.g_pooled[l] = g_pooled[l]; p.dW[l] = dW[l]; p.db[l] = db[l];
    }
    jk_head_bwd_kernel<<<jk_grid(B), 256, smem, as_stream(stream)>>>(p, L, B, D, C, seg_ptr, g_logp, logp,
                                                                     static_cast<float *>(ws), counter);
    DN_LAUNCHED();
    return DN4GL_OK;
}
