// Evaluation over a held-out split (pipelines.py: evaluate): per-sample records of a batch written at the batch's
// offset into split-sized arrays, and a fixed-order reduction of the record columns into the split's metrics.
//
// Classification (graph_neural_networks/main.py:eval_test): one warp per graph row of the (B, C) log-probabilities
// finds the arg-max with torch.max's first-occurrence rule (a NaN counts as the largest value, as in torch), and the
// row's NLL -logp[y]; the correct flag is pred == y.  Counting (subgraph_isomorphism/train.py:evaluate): one thread per
// sample forms r = relu(pred_c), t = float(count) and the three per-element error terms of F.l1_loss, F.mse_loss and
// F.smooth_l1_loss (beta 1).
//
// Reduction: the samples are cut into tiles of EVAL_TILE consecutive rows.  Inside a tile thread t adds rows t, t + 256,
// t + 512, t + 768 in that order in double precision, then the 256 thread sums are combined by a fixed halving tree;
// the tile partials are merged by the last CTA to finish, thread t adding tiles t, t + 256, ... in order, then the same
// tree.  Which CTA computes which tile does not enter the result, so it depends on n and the values only -- not on
// the grid, the SM count or how the records were batched.  No float atomics; the ticket counter is left at zero.
#include "common.cuh"

constexpr int EVAL_THREADS = 256;
constexpr int EVAL_ROWS_PER_THREAD = 4;
constexpr int EVAL_TILE = EVAL_THREADS * EVAL_ROWS_PER_THREAD;
constexpr int EVAL_MAX_COLUMNS = 8;
constexpr int EVAL_CLASS_WARPS = 8;        // rows per CTA of the classification record kernel

// (value, index) order of torch.max along a row: NaN above every number, then larger values, ties to the lower index
__device__ __forceinline__ bool argmax_before(float va, int ia, float vb, int ib) {
    const bool na = va != va, nb = vb != vb;
    if (na != nb) return na;
    if (na || va == vb) return ia < ib;
    return va > vb;
}

__global__ void __launch_bounds__(EVAL_CLASS_WARPS * 32) eval_class_rows_kernel(
    const float *__restrict__ logp, const int64_t *__restrict__ y, int B, int C, int64_t pos0, int32_t *__restrict__ pred,
    float *__restrict__ nll, float *__restrict__ correct) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * EVAL_CLASS_WARPS + (threadIdx.x >> 5);
    if (row >= B) return;
    const float *r = logp + static_cast<int64_t>(row) * C;
    float bv = 0.f;
    int bi = -1;                                    // no candidate yet (lanes with c >= C keep it)
    for (int c = lane; c < C; c += 32) {
        const float v = __ldg(r + c);
        if (bi < 0 || argmax_before(v, c, bv, bi)) { bv = v; bi = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || argmax_before(ov, oi, bv, bi))) { bv = ov; bi = oi; }
    }
    if (lane == 0) {
        const int64_t c = __ldg(y + row);
        const bool in_range = c >= 0 && c < C;
        const bool has_nan = bv != bv;              // a NaN anywhere in the row is its maximum
        // out-of-range targets contribute nothing to the NLL, as in dn4gl_nll_mean_f32; a NaN row is never correct
        const float l = has_nan ? bv : (in_range ? -__ldg(r + c) : 0.f);
        const int64_t p = pos0 + row;
        pred[p] = bi;
        nll[p] = l;
        correct[p] = (!has_nan && in_range && bi == c) ? 1.f : 0.f;
    }
}

__global__ void __launch_bounds__(EVAL_THREADS) eval_count_rows_kernel(const float *__restrict__ pred_c,
                                                                       const int64_t *__restrict__ counts, int B,
                                                                       int64_t pos0, float *__restrict__ pred,
                                                                       float *__restrict__ err) {
    const int i = blockIdx.x * EVAL_THREADS + threadIdx.x;
    if (i >= B) return;
    const float p = __ldg(pred_c + i);
    const float r = p <= 0.f ? 0.f : p;             // relu; NaN passes through as in torch.relu
    const float t = __ll2float_rn(__ldg(counts + i));
    const float d = __fsub_rn(r, t);
    const float z = fabsf(d);
    const int64_t o = pos0 + i;
    pred[o] = p;
    err[3 * o + 0] = z;                                                                  // F.l1_loss
    err[3 * o + 1] = __fmul_rn(d, d);                                                    // F.mse_loss
    err[3 * o + 2] = z < 1.f ? __fmul_rn(__fmul_rn(0.5f, z), z) : __fsub_rn(z, 0.5f);  // F.smooth_l1_loss, beta 1
}

__device__ __forceinline__ double eval_tree(double *red, double s) {
    const int t = threadIdx.x;
    red[t] = s;
    __syncthreads();
#pragma unroll
    for (int o = EVAL_THREADS / 2; o > 0; o >>= 1) {
        if (t < o) red[t] += red[t + o];
        __syncthreads();
    }
    const double out = red[0];
    __syncthreads();                                // red is reused by the caller's next column
    return out;
}

__global__ void __launch_bounds__(EVAL_THREADS) eval_reduce_kernel(const float *__restrict__ v, int64_t n, int k,
                                                                   double *__restrict__ out, double *__restrict__ part,
                                                                   int *counter) {
    __shared__ double red[EVAL_THREADS];
    __shared__ int is_last;
    const int t = threadIdx.x;
    const int64_t tiles = (n + EVAL_TILE - 1) / EVAL_TILE;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        for (int c = 0; c < k; ++c) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < EVAL_ROWS_PER_THREAD; ++j) {
                const int64_t i = tile * EVAL_TILE + j * EVAL_THREADS + t;
                if (i < n) s += static_cast<double>(__ldg(v + i * k + c));
            }
            const double p = eval_tree(red, s);
            if (t == 0) part[tile * k + c] = p;
        }
    }
    if (t == 0) {
        __threadfence();
        is_last = (atomicAdd(counter, 1) == static_cast<int>(gridDim.x) - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    for (int c = 0; c < k; ++c) {
        double s = 0.0;
        for (int64_t tile = t; tile < tiles; tile += EVAL_THREADS) s += __ldcg(part + tile * k + c);
        const double r = eval_tree(red, s);
        if (t == 0) out[c] = r;
    }
    if (t == 0) *counter = 0;
}

extern "C" int dn4gl_eval_class_rows_f32(const float *logp, const int64_t *y, int32_t B, int32_t C, int64_t pos0,
                                         int32_t *pred, float *nll, float *correct, void *stream) {
    DN_ARG(B >= 0 && C >= 1 && pos0 >= 0);
    if (B == 0) return DN4GL_OK;
    DN_ARG(logp != nullptr && y != nullptr && pred != nullptr && nll != nullptr && correct != nullptr);
    eval_class_rows_kernel<<<static_cast<unsigned>(ceil_div64(B, EVAL_CLASS_WARPS)), EVAL_CLASS_WARPS * 32, 0,
                             as_stream(stream)>>>(logp, y, B, C, pos0, pred, nll, correct);
    DN_LAUNCHED();
    return DN4GL_OK;
}

extern "C" int dn4gl_eval_count_rows_f32(const float *pred_c, const int64_t *counts, int32_t B, int64_t pos0, float *pred,
                                         float *err, void *stream) {
    DN_ARG(B >= 0 && pos0 >= 0);
    if (B == 0) return DN4GL_OK;
    DN_ARG(pred_c != nullptr && counts != nullptr && pred != nullptr && err != nullptr);
    eval_count_rows_kernel<<<static_cast<unsigned>(ceil_div64(B, EVAL_THREADS)), EVAL_THREADS, 0, as_stream(stream)>>>(
        pred_c, counts, B, pos0, pred, err);
    DN_LAUNCHED();
    return DN4GL_OK;
}

extern "C" size_t dn4gl_eval_reduce_workspace_bytes(int64_t n, int32_t k) {
    if (n <= 0 || k < 1) return 0;
    return static_cast<size_t>(ceil_div64(n, EVAL_TILE)) * static_cast<size_t>(k) * sizeof(double);
}

extern "C" int dn4gl_eval_reduce_f32(const float *v, int64_t n, int32_t k, double *out, void *ws, size_t ws_bytes,
                                     int32_t *counter, void *stream) {
    DN_ARG(n >= 0 && k >= 1 && k <= EVAL_MAX_COLUMNS && out != nullptr);
    cudaStream_t s = as_stream(stream);
    if (n == 0) {
        DN_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * k, s));
        return DN4GL_OK;
    }
    DN_ARG(v != nullptr && ws != nullptr && counter != nullptr && (reinterpret_cast<uintptr_t>(ws) & 7u) == 0);
    DN_ARG(ws_bytes >= dn4gl_eval_reduce_workspace_bytes(n, k));
    const int64_t tiles = ceil_div64(n, EVAL_TILE);
    const int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * 4;
    eval_reduce_kernel<<<static_cast<int>(tiles < cap ? tiles : cap), EVAL_THREADS, 0, s>>>(
        v, n, k, out, static_cast<double *>(ws), counter);
    DN_LAUNCHED();
    return DN4GL_OK;
}
