// The matching objective of the counting models (subgraph_isomorphism/train.py:776-813 with --match_weights node /
// edge): the dummy column of the ground-truth subisomorphisms, and the match terms of bp_loss as one kernel each way.
//
// Dummy column (train.py:467-472, add_dummy_nodes_edges): every row of sample b's subisomorphism matrix gets one more
// entry, the graph-local id of the graph's dummy node, which is the graph's node count BEFORE augmentation.  One CTA
// per sample copies its S_b rows of np_b ids to rows of np_b + 1; integers only.
//
// Match terms, per kind k in {node, edge} that is present: pred (B, L) left-padded, mask (B, L), flat int32 weights
// (N,) with row offsets seg_ptr (position (b, j) reads row seg_ptr[b] + j - (L - len_b) when j >= L - len_b).  On a
// masked or padded position both the prediction and the target count as 0 (the reference zeroes them in place,
// train.py:783-784), so the loss term vanishes there but the regulariser term crit(relu(0 - pred_c[b])) does not.
//   loss_k = mean over B*L of crit(leaky(p, neg_slp) - w) * L = sum / B
//   reg_k  = mean over B*L of crit(relu(p - pred_c[b]))   * L = sum / B
//   out    = match_loss_w * (loss_v + loss_e) + match_reg_w * (reg_v + reg_e)
// Elements are formed in double from the fp32 inputs.
//
// Summation order: one CTA per graph; thread t adds the node positions t, t + 256, ... and then the edge positions
// t, t + 256, ... of its graph in double, and a fixed halving tree combines the 256 thread sums.  The forward's per-graph
// partials are merged by the last CTA to finish, thread t adding graphs t, t + 256, ... in order, then the same tree.
// The order depends on B and the padded lengths only -- not on the grid or the SM count.  No float atomics; the ticket
// counter is left at zero, so the launch replays inside a captured CUDA graph.  pred_c's gradient is the per-graph sum
// of the regulariser's derivative over the L_v + L_e positions, in the same order.
#include "common.cuh"

constexpr int DUMMY_THREADS = 128;
constexpr int MATCH_THREADS = 256;
enum { CRIT_MAE = 0, CRIT_MSE = 1, CRIT_SMSE = 2 };

__global__ void __launch_bounds__(DUMMY_THREADS) subiso_append_dummy_kernel(
    const int32_t *__restrict__ val_ptr, const int32_t *__restrict__ values, const int32_t *__restrict__ rows,
    const int32_t *__restrict__ g_node_ptr, const int32_t *__restrict__ out_ptr, int32_t *__restrict__ out) {
    const int b = blockIdx.x;
    const int S = rows[b];
    if (S <= 0) return;
    const int v0 = val_ptr[b];
    const int np_ = (val_ptr[b + 1] - v0) / S;
    const int w = np_ + 1;
    const int n_b = g_node_ptr[b + 1] - g_node_ptr[b];
    const int64_t total = static_cast<int64_t>(S) * w;
    int32_t *o = out + out_ptr[b];
    for (int64_t k = threadIdx.x; k < total; k += DUMMY_THREADS) {
        const int64_t s = k / w;
        const int c = static_cast<int>(k - s * w);
        o[k] = c < np_ ? values[v0 + s * np_ + c] : n_b;
    }
}

struct MatchKind {
    const float *pred;
    const uint8_t *mask;
    const int32_t *w;
    const int32_t *seg_ptr;
    int L;
};

// F.l1_loss / F.mse_loss / F.smooth_l1_loss (beta 1) per element of d = input - target, and their derivatives in d
// with torch's conventions: sign(0) = 0; smooth-L1 is quadratic for |d| < 1 and its derivative is clamp(d, -1, 1)
__device__ __forceinline__ double crit_value(int crit, double d) {
    const double a = fabs(d);
    if (crit == CRIT_MAE) return a;
    if (crit == CRIT_MSE) return d * d;
    return a < 1.0 ? 0.5 * d * d : a - 0.5;
}

__device__ __forceinline__ double crit_grad(int crit, double d) {
    if (crit == CRIT_MAE) return d > 0.0 ? 1.0 : (d < 0.0 ? -1.0 : 0.0);
    if (crit == CRIT_MSE) return 2.0 * d;
    return d < -1.0 ? -1.0 : (d > 1.0 ? 1.0 : d);
}

// (prediction, target) of position j of graph b, both 0 on masked and padded positions
__device__ __forceinline__ void match_at(const MatchKind &k, int b, int j, double &p, double &w) {
    const int64_t at = static_cast<int64_t>(b) * k.L + j;
    p = w = 0.0;
    if (!k.mask[at]) return;
    p = static_cast<double>(k.pred[at]);
    const int s0 = k.seg_ptr[b], len = k.seg_ptr[b + 1] - s0;
    const int pad = k.L - len;
    if (j >= pad) w = static_cast<double>(k.w[s0 + j - pad]);
}

__device__ __forceinline__ double match_tree(double *red, double s) {
    const int t = threadIdx.x;
    red[t] = s;
    __syncthreads();
#pragma unroll
    for (int o = MATCH_THREADS / 2; o > 0; o >>= 1) {
        if (t < o) red[t] += red[t + o];
        __syncthreads();
    }
    const double out = red[0];
    __syncthreads();                                // red is reused by the caller's next sum
    return out;
}

__global__ void __launch_bounds__(MATCH_THREADS) match_loss_kernel(
    int B, const float *__restrict__ pred_c, MatchKind kv, MatchKind ke, int crit, const float *__restrict__ neg_slp,
    const float *__restrict__ match_loss_w, const float *__restrict__ match_reg_w, float *__restrict__ out,
    double *__restrict__ part, int *counter) {
    __shared__ double red[MATCH_THREADS];
    __shared__ int is_last;
    const int t = threadIdx.x, b = blockIdx.x;
    const double slp = static_cast<double>(*neg_slp), c = static_cast<double>(pred_c[b]);
    double sl = 0.0, sr = 0.0;
    for (int kind = 0; kind < 2; ++kind) {
        const MatchKind &k = kind == 0 ? kv : ke;
        if (k.pred == nullptr) continue;
        for (int j = t; j < k.L; j += MATCH_THREADS) {
            double p, w;
            match_at(k, b, j, p, w);
            sl += crit_value(crit, (p > 0.0 ? p : p * slp) - w);
            const double x = p - c;
            sr += crit_value(crit, x > 0.0 ? x : 0.0);
        }
    }
    sl = match_tree(red, sl);
    sr = match_tree(red, sr);
    if (t == 0) {
        part[2 * b] = sl;
        part[2 * b + 1] = sr;
        __threadfence();
        is_last = (atomicAdd(counter, 1) == B - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    double tl = 0.0, tr = 0.0;
    for (int g = t; g < B; g += MATCH_THREADS) {
        tl += __ldcg(part + 2 * g);
        tr += __ldcg(part + 2 * g + 1);
    }
    tl = match_tree(red, tl);
    tr = match_tree(red, tr);
    if (t == 0) {
        const double r = (static_cast<double>(*match_loss_w) * tl + static_cast<double>(*match_reg_w) * tr) / B;
        *out = static_cast<float>(r);
        *counter = 0;
    }
}

__global__ void __launch_bounds__(MATCH_THREADS) match_loss_bwd_kernel(
    int B, const float *__restrict__ g_out, const float *__restrict__ pred_c, MatchKind kv, MatchKind ke, int crit,
    const float *__restrict__ neg_slp, const float *__restrict__ match_loss_w, const float *__restrict__ match_reg_w,
    float *__restrict__ g_pred_v, float *__restrict__ g_pred_e, float *__restrict__ g_pred_c) {
    __shared__ double red[MATCH_THREADS];
    const int t = threadIdx.x, b = blockIdx.x;
    const double g = static_cast<double>(*g_out);
    const double gl = g * static_cast<double>(*match_loss_w) / B, gr = g * static_cast<double>(*match_reg_w) / B;
    const double slp = static_cast<double>(*neg_slp), c = static_cast<double>(pred_c[b]);
    double sc = 0.0;
    for (int kind = 0; kind < 2; ++kind) {
        const MatchKind &k = kind == 0 ? kv : ke;
        float *gp = kind == 0 ? g_pred_v : g_pred_e;
        if (k.pred == nullptr) continue;
        for (int j = t; j < k.L; j += MATCH_THREADS) {
            double p, w;
            match_at(k, b, j, p, w);
            // loss term: zero on masked positions (p = w = 0 gives d = 0, whose derivative is 0 under every criterion)
            const double dl = crit_grad(crit, (p > 0.0 ? p : p * slp) - w) * (p > 0.0 ? 1.0 : slp);
            // regulariser: relu's derivative is 0 at 0, and so is every criterion's at d = 0
            const double x = p - c;
            const double dr = x > 0.0 ? crit_grad(crit, x) : 0.0;
            gp[static_cast<int64_t>(b) * k.L + j] = static_cast<float>(gl * dl + gr * dr);
            sc += dr;
        }
    }
    sc = match_tree(red, sc);
    if (t == 0) g_pred_c[b] = static_cast<float>(-gr * sc);
}

extern "C" int dn4gl_subiso_append_dummy(int32_t B, const int32_t *val_ptr, const int32_t *values, const int32_t *rows,
                                         const int32_t *g_node_ptr, const int32_t *out_ptr, int64_t out_total,
                                         int32_t *out, void *stream) {
    DN_ARG(B >= 0 && out_total >= 0);
    if (B == 0 || out_total == 0) return DN4GL_OK;
    DN_ARG(val_ptr != nullptr && rows != nullptr && g_node_ptr != nullptr && out_ptr != nullptr && out != nullptr);
    subiso_append_dummy_kernel<<<B, DUMMY_THREADS, 0, as_stream(stream)>>>(val_ptr, values, rows, g_node_ptr, out_ptr,
                                                                           out);
    DN_LAUNCHED();
    return DN4GL_OK;
}

static bool match_kind_ok(const MatchKind &k) {
    return k.pred == nullptr || (k.L >= 0 && (k.L == 0 || (k.mask != nullptr && k.seg_ptr != nullptr)));
}

extern "C" size_t dn4gl_match_loss_workspace_bytes(int32_t B) {
    return B > 0 ? 2 * static_cast<size_t>(B) * sizeof(double) : 0;
}

extern "C" int dn4gl_match_loss_f32(int32_t B, const float *pred_c, const float *pred_v, const uint8_t *mask_v,
                                    const int32_t *w_v, const int32_t *ptr_v, int32_t Lv, const float *pred_e,
                                    const uint8_t *mask_e, const int32_t *w_e, const int32_t *ptr_e, int32_t Le,
                                    int32_t crit, const float *neg_slp, const float *match_loss_w,
                                    const float *match_reg_w, float *out, void *ws, size_t ws_bytes, int32_t *counter,
                                    void *stream) {
    const MatchKind kv{pred_v, mask_v, w_v, ptr_v, Lv}, ke{pred_e, mask_e, w_e, ptr_e, Le};
    DN_ARG(B >= 0 && crit >= CRIT_MAE && crit <= CRIT_SMSE && out != nullptr && match_kind_ok(kv) && match_kind_ok(ke));
    cudaStream_t s = as_stream(stream);
    if (B == 0) {
        DN_CUDA(cudaMemsetAsync(out, 0, sizeof(float), s));
        return DN4GL_OK;
    }
    DN_ARG(pred_c != nullptr && neg_slp != nullptr && match_loss_w != nullptr && match_reg_w != nullptr);
    DN_ARG(ws != nullptr && counter != nullptr && (reinterpret_cast<uintptr_t>(ws) & 7u) == 0);
    DN_ARG(ws_bytes >= dn4gl_match_loss_workspace_bytes(B));
    match_loss_kernel<<<B, MATCH_THREADS, 0, s>>>(B, pred_c, kv, ke, crit, neg_slp, match_loss_w, match_reg_w, out,
                                                  static_cast<double *>(ws), counter);
    DN_LAUNCHED();
    return DN4GL_OK;
}

extern "C" int dn4gl_match_loss_bwd_f32(int32_t B, const float *g_out, const float *pred_c, const float *pred_v,
                                        const uint8_t *mask_v, const int32_t *w_v, const int32_t *ptr_v, int32_t Lv,
                                        const float *pred_e, const uint8_t *mask_e, const int32_t *w_e,
                                        const int32_t *ptr_e, int32_t Le, int32_t crit, const float *neg_slp,
                                        const float *match_loss_w, const float *match_reg_w, float *g_pred_v,
                                        float *g_pred_e, float *g_pred_c, void *stream) {
    const MatchKind kv{pred_v, mask_v, w_v, ptr_v, Lv}, ke{pred_e, mask_e, w_e, ptr_e, Le};
    DN_ARG(B >= 0 && crit >= CRIT_MAE && crit <= CRIT_SMSE && match_kind_ok(kv) && match_kind_ok(ke));
    if (B == 0) return DN4GL_OK;
    DN_ARG(g_out != nullptr && pred_c != nullptr && g_pred_c != nullptr && neg_slp != nullptr &&
           match_loss_w != nullptr && match_reg_w != nullptr);
    DN_ARG((pred_v == nullptr || g_pred_v != nullptr) && (pred_e == nullptr || g_pred_e != nullptr));
    match_loss_bwd_kernel<<<B, MATCH_THREADS, 0, as_stream(stream)>>>(B, g_out, pred_c, kv, ke, crit, neg_slp,
                                                                      match_loss_w, match_reg_w, g_pred_v, g_pred_e,
                                                                      g_pred_c);
    DN_LAUNCHED();
    return DN4GL_OK;
}
