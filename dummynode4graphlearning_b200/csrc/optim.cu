// libdn4gl.so -- optimizer step over FLAT parameter / gradient / moment buffers.
//
// The reference steps torch.optim.Adam (graph_classification/graph_neural_networks/main.py:43, optimizer built at
// main.py:253) or AdamW(amsgrad=True) (subgraph_isomorphism/train.py:1380-1386 region) once per mini-batch.  The stock
// capturable implementation issues ~75 tiny kernels per step for the 50k-parameter GIN (profiles/r1d launch list:
// ~220 us of a 2.4 ms step); with parameters and gradients held as views of flat buffers (parallel.GradientBucket,
// optim.FlatAdam) the whole update is ONE streaming pass: 4 reads + 3 writes of 4 bytes per parameter.
// Hyper-parameters and the step counter live in device memory, so a captured CUDA graph replays the step with the
// current learning rate and an advancing bias correction.
#include "common.cuh"

struct AdamHyper { float lr, beta1, beta2, eps, weight_decay; };

__device__ __forceinline__ void adam_one(float &p, float g, float &m, float &v, float *vmax, const AdamHyper h,
                                         float step_size, float inv_bc2_sqrt, bool decoupled) {
    if (h.weight_decay != 0.f) {
        if (decoupled) p = p * (1.f - h.lr * h.weight_decay);       // AdamW: param.mul_(1 - lr * wd)
        else g = g + h.weight_decay * p;                           // Adam: grad.add(param, alpha=wd)
    }
    m = m + (g - m) * (1.f - h.beta1);                             // exp_avg.lerp_(grad, 1 - beta1)
    v = v * h.beta2 + (1.f - h.beta2) * g * g;                     // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    float vv = v;
    if (vmax) { vv = fmaxf(*vmax, v); *vmax = vv; }                // amsgrad: running maximum of the second moment
    const float denom = sqrtf(vv) * inv_bc2_sqrt + h.eps;          // (sqrt(v) / sqrt(bc2)).add_(eps)
    p = p - step_size * (m / denom);                               // param.addcdiv_(exp_avg, denom, value=-lr / bc1)
}

__global__ void __launch_bounds__(256) adam_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                                                   float *__restrict__ v, float *__restrict__ vmax, int64_t n,
                                                   const float *__restrict__ hyper, float *step, int decoupled,
                                                   int32_t *counter) {
    const AdamHyper h = {hyper[0], hyper[1], hyper[2], hyper[3], hyper[4]};
    // bias corrections in double, once per CTA (pow is ~200 FP64 instructions)
    __shared__ float sh_step_size, sh_inv_bc2_sqrt, sh_t;
    if (threadIdx.x == 0) {
        const double t = static_cast<double>(*reinterpret_cast<volatile float *>(step)) + 1.0;
        const double bc1 = 1.0 - pow(static_cast<double>(h.beta1), t), bc2 = 1.0 - pow(static_cast<double>(h.beta2), t);
        sh_step_size = static_cast<float>(static_cast<double>(h.lr) / bc1);
        sh_inv_bc2_sqrt = static_cast<float>(1.0 / sqrt(bc2));
        sh_t = static_cast<float>(t);
    }
    __syncthreads();
    const float step_size = sh_step_size, inv_bc2_sqrt = sh_inv_bc2_sqrt;
    const int64_t n4 = n >> 2;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    float4 *p4 = reinterpret_cast<float4 *>(p), *m4 = reinterpret_cast<float4 *>(m), *v4 = reinterpret_cast<float4 *>(v);
    float4 *x4 = reinterpret_cast<float4 *>(vmax);
    const float4 *g4 = reinterpret_cast<const float4 *>(g);
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 P = p4[i], M = m4[i], V = v4[i], X = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 G = g4[i];
        if (vmax) X = x4[i];
        adam_one(P.x, G.x, M.x, V.x, vmax ? &X.x : nullptr, h, step_size, inv_bc2_sqrt, decoupled);
        adam_one(P.y, G.y, M.y, V.y, vmax ? &X.y : nullptr, h, step_size, inv_bc2_sqrt, decoupled);
        adam_one(P.z, G.z, M.z, V.z, vmax ? &X.z : nullptr, h, step_size, inv_bc2_sqrt, decoupled);
        adam_one(P.w, G.w, M.w, V.w, vmax ? &X.w : nullptr, h, step_size, inv_bc2_sqrt, decoupled);
        p4[i] = P; m4[i] = M; v4[i] = V;
        if (vmax) x4[i] = X;
    }
    for (int64_t i = (n4 << 2) + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        adam_one(p[i], g[i], m[i], v[i], vmax ? vmax + i : nullptr, h, step_size, inv_bc2_sqrt, decoupled);
    // the last CTA to finish advances the step counter (every CTA has read it by then) and re-arms the ticket
    __shared__ int last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = (atomicAdd(counter, 1) == static_cast<int>(gridDim.x) - 1);
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        *step = sh_t;
        *counter = 0;
    }
}

extern "C" int dn4gl_adam_f32(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *max_exp_avg_sq,
                              int64_t n, const float *hyper, float *step, int32_t decoupled, int32_t *counter,
                              void *stream) {
    DN_ARG(n >= 0 && hyper != nullptr && step != nullptr && counter != nullptr);
    if (n == 0) return DN4GL_OK;
    DN_ARG(param && grad && exp_avg && exp_avg_sq && aligned16(param) && aligned16(grad) && aligned16(exp_avg) &&
           aligned16(exp_avg_sq) && (max_exp_avg_sq == nullptr || aligned16(max_exp_avg_sq)));
    int64_t want = ceil_div64(ceil_div64(n, 4), 256);
    const int64_t cap = static_cast<int64_t>(dn4gl_num_sms()) * 8;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    adam_kernel<<<static_cast<unsigned>(want), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, max_exp_avg_sq, n,
                                                                            hyper, step, decoupled, counter);
    DN_LAUNCHED();
    return DN4GL_OK;
}
