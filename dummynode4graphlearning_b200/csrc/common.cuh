// Shared helpers for libdn4gl.so (sm_100a).  Host-side error plumbing + device utilities.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "dn4gl.h"

void dn4gl_set_error(const char *fmt, ...);

#define DN_ARG(cond)                                                                         \
    do {                                                                                     \
        if (!(cond)) {                                                                       \
            dn4gl_set_error("%s: invalid argument: %s", __func__, #cond);                    \
            return DN4GL_EINVAL;                                                             \
        }                                                                                    \
    } while (0)

#define DN_CUDA(call)                                                                        \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            dn4gl_set_error("%s: %s -> %s", __func__, #call, cudaGetErrorString(e__));       \
            return DN4GL_ECUDA;                                                              \
        }                                                                                    \
    } while (0)

// checks the launches issued since the previous check and adds them to the process-wide kernel counter
// (dn4gl_launch_count(); bench.py reports it as gpu_launches)
void dn4gl_note_launches(int n);
#define DN_LAUNCHED_N(n)                                                                     \
    do {                                                                                     \
        cudaError_t e__ = cudaGetLastError();                                                \
        if (e__ != cudaSuccess) {                                                            \
            dn4gl_set_error("%s: launch failed: %s", __func__, cudaGetErrorString(e__));     \
            return DN4GL_ECUDA;                                                              \
        }                                                                                    \
        dn4gl_note_launches(n);                                                              \
    } while (0)
#define DN_LAUNCHED() DN_LAUNCHED_N(1)

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }
static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// B200: 148 SMs.  Queried once per process (benign cache; the library targets one GPU per process).
int dn4gl_num_sms();

// carve sub-buffers out of the caller's workspace (256-byte aligned pieces)
struct WsCarver {
    char *base;
    size_t off, cap;
    WsCarver(void *ws, size_t bytes) : base(static_cast<char *>(ws)), off(0), cap(bytes) {}
    template <typename T> T *take(size_t n) {
        size_t b = align_up(n * sizeof(T), 256);
        if (off + b > cap) return nullptr;
        T *p = reinterpret_cast<T *>(base + off);
        off += b;
        return p;
    }
};

#ifdef __CUDACC__
__device__ __forceinline__ float4 ldg4(const float4 *p) { return __ldg(p); }
// packed fp32 pairs (sm_100 add/mul.rn.f32x2 -> SASS FADD2 / FMUL2): two IEEE round-to-nearest results per issue slot
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void add4(float4 &a, const float4 &b) {
    unsigned long long a0 = pack2(a.x, a.y), a1 = pack2(a.z, a.w);
    const unsigned long long b0 = pack2(b.x, b.y), b1 = pack2(b.z, b.w);
    asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a0) : "l"(b0));
    asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a1) : "l"(b1));
    unpack2(a0, a.x, a.y);
    unpack2(a1, a.z, a.w);
}
__device__ __forceinline__ void sub4(float4 &a, const float4 &b) {
    a.x = __fsub_rn(a.x, b.x); a.y = __fsub_rn(a.y, b.y); a.z = __fsub_rn(a.z, b.z); a.w = __fsub_rn(a.w, b.w);
}
// a += s * b with a separately rounded product (matches torch's  out + (1 + eps) * x ).  The product stays scalar:
// ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (single rounding), __fmul_rn is never contracted.
__device__ __forceinline__ void axpy4_rn(float4 &a, float s, const float4 &b) {
    const float4 t = make_float4(__fmul_rn(s, b.x), __fmul_rn(s, b.y), __fmul_rn(s, b.z), __fmul_rn(s, b.w));
    add4(a, t);
}
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// largest g in [0, B) with ptr[g] <= i  (ptr non-decreasing, ptr[0] <= i < ptr[B])
__device__ __forceinline__ int segment_of(const int32_t *__restrict__ ptr, int B, int64_t i) {
    int lo = 0, hi = B;  // invariant: ptr[lo] <= i < ptr[hi]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (static_cast<int64_t>(__ldg(ptr + mid)) <= i) lo = mid; else hi = mid;
    }
    return lo;
}
#endif
