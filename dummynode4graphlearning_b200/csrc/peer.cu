// libdn4gl.so -- one-shot all-reduce of the flat gradient bucket over NVLink peer memory (one node, <= 8 GPUs).
//
// The data-parallel step (SURVEY.md 8(e); the reference itself is single-device) has ONE exchange: the sum over ranks
// of the weighted flat gradient bucket, 40 KB (GIN) to 0.7 MB (DMPNN).  At that size a library all-reduce is pure
// latency -- measured on 8 B200s: +0.053 ms on a 0.88 ms step (profiles/r3l_*), with a `flat *= B_r / B` kernel in front
// of it.  Every rank can read every other rank's memory directly (NVSwitch; peer mappings exchanged once as CUDA IPC
// handles by parallel.PeerAllReduce), so the reduction is one kernel per rank, and block b of every rank only ever talks
// to block b of the other ranks (all ranks launch the same grid):
//
//   0  block b copies weight * bucket[its range] into this rank's EXPOSED buffer of the step's parity (two buffers,
//      alternating), then writes the step's epoch into slot (rank, b) of every peer's signal words (st.release.sys over
//      NVLink) and waits until its own slots (r, b) carry the epoch from every rank r;
//   1  block b adds the ranks' exposed ranges in RANK ORDER (r = 0 .. W-1) and writes the sum into the bucket: every
//      rank computes the same bits, nothing else is exchanged.
//
// One barrier is enough because of the two exposed buffers: a rank rewrites buffer p two steps later, after it has passed
// the barrier of the step in between -- which every peer only signals after it has finished reading buffer p.  Flags
// and epochs are monotonic per block: nothing is reset, no block waits for a block of its own grid (so no cooperative
// launch), and the kernel replays inside a CUDA graph.  Waits are bounded (__trap after 2^26 polls): a missing peer
// fails loudly instead of hanging the device.
#include <cstring>
#include "common.cuh"

namespace {

constexpr int PEER_MAX = 8, PEER_MAX_BLOCKS = 128;
// signal words (int32) of a rank: [r * 128 + b] epoch written by block b of rank r, [1024 + b] epoch block b completed last
constexpr int SIG_READY = 0, SIG_EPOCH = PEER_MAX * PEER_MAX_BLOCKS;

struct PeerPtrs {
    float *exposed[PEER_MAX];      // 2 n floats per rank
    int32_t *sig[PEER_MAX];
};

__device__ __forceinline__ void st_release_sys(int32_t *p, int32_t v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int32_t ld_acquire_sys(const int32_t *p) {
    int32_t v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_sys_v4(const float *p) {      // coherent at system scope: never a stale L1 line
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}

template <int W>
__global__ void __launch_bounds__(256) peer_allreduce_kernel(PeerPtrs pp, int rank, int64_t n4, float weight,
                                                             float4 *__restrict__ bucket) {
    constexpr int world = W;
    int32_t *mine = pp.sig[rank];
    const int b = static_cast<int>(blockIdx.x), t = static_cast<int>(threadIdx.x);
    const int32_t epoch = mine[SIG_EPOCH + b] + 1;                  // this block's own counter (written back at the end)
    const int64_t per = (n4 + gridDim.x - 1) / gridDim.x, i0 = b * per, i1 = (i0 + per < n4) ? i0 + per : n4;
    const int64_t par = static_cast<int64_t>(epoch & 1) * n4;       // which exposed buffer (in float4)
    // ---- 0: expose weight * bucket, tell the peers, wait for theirs
    float4 *mine_x = reinterpret_cast<float4 *>(pp.exposed[rank]) + par;
    for (int64_t i = i0 + t; i < i1; i += 256) {
        const float4 g = bucket[i];
        mine_x[i] = make_float4(weight * g.x, weight * g.y, weight * g.z, weight * g.w);
    }
    __syncthreads();
    if (t < world) {
        __threadfence_system();
        st_release_sys(pp.sig[t] + SIG_READY + rank * PEER_MAX_BLOCKS + b, epoch);
        unsigned spins = 0;
        while (ld_acquire_sys(mine + SIG_READY + t * PEER_MAX_BLOCKS + b) - epoch < 0)
            if (++spins > (1u << 26)) __trap();
    }
    __syncthreads();
    // ---- 1: sum in rank order
    for (int64_t i = i0 + t; i < i1; i += 256) {
        float4 v[W];
#pragma unroll
        for (int r = 0; r < W; ++r) v[r] = ld_sys_v4(pp.exposed[r] + 4 * (par + i));
        float4 acc = v[0];
#pragma unroll
        for (int r = 1; r < W; ++r) { acc.x += v[r].x; acc.y += v[r].y; acc.z += v[r].z; acc.w += v[r].w; }
        bucket[i] = acc;
    }
    if (t == 0) mine[SIG_EPOCH + b] = epoch;
}

}  // namespace

// Map another process's allocation (a cudaIpcMemHandle_t exported there, e.g. by torch's storage._share_cuda_()) into
// the CURRENT device's context, with peer access to the exporting device enabled on demand: kernels of this device may
// dereference *base_out.  One mapping per handle and process (the caller caches); dn4gl_ipc_close unmaps.
extern "C" int dn4gl_ipc_open(const void *handle, void **base_out) {
    DN_ARG(handle != nullptr && base_out != nullptr);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    const cudaError_t rc = cudaIpcOpenMemHandle(base_out, h, cudaIpcMemLazyEnablePeerAccess);
    if (rc != cudaSuccess) (void)cudaGetLastError();      // the caller falls back to the library collective: leave no sticky error
    DN_CUDA(rc);
    return DN4GL_OK;
}

extern "C" int dn4gl_ipc_close(void *base) {
    if (base == nullptr) return DN4GL_OK;
    DN_CUDA(cudaIpcCloseMemHandle(base));
    return DN4GL_OK;
}

extern "C" int32_t dn4gl_peer_allreduce_grid(int64_t n) {
    if (n <= 0) return 0;
    const int64_t n4 = (n + 3) / 4, want = (n4 + 511) / 512;
    return static_cast<int32_t>(want > PEER_MAX_BLOCKS ? PEER_MAX_BLOCKS : want);
}

extern "C" int dn4gl_peer_allreduce_f32(float *bucket, int64_t n, float weight, float *const *exposed, int32_t *const *signals,
                                        int32_t rank, int32_t world, void *stream) {
    DN_ARG(world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world && n >= 0 && n % 4 == 0 && exposed && signals);
    if (n == 0) return DN4GL_OK;
    DN_ARG(bucket != nullptr && aligned16(bucket));
    PeerPtrs pp = {};
    for (int r = 0; r < world; ++r) {
        DN_ARG(exposed[r] != nullptr && signals[r] != nullptr && aligned16(exposed[r]));
        pp.exposed[r] = exposed[r];
        pp.sig[r] = signals[r];
    }
    const int grid = dn4gl_peer_allreduce_grid(n);
    cudaStream_t st = as_stream(stream);
    float4 *b4 = reinterpret_cast<float4 *>(bucket);
    const int rk = static_cast<int>(rank);
    switch (world) {
    case 1: peer_allreduce_kernel<1><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    case 2: peer_allreduce_kernel<2><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    case 3: peer_allreduce_kernel<3><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    case 4: peer_allreduce_kernel<4><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    case 5: peer_allreduce_kernel<5><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    case 6: peer_allreduce_kernel<6><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    case 7: peer_allreduce_kernel<7><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    default: peer_allreduce_kernel<8><<<grid, 256, 0, st>>>(pp, rk, n / 4, weight, b4); break;
    }
    DN_LAUNCHED();
    return DN4GL_OK;
}
