// libdn4gl.so -- K1, tiled variant: sum aggregation as a warp-specialised producer/consumer pipeline.
//
// A mini-batch is block-diagonal: every neighbour of a row of graph g is a row of graph g.  Rows are cut into TILES
// (dn4gl_make_row_tiles): tile k starts at the first graph boundary inside [kC, (k+1)C), or at kC itself when a graph is
// longer than the window (a "cut" tile).  A persistent CTA walks tiles t = blockIdx.x, += gridDim.x through a ring of
// STAGES shared-memory buffers:
//   * warp 0 (one elected lane) is the PRODUCER: for every tile it issues three bulk asynchronous copies on the TMA
//     engine's 1-D path (cp.async.bulk ... mbarrier::complete_tx; SASS UBLKCP) -- the tile's feature rows x[r0:r1)
//     (one contiguous slab), its row_ptr slice and its col slice -- into the next free stage, as soon as the consumers
//     have released it (empty mbarrier);
//   * warps 1..15 are CONSUMERS: they wait on the stage's full mbarrier, resolve every neighbour index against shared
//     memory, accumulate in CSR order and stream the output rows to HBM with 128-bit stores.
// DRAM therefore sees each feature row once as a streaming read and each output row once as a streaming write (the
// algorithmic bytes of SURVEY.md 8(d)); there is no dependent row_ptr -> col -> x gather chain on DRAM (the latency
// chain that bounded the per-row kernel, profiles/r1a), and the loads of tile k+1 overlap the arithmetic of tile k.
//
// Correctness never depends on the tiling: an index outside the staged window, a col position beyond the staged
// slice, or a tile larger than a stage falls back to global loads inside the same kernel.
//
// Rows with more than SPLIT neighbours:
//   * in a graph-aligned (self-contained) tile all neighbours are in shared memory: the sub-groups of the row's warp
//     split the list and combine with a fixed butterfly (deterministic);
//   * in a cut tile (graph longer than the window) the neighbours are in HBM: such rows are listed once per tiling
//     (dn4gl_make_row_tiles) and run FIRST as "virtual tiles": all 15 consumer warps of a CTA stride one row's list
//     and combine through the idle stage buffer in a fixed order.
// Per-row accumulation order for rows with <= SPLIT neighbours is CSR order with separately rounded adds, i.e.
// bit-identical to the per-row kernel and to the sequential oracle.
#include "common.cuh"

constexpr int TP_NCW_MAX = 31;                // consumer warps: 15 (512 threads, <=128 registers) or 31 (1024 threads, 64)
constexpr int TP_SPLIT = 64;                  // rows above this many neighbours are split (== graph.py HEAVY_THRESHOLD)
constexpr int TP_MAX_STAGES = 4;
constexpr uint32_t TP_BULK_CHUNK = 32768u;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// ---- optional per-CTA timeline (debug build -DDN4GL_TIMELINE = libdn4gl_tl.so, tools/k1_timeline.py): %globaltimer
// stamps of the first consumer warp's lane 0 and of the producer, 32 slots per CTA: [0] entry, [1] after the prologue,
// then per work item two stamps (full barrier passed, item done); producer stamps in slots 16.. (stage free).
// Compiled out of the product build.
#ifdef DN4GL_TIMELINE
__device__ unsigned long long g_timeline[148 * 32];
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TL_STAMP(slot) do { if ((slot) < 32 && blockIdx.x < 148) g_timeline[blockIdx.x * 32 + (slot)] = gtime(); } while (0)
#define TL_STAMP_LO(slot) do { if ((slot) < 16) TL_STAMP(slot); } while (0)
extern "C" int dn4gl_debug_read_timeline(unsigned long long *host_out) {
    return cudaMemcpyFromSymbol(host_out, g_timeline, sizeof(unsigned long long) * 148 * 32) == cudaSuccess ? 0 : -2;
}
extern "C" int dn4gl_debug_clear_timeline(void) {
    static unsigned long long zeros[148 * 32];
    return cudaMemcpyToSymbol(g_timeline, zeros, sizeof(zeros)) == cudaSuccess ? 0 : -2;
}
#else
#define TL_STAMP(slot) do { } while (0)
#define TL_STAMP_LO(slot) do { } while (0)
#endif

template <int NCW>
__device__ __forceinline__ void consumer_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NCW * 32) : "memory"); }

// shared-memory carve-up of ONE stage: [cap_rows][DV] float4 feature rows | col slice | row_ptr slice
struct TileCfg {
    int stages, cap_rows, cap_nnz;
    uint32_t stage_bytes, off_col, off_rp;
};
__host__ __device__ inline TileCfg tile_cfg(int smem_bytes, int stages, int DV, int nnz_per_row) {
    TileCfg L;
    L.stages = stages;
    L.stage_bytes = (static_cast<uint32_t>(smem_bytes) / stages) & ~127u;
    const int per_row = DV * 16 + nnz_per_row * 4 + 4;
    int cap = (static_cast<int>(L.stage_bytes) - 96) / per_row;   // 96: alignment pads of the two index slices
    if (cap < 0) cap = 0;
    L.cap_rows = cap;
    L.cap_nnz = cap * nnz_per_row;
    L.off_col = static_cast<uint32_t>(cap) * DV * 16u;
    L.off_rp = L.off_col + ((((static_cast<uint32_t>(L.cap_nnz) + 8u) * 4u) + 15u) & ~15u);
    return L;
}

// explicit shared-state-space loads on 32-bit addresses: no generic->shared conversion and no 64-bit address
// registers in the inner loops (the generic-pointer version spent most of its issue slots on address arithmetic,
// profiles/r1b).  volatile keeps them behind the mbarrier wait.
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ int lds32(uint32_t a) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// butterfly over the sub-groups of a warp (fixed order -> deterministic); every sub-group ends with the total
template <int LANES>
__device__ __forceinline__ void subgroup_allreduce(float4 &acc) {
#pragma unroll
    for (int o = LANES; o < 32; o <<= 1) {
        float4 t;
        t.x = __shfl_xor_sync(0xffffffffu, acc.x, o); t.y = __shfl_xor_sync(0xffffffffu, acc.y, o);
        t.z = __shfl_xor_sync(0xffffffffu, acc.z, o); t.w = __shfl_xor_sync(0xffffffffu, acc.w, o);
        add4(acc, t);
    }
}

// a staged tile seen through 32-bit shared addresses (all pre-offset so that absolute row / col positions index them):
//   row_ptr[i]  at rp_a + 4*i      (i in [r0, r1])        col[q] at col_a + 4*q   (q in [e0, e0 + nst))
//   x[c, lane's float4 k] at x_a + c*ROWB + k*LANES*16     (c in [r0, r1))
template <int LANES, int VEC>
struct TileAddr {
    static constexpr int DV = LANES * VEC;
    static constexpr uint32_t ROWB = DV * 16u;
    uint32_t rp_a, col_a, x_a;
    int r0, r1, e0, nst;
};

// CHECKED path (cut / unverified tiles, partially staged col slices, tiles larger than a stage when !STAGED):
// every index is tested against the staged window and falls back to global loads.
template <int LANES, int VEC, int NCW, bool STAGED>
__device__ __forceinline__ void process_tile(const TileAddr<LANES, VEC> &ta, const int32_t *__restrict__ row_ptr,
                                             const int32_t *__restrict__ col, const float4 *__restrict__ x,
                                             float4 *__restrict__ out, float self_scale, bool cut, int cw, int lane) {
    constexpr int RPW = 32 / LANES;   // rows per warp iteration
    constexpr int DV = LANES * VEC;
    constexpr uint32_t ROWB = DV * 16u;
    const int sub = lane / LANES, sl = lane % LANES;
    auto colv = [&](int q) -> int {
        return (STAGED && q - ta.e0 < ta.nst) ? lds32(ta.col_a + 4u * static_cast<uint32_t>(q)) : __ldg(col + q);
    };
    auto xv = [&](int c, int k) -> float4 {
        return (STAGED && c >= ta.r0 && c < ta.r1) ? lds128(ta.x_a + static_cast<uint32_t>(c) * ROWB + k * (LANES * 16))
                                                   : ldg4(x + static_cast<int64_t>(c) * DV + sl + k * LANES);
    };
#pragma unroll 1
    for (int rb = ta.r0 + cw * RPW; rb < ta.r1; rb += NCW * RPW) {
        const int row = rb + sub;
        const bool valid = row < ta.r1;
        int beg = 0, end = 0;
        if (valid) {
            beg = STAGED ? lds32(ta.rp_a + 4u * static_cast<uint32_t>(row)) : __ldg(row_ptr + row);
            end = STAGED ? lds32(ta.rp_a + 4u * static_cast<uint32_t>(row) + 4u) : __ldg(row_ptr + row + 1);
        }
        const bool big = valid && (end - beg > TP_SPLIT);
        if (valid && (!big || (LANES == 32 && !cut))) {
            float4 acc[VEC];
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[k] = zero4();
            int p = beg;
            if constexpr (VEC == 1) {   // four neighbours in flight: out-of-window rows come from L2 / HBM
#pragma unroll 1
                for (; p + 4 <= end; p += 4) {
                    const int c0 = colv(p), c1 = colv(p + 1), c2 = colv(p + 2), c3 = colv(p + 3);
                    const float4 v0 = xv(c0, 0), v1 = xv(c1, 0), v2 = xv(c2, 0), v3 = xv(c3, 0);
                    add4(acc[0], v0); add4(acc[0], v1); add4(acc[0], v2); add4(acc[0], v3);
                }
            }
#pragma unroll 1
            for (; p + 2 <= end; p += 2) {
                const int c0 = colv(p), c1 = colv(p + 1);
                float4 v0[VEC], v1[VEC];
#pragma unroll
                for (int k = 0; k < VEC; ++k) { v0[k] = xv(c0, k); v1[k] = xv(c1, k); }
#pragma unroll
                for (int k = 0; k < VEC; ++k) { add4(acc[k], v0[k]); add4(acc[k], v1[k]); }
            }
            if (p < end) {
                const int c0 = colv(p);
#pragma unroll
                for (int k = 0; k < VEC; ++k) add4(acc[k], xv(c0, k));
            }
            if (self_scale != 0.f) {
#pragma unroll
                for (int k = 0; k < VEC; ++k) axpy4_rn(acc[k], self_scale, xv(row, k));
            }
#pragma unroll
            for (int k = 0; k < VEC; ++k) out[static_cast<int64_t>(row) * DV + sl + k * LANES] = acc[k];
        }
        if constexpr (LANES < 32) {
            // long rows of this warp iteration, one after the other, split over the RPW sub-groups
            unsigned m = __ballot_sync(0xffffffffu, big && !cut);
            while (m) {
                const int src_lane = __ffs(m) - 1;   // first lane of the owning sub-group
                m &= ~(((1u << LANES) - 1u) << src_lane);
                const int brow = rb + src_lane / LANES;
                const int bbeg = __shfl_sync(0xffffffffu, beg, src_lane), bend = __shfl_sync(0xffffffffu, end, src_lane);
                float4 acc = zero4();
#pragma unroll 1
                for (int p = bbeg + sub; p < bend; p += 2 * RPW) {
                    const int c0 = colv(p);
                    const int c1 = (p + RPW < bend) ? colv(p + RPW) : -1;
                    const float4 v0 = xv(c0, 0);
                    float4 v1 = zero4();
                    if (c1 >= 0) v1 = xv(c1, 0);
                    add4(acc, v0);
                    if (c1 >= 0) add4(acc, v1);
                }
                subgroup_allreduce<LANES>(acc);
                if (sub == 0) {
                    if (self_scale != 0.f) axpy4_rn(acc, self_scale, xv(brow, 0));
                    out[static_cast<int64_t>(brow) * DV + sl] = acc;
                }
            }
        }
    }
}

// FAST path: a verified self-contained tile (every col index inside [r0, r1), checked once by dn4gl_make_row_tiles)
// whose col slice is fully staged.  No window checks, no fallbacks: per neighbour one 32-bit and VEC 128-bit shared
// loads, one integer multiply-add and 2*VEC packed adds.  This is the loop that bounds the kernel.
template <int LANES, int VEC, int NCW>
__device__ __forceinline__ void process_tile_fast(const TileAddr<LANES, VEC> &ta, float4 *__restrict__ out,
                                                  float self_scale, int cw, int lane) {
    constexpr int RPW = 32 / LANES;
    constexpr int DV = LANES * VEC;
    constexpr uint32_t ROWB = DV * 16u;
    constexpr uint32_t KB = LANES * 16u;   // byte distance between a lane's consecutive float4 of one row
    const int sub = lane / LANES, sl = lane % LANES;
    const uint32_t xa = ta.x_a, ca_base = ta.col_a;
    float4 *outl = out + sl;
#pragma unroll 1
    for (int rb = ta.r0 + cw * RPW; rb < ta.r1; rb += NCW * RPW) {
        const int row = rb + sub;
        const bool valid = row < ta.r1;
        int beg = 0, end = 0;
        if (valid) {
            const uint32_t ra = ta.rp_a + 4u * static_cast<uint32_t>(row);
            beg = lds32(ra);
            end = lds32(ra + 4u);
        }
        const bool big = (LANES < 32) && (end - beg > TP_SPLIT);
        if (valid && !big) {
            float4 acc[VEC];
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[k] = zero4();
            uint32_t ca = ca_base + 4u * static_cast<uint32_t>(beg);
            const uint32_t ce = ca_base + 4u * static_cast<uint32_t>(end);
#pragma unroll 1
            for (; ca + 16u <= ce; ca += 16u) {
                const uint32_t a0 = xa + static_cast<uint32_t>(lds32(ca)) * ROWB;
                const uint32_t a1 = xa + static_cast<uint32_t>(lds32(ca + 4u)) * ROWB;
                const uint32_t a2 = xa + static_cast<uint32_t>(lds32(ca + 8u)) * ROWB;
                const uint32_t a3 = xa + static_cast<uint32_t>(lds32(ca + 12u)) * ROWB;
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    const float4 v0 = lds128(a0 + k * KB), v1 = lds128(a1 + k * KB);
                    const float4 v2 = lds128(a2 + k * KB), v3 = lds128(a3 + k * KB);
                    add4(acc[k], v0); add4(acc[k], v1); add4(acc[k], v2); add4(acc[k], v3);
                }
            }
#pragma unroll 1
            for (; ca < ce; ca += 4u) {
                const uint32_t a0 = xa + static_cast<uint32_t>(lds32(ca)) * ROWB;
#pragma unroll
                for (int k = 0; k < VEC; ++k) add4(acc[k], lds128(a0 + k * KB));
            }
            if (self_scale != 0.f) {
                const uint32_t a0 = xa + static_cast<uint32_t>(row) * ROWB;
#pragma unroll
                for (int k = 0; k < VEC; ++k) axpy4_rn(acc[k], self_scale, lds128(a0 + k * KB));
            }
            float4 *o = outl + static_cast<int64_t>(row) * DV;
#pragma unroll
            for (int k = 0; k < VEC; ++k) o[k * LANES] = acc[k];
        }
        if constexpr (LANES < 32) {
            unsigned m = __ballot_sync(0xffffffffu, valid && big);
            while (m) {   // long rows of this iteration, split over the RPW sub-groups of the warp
                const int src_lane = __ffs(m) - 1;
                m &= ~(((1u << LANES) - 1u) << src_lane);
                const int brow = rb + src_lane / LANES;
                const int bbeg = __shfl_sync(0xffffffffu, beg, src_lane), bend = __shfl_sync(0xffffffffu, end, src_lane);
                float4 acc = zero4();
                uint32_t ca = ca_base + 4u * static_cast<uint32_t>(bbeg + sub);
                const uint32_t ce = ca_base + 4u * static_cast<uint32_t>(bend);
#pragma unroll 1
                for (; ca + 12u * RPW < ce; ca += 16u * RPW) {
                    const uint32_t a0 = xa + static_cast<uint32_t>(lds32(ca)) * ROWB;
                    const uint32_t a1 = xa + static_cast<uint32_t>(lds32(ca + 4u * RPW)) * ROWB;
                    const uint32_t a2 = xa + static_cast<uint32_t>(lds32(ca + 8u * RPW)) * ROWB;
                    const uint32_t a3 = xa + static_cast<uint32_t>(lds32(ca + 12u * RPW)) * ROWB;
                    const float4 v0 = lds128(a0), v1 = lds128(a1), v2 = lds128(a2), v3 = lds128(a3);
                    add4(acc, v0); add4(acc, v1); add4(acc, v2); add4(acc, v3);
                }
#pragma unroll 1
                for (; ca < ce; ca += 4u * RPW) add4(acc, lds128(xa + static_cast<uint32_t>(lds32(ca)) * ROWB));
                subgroup_allreduce<LANES>(acc);
                if (sub == 0) {
                    if (self_scale != 0.f) axpy4_rn(acc, self_scale, lds128(xa + static_cast<uint32_t>(brow) * ROWB));
                    outl[static_cast<int64_t>(brow) * DV] = acc;
                }
            }
        }
    }
}

// one listed long row of a cut tile, reduced by all consumer warps of the CTA through `scratch` (an idle stage)
template <int LANES, int VEC, int NCW>
__device__ __forceinline__ void process_heavy_row(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col,
                                                  const float4 *__restrict__ x, float4 *__restrict__ out, int row,
                                                  float self_scale, float4 *scratch, int cw, int lane) {
    constexpr int RPW = 32 / LANES;
    constexpr int DV = LANES * VEC;
    constexpr int SG = NCW * RPW;   // sub-groups in the CTA
    constexpr int UH = (VEC == 4 || (NCW > 15 && VEC > 1)) ? 2 : 4;
    const int sub = lane / LANES, sl = lane % LANES;
    const int sg = cw * RPW + sub;
    const int beg = __ldg(row_ptr + row), end = __ldg(row_ptr + row + 1);
    float4 acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = zero4();
    for (int p = beg + sg; p < end; p += SG * UH) {
        int c[UH];
#pragma unroll
        for (int u = 0; u < UH; ++u) c[u] = (p + u * SG < end) ? __ldg(col + p + u * SG) : -1;
        float4 v[UH][VEC];
#pragma unroll
        for (int u = 0; u < UH; ++u)
            if (c[u] >= 0) {
#pragma unroll
                for (int k = 0; k < VEC; ++k) v[u][k] = ldg4(x + static_cast<int64_t>(c[u]) * DV + sl + k * LANES);
            }
#pragma unroll
        for (int u = 0; u < UH; ++u)
            if (c[u] >= 0) {
#pragma unroll
                for (int k = 0; k < VEC; ++k) add4(acc[k], v[u][k]);
            }
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) scratch[static_cast<size_t>(sg) * DV + sl + k * LANES] = acc[k];
    consumer_bar_sync<NCW>();
    if (cw == 0) {
        // sub-group `sub` adds the partials sub, sub+RPW, ... in ascending order, then a fixed butterfly over sub-groups
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = zero4();
        for (int g = sub; g < SG; g += RPW) {
#pragma unroll
            for (int k = 0; k < VEC; ++k) add4(acc[k], scratch[static_cast<size_t>(g) * DV + sl + k * LANES]);
        }
#pragma unroll
        for (int o = LANES; o < 32; o <<= 1) {
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                float4 t;
                t.x = __shfl_xor_sync(0xffffffffu, acc[k].x, o); t.y = __shfl_xor_sync(0xffffffffu, acc[k].y, o);
                t.z = __shfl_xor_sync(0xffffffffu, acc[k].z, o); t.w = __shfl_xor_sync(0xffffffffu, acc[k].w, o);
                add4(acc[k], t);
            }
        }
        if (sub == 0) {
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
                if (self_scale != 0.f) axpy4_rn(acc[k], self_scale, ldg4(x + static_cast<int64_t>(row) * DV + sl + k * LANES));
                out[static_cast<int64_t>(row) * DV + sl + k * LANES] = acc[k];
            }
        }
    }
    // the scratch words were written through the generic proxy and the stage is refilled through the async proxy
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

template <int LANES, int VEC, int NCW>
__global__ void __launch_bounds__((NCW + 1) * 32, 1)
spmm_pipe_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col, const float4 *__restrict__ x,
                 float4 *__restrict__ out, const int4 *__restrict__ tiles, int num_tiles,
                 const int32_t *__restrict__ heavy_list, const int32_t *__restrict__ heavy_count, float self_scale,
                 const float *__restrict__ eps_dev, int smem_bytes, int stages, int nnz_per_row) {
    constexpr int DV = LANES * VEC;
    if (eps_dev != nullptr) self_scale = 1.f + __ldg(eps_dev);   // trainable GIN eps lives on the device
    if (threadIdx.x == 32) TL_STAMP(0);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t full_bar[TP_MAX_STAGES], empty_bar[TP_MAX_STAGES];
    const TileCfg L = tile_cfg(smem_bytes, stages, DV, nnz_per_row);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], NCW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int H = (heavy_list != nullptr && heavy_count != nullptr) ? __ldg(heavy_count) : 0;
    const int total = H + num_tiles;
    if (threadIdx.x == 32) TL_STAMP(1);

    if (warp == 0) {
        // ------------------------------------------------------------------ producer (one lane)
        if (lane != 0) return;
        int s = 0;
        uint32_t use = 0;   // how many times stage s has been filled before
        [[maybe_unused]] int tl_p = 16;
        for (int t = blockIdx.x; t < total; t += gridDim.x) {
            if (use > 0) mbar_wait(&empty_bar[s], (use - 1) & 1u);
            TL_STAMP(tl_p); ++tl_p;
            bool issued = false;
            if (t >= H) {
                const int4 td = __ldg(tiles + (t - H));
                const int r0 = td.x, r1 = td.y, e0 = td.z, e1 = td.w & 0x7fffffff;
                const int rows = r1 - r0;
                if (rows > 0 && rows <= L.cap_rows) {
                    unsigned char *base = smem_raw + static_cast<size_t>(s) * L.stage_bytes;
                    const uint32_t xbytes = static_cast<uint32_t>(rows) * DV * 16u;
                    const int a0 = r0 & ~3;
                    const uint32_t rp_bytes = static_cast<uint32_t>(((r1 + 1 - a0) + 3) & ~3) * 4u;
                    const int c0 = e0 & ~3;
                    const int nst = min(e1 - e0, L.cap_nnz);
                    const uint32_t col_bytes = nst > 0 ? static_cast<uint32_t>(((e0 + nst - c0) + 3) & ~3) * 4u : 0u;
                    mbar_expect_tx(&full_bar[s], xbytes + rp_bytes + col_bytes);
                    bulk_g2s(base + L.off_rp, row_ptr + a0, rp_bytes, &full_bar[s]);
                    if (col_bytes) bulk_g2s(base + L.off_col, col + c0, col_bytes, &full_bar[s]);
                    const char *src = reinterpret_cast<const char *>(x + static_cast<int64_t>(r0) * DV);
                    for (uint32_t off = 0; off < xbytes; off += TP_BULK_CHUNK) {
                        const uint32_t n = xbytes - off < TP_BULK_CHUNK ? xbytes - off : TP_BULK_CHUNK;
                        bulk_g2s(base + off, src + off, n, &full_bar[s]);
                    }
                    issued = true;
                }
            }
            if (!issued) mbar_arrive(&full_bar[s]);
            if (++s == stages) { s = 0; ++use; }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    const int cw = warp - 1;
    int s = 0;
    uint32_t use = 0;
    [[maybe_unused]] int tl_c = 2;
    for (int t = blockIdx.x; t < total; t += gridDim.x) {
        unsigned char *base = smem_raw + static_cast<size_t>(s) * L.stage_bytes;
        if (t < H) {
            const int row = __ldg(heavy_list + t);
            mbar_wait(&full_bar[s], use & 1u);
            if (threadIdx.x == 32) TL_STAMP_LO(tl_c);
            process_heavy_row<LANES, VEC, NCW>(row_ptr, col, x, out, row, self_scale, reinterpret_cast<float4 *>(base), cw, lane);
        } else {
            const int4 td = __ldg(tiles + (t - H));
            const int rows = td.y - td.x;
            mbar_wait(&full_bar[s], use & 1u);
            if (threadIdx.x == 32) TL_STAMP_LO(tl_c);
            if (rows > 0) {
                const bool open = td.w < 0;                          // cut inside a graph or not verified self-contained
                const bool cut = heavy_list != nullptr && open;      // its long rows are on the heavy list
                const int nnz = (td.w & 0x7fffffff) - td.z;
                TileAddr<LANES, VEC> ta;
                {   // pre-offset 32-bit shared addresses (unsigned wrap-around is intended)
                    const uint32_t sbase = smem_u32(base);
                    const int a0 = td.x & ~3, c0 = td.z & ~3;
                    ta.rp_a = sbase + L.off_rp - 4u * static_cast<uint32_t>(a0);
                    ta.col_a = sbase + L.off_col - 4u * static_cast<uint32_t>(c0);
                    ta.x_a = sbase + static_cast<uint32_t>(lane % LANES) * 16u -
                             static_cast<uint32_t>(td.x) * TileAddr<LANES, VEC>::ROWB;
                    ta.r0 = td.x; ta.r1 = td.y; ta.e0 = td.z; ta.nst = min(nnz, L.cap_nnz);
                }
                if (rows <= L.cap_rows && !open && nnz <= L.cap_nnz)
                    process_tile_fast<LANES, VEC, NCW>(ta, out, self_scale, cw, lane);
                else if (rows <= L.cap_rows)
                    process_tile<LANES, VEC, NCW, true>(ta, row_ptr, col, x, out, self_scale, cut, cw, lane);
                else
                    process_tile<LANES, VEC, NCW, false>(ta, row_ptr, col, x, out, self_scale, cut, cw, lane);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
        if (threadIdx.x == 32) TL_STAMP_LO(tl_c + 1);
        tl_c += 2;
        if (++s == stages) { s = 0; ++use; }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// tiling.  boundary(k) = first graph start in [kC, (k+1)C) if there is one (aligned), else kC (cut inside a graph
// longer than the window); boundary(T) = N.  tile k = [boundary(k), boundary(k+1)), desc = {r0, r1, e0, e1 | cut<<31}.
__device__ __forceinline__ int tile_boundary(const int32_t *__restrict__ seg_ptr, int B, int C, int N, int k, int T,
                                             bool *aligned) {
    if (k >= T) { *aligned = true; return N; }
    const int64_t target = static_cast<int64_t>(k) * C;
    int lo = 0, hi = B;   // first g in [0, B] with seg_ptr[g] >= target
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (seg_ptr[mid] >= target) hi = mid; else lo = mid + 1;
    }
    const int gs = seg_ptr[lo];
    if (gs < target + C) { *aligned = true; return gs; }
    *aligned = false;
    return static_cast<int>(target);
}

__global__ void make_row_tiles_kernel(const int32_t *__restrict__ seg_ptr, int B, int C, const int32_t *__restrict__ row_ptr,
                                      int N, int4 *__restrict__ tiles, int T) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= T) return;
    bool a0, a1;
    const int r0 = tile_boundary(seg_ptr, B, C, N, k, T, &a0);
    const int r1 = tile_boundary(seg_ptr, B, C, N, k + 1, T, &a1);
    const int e0 = row_ptr[r0], e1 = row_ptr[r1];
    const bool cut = !(a0 && a1);
    tiles[k] = make_int4(r0, r1, e0, e1 | (cut ? static_cast<int>(0x80000000u) : 0));
}

// one warp per graph-aligned tile: any column index outside [r0, r1) (seg_ptr was not a block partition of this CSR)
// marks the tile "open", which keeps it off the unchecked fast path
__global__ void verify_tiles_kernel(const int32_t *__restrict__ col, int4 *__restrict__ tiles, int T) {
    const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= T) return;
    const int4 td = tiles[k];
    if (td.w < 0) return;
    bool bad = false;
    for (int q = td.z + lane; q < td.w; q += 32) {
        const int c = __ldg(col + q);
        bad |= (c < td.x) || (c >= td.y);
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) tiles[k].w = td.w | static_cast<int>(0x80000000u);
}

// rows with more than TP_SPLIT neighbours that live in cut tiles -> heavy_list (order irrelevant, see kernel)
__global__ void collect_cut_heavy_kernel(const int32_t *__restrict__ row_ptr, int N, int C, const int4 *__restrict__ tiles,
                                         int T, int32_t *__restrict__ heavy_list, int cap, int32_t *__restrict__ heavy_count) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= N) return;
    if (row_ptr[r + 1] - row_ptr[r] <= TP_SPLIT) return;
    int k = r / C;
    if (k >= T) k = T - 1;
    if (r < tiles[k].x) --k;
    if (tiles[k].w < 0) {
        const int i = atomicAdd(heavy_count, 1);
        if (i < cap) heavy_list[i] = r;
    }
}

extern "C" int dn4gl_make_row_tiles(const int32_t *seg_ptr, int32_t B, int32_t window_rows, const int32_t *row_ptr,
                                    const int32_t *col, int64_t N, int32_t *tile_desc, int32_t num_tiles,
                                    int32_t *heavy_list, int32_t heavy_cap, int32_t *heavy_count, void *stream) {
    DN_ARG(seg_ptr && row_ptr && tile_desc && B >= 0 && window_rows > 0 && num_tiles >= 0 && N >= 0 && N < (1ll << 31));
    DN_ARG(static_cast<int64_t>(num_tiles) * window_rows >= N && aligned16(tile_desc));
    cudaStream_t st = as_stream(stream);
    int launched = 0;
    if (heavy_count) DN_CUDA(cudaMemsetAsync(heavy_count, 0, sizeof(int32_t), st));
    if (num_tiles > 0) {
        make_row_tiles_kernel<<<(num_tiles + 255) / 256, 256, 0, st>>>(seg_ptr, B, window_rows, row_ptr, static_cast<int>(N),
                                                                      reinterpret_cast<int4 *>(tile_desc), num_tiles);
        // col == NULL: the caller vouches that the CSR is block-diagonal over seg_ptr (e.g. dn4gl_tu_conj_direct_fill wrote it
        // graph by graph): the per-tile column check -- every col entry read once, 11 us at C2 -- is skipped
        if (col != nullptr)
            verify_tiles_kernel<<<(num_tiles * 32 + 255) / 256, 256, 0, st>>>(col, reinterpret_cast<int4 *>(tile_desc), num_tiles);
        launched += col != nullptr ? 2 : 1;
        if (heavy_list && heavy_count && N > 0) {
            collect_cut_heavy_kernel<<<static_cast<unsigned>(ceil_div64(N, 256)), 256, 0, st>>>(
                row_ptr, static_cast<int>(N), window_rows, reinterpret_cast<const int4 *>(tile_desc), num_tiles, heavy_list,
                heavy_cap, heavy_count);
            ++launched;
        }
    }
    if (launched) DN_LAUNCHED_N(launched);
    return DN4GL_OK;
}

/* rows of width D that one pipeline stage holds for (smem_bytes, stages, nnz_per_row) */
extern "C" int32_t dn4gl_spmm_tiled_cap_rows(int32_t D, int32_t smem_bytes, int32_t stages, int32_t nnz_per_row) {
    if (D <= 0 || D % 4 != 0 || stages < 1 || stages > TP_MAX_STAGES || nnz_per_row < 1) return 0;
    return tile_cfg(smem_bytes, stages, D / 4, nnz_per_row).cap_rows;
}

template <int LANES, int VEC, int NCW>
static int launch_pipe(const int32_t *row_ptr, const int32_t *col, const float *x, float *out, const int32_t *tile_desc,
                       int num_tiles, const int32_t *heavy_list, const int32_t *heavy_count, int heavy_cap,
                       float self_scale, const float *eps_dev, int smem_bytes, int stages, int nnz_per_row, cudaStream_t st) {
    static int attr_done = 0;
    if (attr_done < smem_bytes) {
        if (cudaFuncSetAttribute(spmm_pipe_kernel<LANES, VEC, NCW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 smem_bytes) != cudaSuccess)
            return -1;
        attr_done = smem_bytes;
    }
    // one persistent CTA per SM: the whole shared memory is its ring
    int64_t want = static_cast<int64_t>(num_tiles) + (heavy_list ? heavy_cap : 0);
    int grid = static_cast<int>(want < dn4gl_num_sms() ? want : dn4gl_num_sms());
    if (grid < 1) grid = 1;
    spmm_pipe_kernel<LANES, VEC, NCW><<<grid, (NCW + 1) * 32, smem_bytes, st>>>(
        row_ptr, col, reinterpret_cast<const float4 *>(x), reinterpret_cast<float4 *>(out),
        reinterpret_cast<const int4 *>(tile_desc), num_tiles, heavy_list, heavy_count, self_scale, eps_dev, smem_bytes, stages,
        nnz_per_row);
    return 0;
}

extern "C" int dn4gl_spmm_tiled_f32(const int32_t *row_ptr, const int32_t *col, const float *x, float *out, int64_t N,
                                    int32_t D, float self_scale, const float *eps_dev, const int32_t *tile_desc, int32_t num_tiles,
                                    const int32_t *heavy_list, const int32_t *heavy_count, int32_t heavy_cap,
                                    int32_t smem_bytes, int32_t stages, int32_t nnz_per_row, int32_t warps,
                                    void *stream) {
    DN_ARG(warps == 16 || warps == 24 || warps == 32);
    DN_ARG(N >= 0 && D > 0 && D % 4 == 0 && num_tiles >= 0 && smem_bytes >= 16 * 1024 && smem_bytes <= 220 * 1024);
    DN_ARG(stages >= 1 && stages <= TP_MAX_STAGES && nnz_per_row >= 1 && nnz_per_row <= 64);
    if (N == 0 || num_tiles == 0) return DN4GL_OK;
    DN_ARG(row_ptr && col && x && out && tile_desc && aligned16(x) && aligned16(out) && aligned16(row_ptr) &&
           aligned16(col) && aligned16(tile_desc));
    DN_ARG((heavy_list == nullptr) == (heavy_count == nullptr));
    {   // the CTA-wide reduction of listed rows uses one stage as scratch: (warps - 1) x (32/LANES) partial rows
        const int dv = D / 4, lanes = dv < 32 ? dv : 32;
        const int64_t scratch = static_cast<int64_t>((dv <= 32 ? warps : 16) - 1) * (32 / lanes) * dv * 16;
        DN_ARG(heavy_list == nullptr || scratch <= ((smem_bytes / stages) & ~127));
    }
    cudaStream_t st = as_stream(stream);
    int rc = 0;
#define PIPE_ARGS row_ptr, col, x, out, tile_desc, num_tiles, heavy_list, heavy_count, heavy_cap, self_scale, eps_dev, smem_bytes, stages, nnz_per_row, st
#define PIPE_CASE(L, V)                                                          \
    if constexpr (V == 1) {                                                      \
        if (warps == 32) rc = launch_pipe<L, V, 31>(PIPE_ARGS);                  \
        else if (warps == 24) rc = launch_pipe<L, V, 23>(PIPE_ARGS);             \
        else rc = launch_pipe<L, V, 15>(PIPE_ARGS);                              \
    } else {                                                                     \
        rc = launch_pipe<L, V, 15>(PIPE_ARGS);                                   \
    }                                                                            \
    break
    switch (D / 4) {
        case 4: PIPE_CASE(4, 1);
        case 8: PIPE_CASE(8, 1);
        case 16: PIPE_CASE(16, 1);
        case 32: PIPE_CASE(32, 1);
        case 64: PIPE_CASE(32, 2);
        case 128: PIPE_CASE(32, 4);
        default:
            dn4gl_set_error("dn4gl_spmm_tiled_f32: unsupported D=%d (supported: 16,32,64,128,256,512)", D);
            return DN4GL_EINVAL;
    }
#undef PIPE_CASE
#undef PIPE_ARGS
    if (rc != 0) {
        dn4gl_set_error("dn4gl_spmm_tiled_f32: cudaFuncSetAttribute(MaxDynamicSharedMemorySize=%d) failed", smem_bytes);
        return DN4GL_ECUDA;
    }
    DN_LAUNCHED();
    return DN4GL_OK;
}
