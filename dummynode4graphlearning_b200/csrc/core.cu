// libdn4gl.so -- error plumbing, exclusive scan, stable CSR construction.
#include <type_traits>

#include "common.cuh"

#include <string.h>

// -------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void dn4gl_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#include <atomic>
static std::atomic<long long> g_launches{0};
void dn4gl_note_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" int64_t dn4gl_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int dn4gl_version(void) { return DN4GL_ABI_VERSION; }
extern "C" const char *dn4gl_last_error(void) { return g_err; }

extern "C" int dn4gl_set_device(int device) {
    DN_CUDA(cudaSetDevice(device));
    return DN4GL_OK;
}

int dn4gl_num_sms() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, n = 148;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            cached = 148;
    }
    return cached;
}

// -------------------------------------------------------------------------------------------
// exclusive scan (int32).  Tile = 1024 threads x 4 items.  n <= TILE: one launch.  Otherwise
// reduce -> scan of tile sums (one CTA) -> downsweep: three launches, no atomics, deterministic.
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_ITEMS = 4;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ int block_exclusive_scan(int v, int *total, int *smem /* 33 ints */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) smem[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = (lane < (blockDim.x >> 5)) ? smem[lane] : 0;
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        smem[lane] = wi - w;           // exclusive prefix of warp sums
        if (lane == 31) smem[32] = wi;  // block total
    }
    __syncthreads();
    int res = incl - v + smem[warp];
    if (total) *total = smem[32];
    __syncthreads();
    return res;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sums(const int32_t *__restrict__ in, int64_t n,
                                                               int32_t *__restrict__ tile_sums) {
    __shared__ int sm[33];
    int64_t base = static_cast<int64_t>(blockIdx.x) * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    int s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k)
        if (base + k < n) s += in[base + k];
    int total;
    block_exclusive_scan(s, &total, sm);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// single CTA: in-place exclusive scan of m tile sums
__global__ void __launch_bounds__(SCAN_THREADS) scan_of_sums(int32_t *__restrict__ sums, int64_t m) {
    __shared__ int sm[33];
    int carry = 0;
    for (int64_t start = 0; start < m; start += SCAN_THREADS) {
        int64_t i = start + threadIdx.x;
        int v = (i < m) ? sums[i] : 0;
        int total;
        int ex = block_exclusive_scan(v, &total, sm);
        if (i < m) sums[i] = ex + carry;
        carry += total;
    }
}

// RAW_SUMS: tile_offsets holds the UNSCANNED tile sums and every CTA adds up the ones before it itself (at most
// SCAN_RAW_MAX_TILES of them: a few loads per thread) -- saves the single-CTA scan_of_sums launch in between.
constexpr int SCAN_RAW_MAX_TILES = 8192;
template <bool RAW_SUMS>
__global__ void __launch_bounds__(SCAN_THREADS) scan_downsweep(const int32_t *in, int32_t *out, int64_t n,
                                                               const int32_t *__restrict__ tile_offsets) {
    __shared__ int sm[33];
    int64_t base = static_cast<int64_t>(blockIdx.x) * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS];
    int s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        v[k] = (base + k < n) ? in[base + k] : 0;
        s += v[k];
    }
    int tile_off = 0;
    if (tile_offsets) {
        if constexpr (RAW_SUMS) {
            int part = 0;
            for (int t = threadIdx.x; t < static_cast<int>(blockIdx.x); t += SCAN_THREADS) part += tile_offsets[t];
            block_exclusive_scan(part, &tile_off, sm);
        } else {
            tile_off = tile_offsets[blockIdx.x];
        }
    }
    int total;
    int ex = block_exclusive_scan(s, &total, sm) + tile_off;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (base + k < n) out[base + k] = ex;
        ex += v[k];
        if (base + k == n - 1) out[n] = ex;  // grand total in the extra slot
    }
    if (n == 0 && blockIdx.x == 0 && threadIdx.x == 0) out[0] = 0;
}

extern "C" size_t dn4gl_scan_workspace_bytes(int64_t n) {
    int64_t tiles = ceil_div64(n > 0 ? n : 1, SCAN_TILE);
    return align_up(static_cast<size_t>(tiles) * sizeof(int32_t), 256);
}

extern "C" int dn4gl_exclusive_scan_i32(const int32_t *in, int32_t *out, int64_t n, void *ws, size_t ws_bytes,
                                        void *stream) {
    DN_ARG(n >= 0 && out != nullptr && (in != nullptr || n == 0));
    cudaStream_t st = as_stream(stream);
    int64_t tiles = ceil_div64(n > 0 ? n : 1, SCAN_TILE);
    if (tiles == 1) {
        scan_downsweep<false><<<1, SCAN_THREADS, 0, st>>>(in, out, n, nullptr);
        DN_LAUNCHED();
        return DN4GL_OK;
    }
    if (ws == nullptr || ws_bytes < dn4gl_scan_workspace_bytes(n)) {
        dn4gl_set_error("dn4gl_exclusive_scan_i32: workspace too small");
        return DN4GL_EWORKSPACE;
    }
    int32_t *sums = static_cast<int32_t *>(ws);
    scan_tile_sums<<<static_cast<unsigned>(tiles), SCAN_THREADS, 0, st>>>(in, n, sums);
    DN_LAUNCHED();
    if (tiles <= SCAN_RAW_MAX_TILES) {
        scan_downsweep<true><<<static_cast<unsigned>(tiles), SCAN_THREADS, 0, st>>>(in, out, n, sums);
        DN_LAUNCHED();
        return DN4GL_OK;
    }
    scan_of_sums<<<1, SCAN_THREADS, 0, st>>>(sums, tiles);
    DN_LAUNCHED();
    scan_downsweep<false><<<static_cast<unsigned>(tiles), SCAN_THREADS, 0, st>>>(in, out, n, sums);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// -------------------------------------------------------------------------------------------
// CSR build: histogram -> scan -> atomic scatter -> per-row sort by item id (restores the
// stable order, which makes the result deterministic and equal to a sequential counting sort).
__global__ void csr_histogram(const int32_t *__restrict__ key, int64_t E, int32_t *__restrict__ cnt) {
    int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e < E) atomicAdd(cnt + key[e], 1);
}

__global__ void csr_scatter(const int32_t *__restrict__ key, int64_t E, const int32_t *__restrict__ row_ptr,
                            int32_t *__restrict__ cursor, int32_t *__restrict__ eid) {
    int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e < E) {
        int k = key[e];
        int p = row_ptr[k] + atomicAdd(cursor + k, 1);
        eid[p] = static_cast<int32_t>(e);
    }
}

// sort key of an item: (primary[item], item) lexicographic; primary == NULL -> item only
__device__ __forceinline__ unsigned long long sort_key(const int32_t *__restrict__ primary, int item) {
    unsigned long long hi = primary ? static_cast<unsigned int>(primary[item]) : 0u;
    return (hi << 32) | static_cast<unsigned int>(item);
}

constexpr int LIGHT_SORT_MAX = 32;
constexpr int HEAVY_SORT_MID = 4096;

// compare-exchange of a sorting network
template <typename K>
__device__ __forceinline__ void cswap(K &a, K &b) {
    const K lo = a < b ? a : b, hi = a < b ? b : a;
    a = lo; b = hi;
}

// Batcher's odd-even merge sort of 8 keys held in registers (19 comparators)
template <typename K>
__device__ __forceinline__ void sort8(K (&a)[8]) {
    cswap(a[0], a[1]); cswap(a[2], a[3]); cswap(a[4], a[5]); cswap(a[6], a[7]);
    cswap(a[0], a[2]); cswap(a[1], a[3]); cswap(a[4], a[6]); cswap(a[5], a[7]);
    cswap(a[1], a[2]); cswap(a[5], a[6]);
    cswap(a[0], a[4]); cswap(a[1], a[5]); cswap(a[2], a[6]); cswap(a[3], a[7]);
    cswap(a[2], a[4]); cswap(a[3], a[5]);
    cswap(a[1], a[2]); cswap(a[3], a[4]); cswap(a[5], a[6]);
}

// one thread per row.  Rows with <= 8 items (almost every non-dummy row of the configs: mean degree 2-7) are sorted
// by a register sorting network; rows with <= 32 items by an insertion sort in local memory.  Longer rows are appended
// to a work list for the CTA-per-row kernels.
template <bool HAS_PRIMARY>
__global__ void sort_rows_light(const int32_t *__restrict__ row_ptr, int64_t N, int32_t *__restrict__ items,
                                const int32_t *__restrict__ primary, int32_t *__restrict__ worklist,
                                int32_t *__restrict__ work_count, const int32_t *__restrict__ val,
                                int32_t *__restrict__ col) {
    // col (optional): col[p] = val[items[p]] (or items[p]) of the SORTED row, written by whichever kernel sorts the row
    int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= N) return;
    int beg = row_ptr[r], d = row_ptr[r + 1] - beg;
    if (d <= 1) {
        if (d == 1 && col) { const int it = items[beg]; col[beg] = val ? val[it] : it; }
        return;
    }
    if (d > LIGHT_SORT_MAX) {
        worklist[atomicAdd(work_count, 1)] = static_cast<int32_t>(r);
        if (d > HEAVY_SORT_MID) atomicAdd(work_count + 1, 1);
        return;
    }
    if (d <= 8) {
        if constexpr (HAS_PRIMARY) {
            unsigned long long a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = (i < d) ? sort_key(primary, items[beg + i]) : ~0ull;
            sort8(a);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < d) {
                    const int it = static_cast<int32_t>(a[i] & 0xffffffffu);
                    items[beg + i] = it;
                    if (col) col[beg + i] = val ? val[it] : it;
                }
        } else {
            int a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = (i < d) ? items[beg + i] : INT32_MAX;
            sort8(a);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i < d) {
                    items[beg + i] = a[i];
                    if (col) col[beg + i] = val ? val[a[i]] : a[i];
                }
        }
        return;
    }
    unsigned long long a[LIGHT_SORT_MAX];
    for (int i = 0; i < d; ++i) a[i] = sort_key(HAS_PRIMARY ? primary : nullptr, items[beg + i]);
    for (int i = 1; i < d; ++i) {
        unsigned long long k = a[i];
        int j = i - 1;
        while (j >= 0 && a[j] > k) { a[j + 1] = a[j]; --j; }
        a[j + 1] = k;
    }
    for (int i = 0; i < d; ++i) {
        const int it = static_cast<int32_t>(a[i] & 0xffffffffu);
        items[beg + i] = it;
        if (col) col[beg + i] = val ? val[it] : it;
    }
}

// one CTA per listed row with LIGHT_SORT_MAX < d <= HEAVY_SORT_MID items (the dummy rows: one per graph, as long as
// the graph): bitonic sort of the keys (primary[item], item) in shared memory, O(d log^2 d) instead of the O(d^2)
// rank sort that the 2 000-item dummy rows of the largest C2 graphs made the long pole of every CSR build (profiles/r1d:
// 38-62 us per call).
constexpr int BITONIC_THREADS = 512;
template <bool HAS_PRIMARY>
__global__ void __launch_bounds__(BITONIC_THREADS) sort_rows_bitonic(const int32_t *__restrict__ row_ptr,
                                                                     int32_t *__restrict__ items,
                                                                     const int32_t *__restrict__ primary,
                                                                     const int32_t *__restrict__ worklist,
                                                                     const int32_t *__restrict__ work_count,
                                                                     const int32_t *__restrict__ val,
                                                                     int32_t *__restrict__ col) {
    using K = typename std::conditional<HAS_PRIMARY, unsigned long long, unsigned int>::type;
    __shared__ K keys[HEAVY_SORT_MID];
    const int n_work = work_count[0];
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        const int r = worklist[w];
        const int beg = row_ptr[r], d = row_ptr[r + 1] - beg;
        if (d <= LIGHT_SORT_MAX || d > HEAVY_SORT_MID) continue;
        int P = 64;
        while (P < d) P <<= 1;
        for (int i = threadIdx.x; i < P; i += BITONIC_THREADS) {
            K k = static_cast<K>(~static_cast<K>(0));
            if (i < d) {
                const int it = items[beg + i];
                if constexpr (HAS_PRIMARY) k = sort_key(primary, it); else k = static_cast<unsigned int>(it);
            }
            keys[i] = k;
        }
        __syncthreads();
        for (int k = 2; k <= P; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = threadIdx.x; t < (P >> 1); t += BITONIC_THREADS) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));   // index with bit j clear
                    const int x = i | j;
                    const bool asc = (i & k) == 0;
                    const K a = keys[i], b = keys[x];
                    if ((a > b) == asc) { keys[i] = b; keys[x] = a; }
                }
                __syncthreads();
            }
        }
        for (int i = threadIdx.x; i < d; i += BITONIC_THREADS) {
            const int it = static_cast<int32_t>(keys[i] & 0xffffffffu);
            items[beg + i] = it;
            if (col) col[beg + i] = val ? val[it] : it;
        }
        __syncthreads();
    }
}

// one CTA per listed row: rank sort in shared memory on the unique key (primary[item], item).  Keys are kept as two
// int32 arrays and compared four at a time (128-bit shared loads).  Rows longer than `cap` are left to the next
// (larger) instantiation; rows longer than DN4GL_MAX_ROW_DEGREE raise err_flag.
template <bool HAS_PRIMARY>
__global__ void __launch_bounds__(256) sort_rows_heavy(const int32_t *__restrict__ row_ptr,
                                                       int32_t *__restrict__ items,
                                                       const int32_t *__restrict__ primary,
                                                       const int32_t *__restrict__ worklist,
                                                       const int32_t *__restrict__ work_count, int lo, int cap,
                                                       int only_if_flagged, int32_t *err_flag,
                                                       const int32_t *__restrict__ val, int32_t *__restrict__ col) {
    extern __shared__ __align__(16) int32_t skeys[];
    int32_t *ki = skeys, *kp = skeys + cap;
    if (only_if_flagged && work_count[1] == 0) return;   // no row exceeded the mid capacity: nothing to do
    const int n_work = work_count[0];
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        int r = worklist[w];
        int beg = row_ptr[r], d = row_ptr[r + 1] - beg;
        if (d <= lo) continue;
        if (d > cap) {
            if (cap >= DN4GL_MAX_ROW_DEGREE) {
                // above the documented limit: the row is reported through err_flag and left UNSORTED, but `col` still gets
                // valid indices (the scatter's order), so that an aggregation launched before the flag is read gathers
                // real rows in a wrong order instead of reading uninitialised memory
                if (err_flag && threadIdx.x == 0) atomicExch(err_flag, DN4GL_ELIMIT);
                if (col)
                    for (int i = threadIdx.x; i < d; i += blockDim.x) {
                        const int it = items[beg + i];
                        col[beg + i] = val ? val[it] : it;
                    }
            }
            continue;
        }
        const int dpad = (d + 3) & ~3;
        for (int i = threadIdx.x; i < dpad; i += blockDim.x) {
            int it = (i < d) ? items[beg + i] : INT32_MAX;
            ki[i] = it;
            if (HAS_PRIMARY) kp[i] = (i < d) ? primary[it] : INT32_MAX;
        }
        __syncthreads();
        const int4 *ki4 = reinterpret_cast<const int4 *>(ki);
        const int4 *kp4 = reinterpret_cast<const int4 *>(kp);
        for (int i = threadIdx.x; i < d; i += blockDim.x) {
            const int k = ki[i];
            int rank = 0;
            if (HAS_PRIMARY) {
                const int p = kp[i];
                for (int j = 0; j < dpad / 4; ++j) {
                    int4 a = ki4[j], q = kp4[j];
                    rank += (q.x < p || (q.x == p && a.x < k)) + (q.y < p || (q.y == p && a.y < k)) +
                            (q.z < p || (q.z == p && a.z < k)) + (q.w < p || (q.w == p && a.w < k));
                }
            } else {
                for (int j = 0; j < dpad / 4; ++j) {
                    int4 a = ki4[j];
                    rank += (a.x < k) + (a.y < k) + (a.z < k) + (a.w < k);
                }
            }
            items[beg + rank] = k;
            if (col) col[beg + rank] = val ? val[k] : k;
        }
        __syncthreads();
    }
}

// sorts the items of every row by (primary[item], item); shared by the CSR build and coalesce
int dn4gl_sort_rows(const int32_t *row_ptr, int64_t N, int32_t *items, const int32_t *primary,
                    int32_t *worklist, int32_t *work_count, int32_t *err_flag, cudaStream_t st, const int32_t *val,
                    int32_t *col, bool work_count_zeroed) {
    if (N == 0) return DN4GL_OK;
    if (!work_count_zeroed) DN_CUDA(cudaMemsetAsync(work_count, 0, 2 * sizeof(int32_t), st));
    if (primary)
        sort_rows_light<true><<<static_cast<unsigned>(ceil_div64(N, 128)), 128, 0, st>>>(row_ptr, N, items, primary, worklist,
                                                                                          work_count, val, col);
    else
        sort_rows_light<false><<<static_cast<unsigned>(ceil_div64(N, 128)), 128, 0, st>>>(row_ptr, N, items, primary, worklist,
                                                                                           work_count, val, col);
    DN_LAUNCHED();
    const int sms = dn4gl_num_sms();
    // rows above HEAVY_SORT_MID items (up to DN4GL_MAX_ROW_DEGREE keys x 2 int32 arrays = 196608 B of dynamic shared
    // memory) keep the rank sort; that launch returns immediately unless the light pass flagged such a row
    const size_t big = static_cast<size_t>(DN4GL_MAX_ROW_DEGREE) * 2 * sizeof(int32_t);
    static bool attr_set = false;
    if (!attr_set) {
        DN_CUDA(cudaFuncSetAttribute(sort_rows_heavy<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(big)));
        DN_CUDA(cudaFuncSetAttribute(sort_rows_heavy<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(big)));
        attr_set = true;
    }
    if (primary) {
        sort_rows_bitonic<true><<<sms * 2, BITONIC_THREADS, 0, st>>>(row_ptr, items, primary, worklist, work_count, val, col);
        sort_rows_heavy<true><<<sms, 256, big, st>>>(row_ptr, items, primary, worklist, work_count, HEAVY_SORT_MID,
                                                     DN4GL_MAX_ROW_DEGREE, 1, err_flag, val, col);
    } else {
        sort_rows_bitonic<false><<<sms * 4, BITONIC_THREADS, 0, st>>>(row_ptr, items, primary, worklist, work_count, val, col);
        sort_rows_heavy<false><<<sms, 256, big, st>>>(row_ptr, items, primary, worklist, work_count, HEAVY_SORT_MID,
                                                      DN4GL_MAX_ROW_DEGREE, 1, err_flag, val, col);
    }
    DN_LAUNCHED_N(2);
    return DN4GL_OK;
}

extern "C" size_t dn4gl_sort_rows_workspace_bytes(int64_t N) {
    return align_up(static_cast<size_t>(N > 0 ? N : 1) * sizeof(int32_t), 256) + 256;
}

extern "C" int dn4gl_sort_csr_rows(const int32_t *row_ptr, int64_t N, int32_t *items, const int32_t *primary, void *ws,
                                   size_t ws_bytes, int32_t *err_flag, void *stream) {
    DN_ARG(N >= 0 && row_ptr != nullptr && N < INT32_MAX);
    if (N == 0) return DN4GL_OK;
    DN_ARG(items != nullptr);
    WsCarver w(ws, ws_bytes);
    int32_t *worklist = w.take<int32_t>(N);
    int32_t *work_count = w.take<int32_t>(2);
    if (!worklist || !work_count) {
        dn4gl_set_error("dn4gl_sort_csr_rows: workspace too small");
        return DN4GL_EWORKSPACE;
    }
    return dn4gl_sort_rows(row_ptr, N, items, primary, worklist, work_count, err_flag, as_stream(stream), nullptr, nullptr, false);
}

extern "C" size_t dn4gl_csr_workspace_bytes(int64_t N, int64_t E) {
    (void)E;
    size_t n = static_cast<size_t>(N > 0 ? N : 1);
    return align_up((n + 1) * sizeof(int32_t), 256) * 3 + 256 + dn4gl_scan_workspace_bytes(N + 1);
}

extern "C" int dn4gl_build_csr(const int32_t *key, const int32_t *val, int64_t N, int64_t E, int32_t *row_ptr,
                               int32_t *col, int32_t *eid, void *ws, size_t ws_bytes, int32_t *err_flag,
                               void *stream) {
    DN_ARG(N >= 0 && E >= 0 && N < INT32_MAX && E < INT32_MAX);
    DN_ARG(row_ptr != nullptr && (E == 0 || (key != nullptr && eid != nullptr)));
    cudaStream_t st = as_stream(stream);
    WsCarver wsc(ws, ws_bytes);
    // counts | cursor | work_count are adjacent: ONE memset zeroes all three
    int32_t *cnt = wsc.take<int32_t>(N + 1);
    int32_t *cursor = wsc.take<int32_t>(N + 1);
    int32_t *work_count = wsc.take<int32_t>(2);
    int32_t *worklist = wsc.take<int32_t>(N + 1);
    size_t scan_bytes = dn4gl_scan_workspace_bytes(N + 1);
    char *scan_ws = wsc.take<char>(scan_bytes);
    if (!cnt || !cursor || !worklist || !work_count || !scan_ws) {
        dn4gl_set_error("dn4gl_build_csr: workspace too small (%zu < %zu)", ws_bytes, dn4gl_csr_workspace_bytes(N, E));
        return DN4GL_EWORKSPACE;
    }
    const size_t zero_bytes = static_cast<size_t>(reinterpret_cast<char *>(work_count + 2) - reinterpret_cast<char *>(cnt));
    DN_CUDA(cudaMemsetAsync(cnt, 0, zero_bytes, st));
    if (E > 0) {
        csr_histogram<<<static_cast<unsigned>(ceil_div64(E, 256)), 256, 0, st>>>(key, E, cnt);
        DN_LAUNCHED();
    }
    int rc = dn4gl_exclusive_scan_i32(cnt, row_ptr, N, scan_ws, scan_bytes, stream);
    if (rc != DN4GL_OK) return rc;
    if (E == 0) return DN4GL_OK;
    csr_scatter<<<static_cast<unsigned>(ceil_div64(E, 256)), 256, 0, st>>>(key, E, row_ptr, cursor, eid);
    DN_LAUNCHED();
    // the row sorts restore the stable order and write col = val[eid] (or eid) on the way out
    return dn4gl_sort_rows(row_ptr, N, eid, nullptr, worklist, work_count, err_flag, st, val, col, true);
}

// CSR of items whose keys are already non-decreasing (the (src, dst)-sorted edge list that coalesce / PyG hand over):
// no histogram, scan, scatter or sort -- one pass marks the row boundaries.  Thread e writes row_ptr[r] = e for every
// row r in (key[e-1], key[e]]; thread E closes the rows after the last key.
__global__ void csr_from_sorted(const int32_t *__restrict__ key, const int32_t *__restrict__ val, int64_t N, int64_t E,
                                int32_t *__restrict__ row_ptr, int32_t *__restrict__ col, int32_t *__restrict__ eid,
                                int32_t *__restrict__ err_flag) {
    const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e > E) return;
    const int64_t k = (e < E) ? key[e] : N;
    const int64_t kp = (e > 0) ? key[e - 1] : -1;
    if (e < E) {
        if (col) col[e] = val ? val[e] : static_cast<int32_t>(e);
        if (eid) eid[e] = static_cast<int32_t>(e);
    }
    if (k < kp || k < 0 || k > N || (e < E && k >= N)) {   // not sorted / out of range: reported, nothing written
        if (err_flag) atomicExch(err_flag, DN4GL_EINVAL);
        return;
    }
    for (int64_t r = kp + 1; r <= k; ++r) row_ptr[r] = static_cast<int32_t>(e);
}

extern "C" int dn4gl_build_csr_sorted(const int32_t *key, const int32_t *val, int64_t N, int64_t E, int32_t *row_ptr,
                                      int32_t *col, int32_t *eid, int32_t *err_flag, void *stream) {
    DN_ARG(N >= 0 && E >= 0 && N < INT32_MAX && E < INT32_MAX);
    DN_ARG(row_ptr != nullptr && (E == 0 || key != nullptr));
    csr_from_sorted<<<static_cast<unsigned>(ceil_div64(E + 1, 256)), 256, 0, as_stream(stream)>>>(key, val, N, E, row_ptr, col,
                                                                                                 eid, err_flag);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// -------------------------------------------------------------------------------------------
__global__ void collect_heavy(const int32_t *__restrict__ row_ptr, int64_t N, int thr, int32_t *__restrict__ rows,
                              int cap, int32_t *__restrict__ count) {
    // CTA-wide compaction per 1024-row chunk, one atomic per chunk
    __shared__ int sm[33];
    __shared__ int base_sh;
    for (int64_t start = static_cast<int64_t>(blockIdx.x) * blockDim.x; start < N;
         start += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        int64_t r = start + threadIdx.x;
        int flag = (r < N) && (row_ptr[r + 1] - row_ptr[r] > thr);
        int total;
        int ex = block_exclusive_scan(flag, &total, sm);
        if (threadIdx.x == 0) base_sh = total ? atomicAdd(count, total) : 0;
        __syncthreads();
        if (flag && base_sh + ex < cap) rows[base_sh + ex] = static_cast<int32_t>(r);
        __syncthreads();
    }
}

extern "C" int dn4gl_collect_heavy_rows(const int32_t *row_ptr, int64_t N, int32_t threshold, int32_t *heavy_rows,
                                        int32_t cap, int32_t *heavy_count, void *stream) {
    DN_ARG(row_ptr && heavy_rows && heavy_count && cap >= 0 && N >= 0);
    cudaStream_t st = as_stream(stream);
    DN_CUDA(cudaMemsetAsync(heavy_count, 0, sizeof(int32_t), st));
    if (N == 0) return DN4GL_OK;
    // list order is arbitrary (CTAs append chunks as they finish); consumers reduce every listed row
    // independently, so results do not depend on it.  cap must be >= E / threshold + 1.
    unsigned grid = static_cast<unsigned>(ceil_div64(N, 1024));
    if (grid > 4096u) grid = 4096u;
    collect_heavy<<<grid, 1024, 0, st>>>(row_ptr, N, threshold, heavy_rows, cap, heavy_count);
    DN_LAUNCHED();
    return DN4GL_OK;
}

// -------------------------------------------------------------------------------------------
__global__ void gather_rows_kernel(const int32_t *__restrict__ idx, const float4 *__restrict__ x,
                                   float4 *__restrict__ out, int64_t total, int Dv) {
    int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int64_t r = i / Dv;
    int c = static_cast<int>(i - r * Dv);
    out[i] = ldg4(x + static_cast<int64_t>(idx[r]) * Dv + c);
}

extern "C" int dn4gl_gather_rows_f32(const int32_t *idx, const float *x, float *out, int64_t n, int32_t D,
                                     void *stream) {
    DN_ARG(n >= 0 && D > 0 && D % 4 == 0);
    if (n == 0) return DN4GL_OK;
    DN_ARG(idx && x && out && aligned16(x) && aligned16(out));
    int Dv = D / 4;
    int64_t total = n * Dv;
    gather_rows_kernel<<<static_cast<unsigned>(ceil_div64(total, 256)), 256, 0, as_stream(stream)>>>(
        idx, reinterpret_cast<const float4 *>(x), reinterpret_cast<float4 *>(out), total, Dv);
    DN_LAUNCHED();
    return DN4GL_OK;
}
