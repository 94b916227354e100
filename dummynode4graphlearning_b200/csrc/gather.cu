// Segmented gather: assembles a mini-batch from a data set that stays resident in HBM (datasets.py).  For one level of a
// data set (nodes, edges, graphs, subisomorphism values) every selected segment's items are copied, column by column,
// to the batch's offsets; int32 columns that hold node ids are rebased from data-set to batch numbering on the way.
//
// Bound: a C2-sized batch moves ~2.3 MB over three launches; at that size the copy is latency-bound, not bandwidth-bound.
// Each warp owns a contiguous range of output items, finds the segment of its first item by binary search in ptr_out and
// walks forward segment by segment; the lanes copy each segment's words of every column in order (coalesced 4-byte
// words, no shared memory, no atomics: the output is a plain function of the inputs).
#include "common.cuh"

constexpr int GATHER_MAX_COLS = 8;
constexpr int GATHER_WARPS = 8;           // warps per CTA
constexpr int GATHER_CTAS_PER_SM = 2;

struct GatherCols {
    const uint32_t *in[GATHER_MAX_COLS];
    uint32_t *out[GATHER_MAX_COLS];
    int32_t words[GATHER_MAX_COLS];
    int32_t rebase[GATHER_MAX_COLS];
};

__global__ void __launch_bounds__(GATHER_WARPS * 32) gather_segments_kernel(
    int K, const int32_t *__restrict__ idx, const int32_t *__restrict__ ptr_in, int64_t n_seg_in,
    const int32_t *__restrict__ ptr_out, const int32_t *__restrict__ rebase_in, const int32_t *__restrict__ rebase_out,
    int ncols, GatherCols c) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = static_cast<int64_t>(gridDim.x) * GATHER_WARPS;
    const int64_t w = static_cast<int64_t>(blockIdx.x) * GATHER_WARPS + (threadIdx.x >> 5);
    const int64_t total = __ldg(ptr_out + K);
    const int64_t per = (total + warps - 1) / warps;
    const int64_t i1 = min(total, (w + 1) * per);
    int64_t j = w * per;
    if (j >= i1) return;
    int k = segment_of(ptr_out, K, j);
    while (j < i1) {
        const int64_t hi = __ldg(ptr_out + k + 1);
        if (hi > j) {
            const int64_t end = min(hi, i1);
            const int g = __ldg(idx + k);
            if (g >= 0 && g < n_seg_in) {       // the host validates idx; an index outside the data set is never read
                const int64_t src0 = static_cast<int64_t>(__ldg(ptr_in + g)) + (j - __ldg(ptr_out + k));
                const int64_t n = end - j;
                const uint32_t delta = rebase_out ? static_cast<uint32_t>(__ldg(rebase_out + k) - __ldg(rebase_in + g)) : 0u;
                for (int q = 0; q < ncols; ++q) {
                    const int64_t wd = c.words[q];
                    const uint32_t add = c.rebase[q] ? delta : 0u;
                    const uint32_t *__restrict__ s = c.in[q] + src0 * wd;
                    uint32_t *__restrict__ d = c.out[q] + j * wd;
                    for (int64_t t = lane; t < n * wd; t += 32) d[t] = __ldg(s + t) + add;
                }
            }
            j = end;
        }
        ++k;
    }
}

extern "C" int dn4gl_gather_segments(int32_t K, const int32_t *idx, const int32_t *ptr_in, int64_t n_seg_in,
                                     const int32_t *ptr_out, const int32_t *rebase_in, const int32_t *rebase_out,
                                     int32_t ncols, const void *const *col_in, void *const *col_out,
                                     const int32_t *col_words, const int32_t *col_rebase, void *stream) {
    DN_ARG(K >= 0 && n_seg_in >= 0);
    if (K == 0) return DN4GL_OK;
    DN_ARG(ncols >= 1 && ncols <= GATHER_MAX_COLS && "at most 8 columns per level");
    DN_ARG(idx && ptr_in && ptr_out && col_in && col_out && col_words && col_rebase && "null index, offset or column array");
    GatherCols c = {};
    bool any_rebase = false;
    for (int q = 0; q < ncols; ++q) {
        DN_ARG(col_in[q] && col_out[q] && "null column pointer");
        DN_ARG(col_words[q] >= 1 && "a column has at least one 4-byte word per item");
        c.in[q] = static_cast<const uint32_t *>(col_in[q]);
        c.out[q] = static_cast<uint32_t *>(col_out[q]);
        c.words[q] = col_words[q];
        c.rebase[q] = col_rebase[q] != 0;
        any_rebase |= c.rebase[q] != 0;
    }
    DN_ARG((!any_rebase || (rebase_in && rebase_out)) && "rebased columns need rebase_in and rebase_out");
    gather_segments_kernel<<<GATHER_CTAS_PER_SM * dn4gl_num_sms(), GATHER_WARPS * 32, 0, as_stream(stream)>>>(
        K, idx, ptr_in, n_seg_in, ptr_out, any_rebase ? rebase_in : nullptr, any_rebase ? rebase_out : nullptr, ncols, c);
    DN_LAUNCHED();
    return DN4GL_OK;
}
