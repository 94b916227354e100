/*
 * dn4gl.h -- C ABI of libdn4gl.so: the B200 (sm_100a) message-passing hot path of
 * DummyNode4GraphLearning.
 *
 * The reference has no FFI of its own: its hot path sits behind Python operator boundaries
 * into third-party extensions (SURVEY.md section 8(b)).  Each entry point below names the
 * reference call site / third-party op it replaces.  A reference maintainer binds these with
 * ctypes (see INTEGRATION.md); dummynode4graphlearning_b200/_lib.py is that binding.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the parameter name ends in _h;
 *  - every function only enqueues work on `stream` (a cudaStream_t passed as void*) and
 *    returns immediately; nothing allocates, nothing synchronises, no global mutable state
 *    except the thread-local error string;
 *  - the caller owns all buffers (sizes documented per function; workspace sizes are queried);
 *  - indices are int32 (the reference uses int64; the host converts once per batch and
 *    checks N, E < 2^31), features are fp32 row-major contiguous with D % 4 == 0 and 16-byte
 *    aligned base pointers (128-bit loads);
 *  - return value: 0 on success, negative DN4GL_E* on failure, text via dn4gl_last_error();
 *  - kernels are deterministic (no floating-point atomics): repeated runs are bit-identical.
 */
#ifndef DN4GL_H
#define DN4GL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DN4GL_OK 0
#define DN4GL_EINVAL (-1)   /* bad shape / alignment / null pointer                         */
#define DN4GL_ECUDA (-2)    /* a CUDA runtime call or launch failed                         */
#define DN4GL_ELIMIT (-3)   /* a documented capacity limit was exceeded                     */
#define DN4GL_EWORKSPACE (-4) /* workspace too small                                        */
#define DN4GL_ECAPACITY (-5)  /* caller-sized output buffer too small / size hint mismatch (asynchronous flag) */

#define DN4GL_ABI_VERSION 1

int dn4gl_version(void);
const char *dn4gl_last_error(void);
/* binds the calling thread to `device` (cudaSetDevice); one process per GPU is the intended use */
int dn4gl_set_device(int device);
/* number of CUDA kernels this library has launched in this process so far (monotonic counter) */
int64_t dn4gl_launch_count(void);

/* ---- integer plumbing ------------------------------------------------------------------- */

size_t dn4gl_scan_workspace_bytes(int64_t n);
/* out[i] = sum_{j<i} in[j]; out has n+1 elements (out[n] = total).  in may alias out.        */
int dn4gl_exclusive_scan_i32(const int32_t *in, int32_t *out, int64_t n,
                             void *ws, size_t ws_bytes, void *stream);

/* CSR build: groups the E items by key[e] in [0, N), STABLE in item order (row r lists its
 * items with ascending e), which is the order DGL's gspmm / torch-scatter's CPU path and the
 * reference's `sorted(graph.incident(v, "in"))` (tu_data_processing.py:266,
 * utils/graph.py:123,219) iterate in.  row_ptr[N+1], col[E] = val[e] (or e if val NULL), eid[E].
 * Limit: a single row may hold at most DN4GL_MAX_ROW_DEGREE items (DN4GL_ELIMIT is reported
 * asynchronously through err_flag if exceeded; pass NULL to skip).                           */
#define DN4GL_MAX_ROW_DEGREE 24576
size_t dn4gl_csr_workspace_bytes(int64_t N, int64_t E);
int dn4gl_build_csr(const int32_t *key, const int32_t *val, int64_t N, int64_t E,
                    int32_t *row_ptr, int32_t *col, int32_t *eid,
                    void *ws, size_t ws_bytes, int32_t *err_flag, void *stream);
/* Same result as dn4gl_build_csr for keys that are already NON-DECREASING (the (row, col)-sorted edge_index that PyG's
 * coalesce -- and dn4gl_coalesce -- produce: graph_neural_networks/dataset.py:151): one boundary-marking pass, no
 * workspace.  A key out of order or outside [0, N) raises DN4GL_EINVAL asynchronously through err_flag (may be NULL). */
int dn4gl_build_csr_sorted(const int32_t *key, const int32_t *val, int64_t N, int64_t E, int32_t *row_ptr,
                           int32_t *col, int32_t *eid, int32_t *err_flag, void *stream);

/* Sorts the items of every CSR row in place by (primary[item], item) (primary NULL: by item).  With primary = dst on the
 * by-source CSR this is DGL's all_edges(order="srcdst") order (dataset.py:1508), also the order dn4gl_coalesce works in.
 * ws: dn4gl_sort_rows_workspace_bytes(N).  Rows above DN4GL_MAX_ROW_DEGREE items raise DN4GL_ELIMIT through err_flag. */
size_t dn4gl_sort_rows_workspace_bytes(int64_t N);
int dn4gl_sort_csr_rows(const int32_t *row_ptr, int64_t N, int32_t *items, const int32_t *primary, void *ws,
                        size_t ws_bytes, int32_t *err_flag, void *stream);


/* list of rows with degree > threshold (for the heavy-row path of the aggregation kernels):
 * heavy_rows[cap], heavy_count[1]; cap >= E / threshold + 1; list order is unspecified.         */
int dn4gl_collect_heavy_rows(const int32_t *row_ptr, int64_t N, int32_t threshold,
                             int32_t *heavy_rows, int32_t cap, int32_t *heavy_count, void *stream);

/* ---- a1 / a4: dummy-node augmentation ---------------------------------------------------- */

/* classification flavour, replaces load_graph_data_from_TUDatadir(with_dummy=True)'s graph
 * construction (graph_classification/data_processing/tu_data_processing.py:186-214):
 * per graph +1 node (LABEL 0, IS_DUMMY 1) and 2n dummy edges INTERLEAVED (n,v),(v,n) after the
 * m real edges.  Inputs: B graphs, node_ptr[B+1], edge_ptr[B+1], global src/dst[E], vlabel[N],
 * elabel[E].  Outputs sized N+B nodes / E+2N edges (+ ptr arrays of B+1).                     */
int dn4gl_tu_add_dummy(int32_t B, const int32_t *node_ptr, const int32_t *edge_ptr,
                       const int32_t *src, const int32_t *dst,
                       const int32_t *vlabel, const int32_t *elabel, int64_t N, int64_t E,
                       int32_t *o_node_ptr, int32_t *o_edge_ptr, int32_t *o_src, int32_t *o_dst,
                       int32_t *o_vlabel, int32_t *o_vdummy, int32_t *o_elabel, int32_t *o_edummy,
                       void *stream);

/* subgraph-isomorphism flavour, replaces add_dummy_nodes_edges, GraphAdj branch
 * (subgraph_isomorphism/train.py:404-474; Graph.add_nodes/add_edges dataset.py:1238-1293):
 * +1 node {id:max_nv, label:max_nvl, is_dummy:1}; 2n edges BLOCKED [u->d]*n then [d->u]*n with
 * id max_ne / max_ne+1, label max_nel / max_nel+1, is_dummy 1, is_reversed 0..0 1..1.
 * e_isrev may be NULL.                                                                       */
int dn4gl_sub_add_dummy(int32_t B, const int32_t *node_ptr, const int32_t *edge_ptr,
                        const int32_t *src, const int32_t *dst,
                        const int32_t *vid, const int32_t *vlabel,
                        const int32_t *eid, const int32_t *elabel, const int32_t *e_isrev,
                        int64_t N, int64_t E,
                        int32_t max_nv, int32_t max_nvl, int32_t max_ne, int32_t max_nel,
                        int32_t *o_node_ptr, int32_t *o_edge_ptr, int32_t *o_src, int32_t *o_dst,
                        int32_t *o_vid, int32_t *o_vlabel, int32_t *o_vdummy,
                        int32_t *o_eid, int32_t *o_elabel, int32_t *o_edummy, int32_t *o_erev,
                        void *stream);

/* ---- a2 / a5: edge-to-vertex ("conjugate") transform -------------------------------------- */

/* classification flavour, replaces convert_conjugate_graph_forward
 * (tu_data_processing.py:223-338) for graphs whose edge IDs are their positions (what
 * load_graph_data_from_TUDatadir produces).  Two phases so the caller can allocate:
 *   _count: needs in_ptr/in_eid = dn4gl_build_csr(key=dst) and out-CSR row_ptr by src
 *           (out_ptr); writes per-edge survivor counts' scan cand_off[E+1], per-graph vertex
 *           and edge offsets o_node_ptr[B+1], o_edge_ptr[B+1], vertex renumbering newid[E].
 *   _fill:  writes o_src/o_dst (global conjugate vertex ids), o_v_origin[V'] (original edge
 *           of each conjugate vertex) and o_e_shared[E'] (shared original vertex of each
 *           conjugate edge) in exactly the reference's order.
 * e_isdummy may be NULL (LINE_ graphs).  ws from dn4gl_conj_workspace_bytes.
 * cap_v / cap_e: rows the caller allocated for o_v_origin / o_src, o_dst, o_e_shared (normally the totals _count wrote;
 * a caller that sized them from a host-side hint passes the hint): nothing is written beyond them, an overflow raises
 * DN4GL_ECAPACITY through err_flag (may be NULL).                                                                  */
size_t dn4gl_conj_workspace_bytes(int32_t B, int64_t N, int64_t E);
int dn4gl_tu_conjugate_count(int32_t B, const int32_t *node_ptr, const int32_t *edge_ptr,
                             const int32_t *src, const int32_t *dst, const int32_t *e_isdummy,
                             int64_t N, int64_t E,
                             const int32_t *in_ptr, const int32_t *in_eid,
                             int32_t *cand_off, int32_t *newid,
                             int32_t *o_node_ptr, int32_t *o_edge_ptr,
                             void *ws, size_t ws_bytes, void *stream);
int dn4gl_tu_conjugate_fill(int32_t B, const int32_t *node_ptr, const int32_t *edge_ptr,
                            const int32_t *src, const int32_t *dst, const int32_t *e_isdummy,
                            int64_t N, int64_t E,
                            const int32_t *in_ptr, const int32_t *in_eid,
                            const int32_t *cand_off, const int32_t *newid,
                            const int32_t *o_node_ptr, const int32_t *o_edge_ptr,
                            int32_t *o_src, int32_t *o_dst, int32_t *o_v_origin, int32_t *o_e_shared,
                            int64_t cap_v, int64_t cap_e, int32_t *err_flag,
                            void *ws, size_t ws_bytes, void *stream);

/* CONJ_ structure in closed form (round 2): the CSR pair of load_graph_data_from_TUDatadir(with_dummy=True) ->
 * convert_conjugate_graph_forward (tu_data_processing.py:125-338) -> PyG read_tu_data's remove_self_loops + coalesce
 * (graph_neural_networks/dataset.py:151), written row by row from the RAW graphs' CSRs without building the
 * dummy-augmented graph, the candidate list, or sorting anything: every node has exactly one dummy out- and in-edge and
 * all dummy edges merge into one conjugate vertex D, so  out(e) = {real out-edges of dst(e)} \ {e} + {D},
 * in(e) = {real in-edges of src(e)} \ {e} + {D},  out(D) = in(D) = all real edges.  Requires every graph to have >= 1 node.
 *   out_ptr / out_eid, in_ptr / in_eid: the raw graphs' CSR by source / by destination (dn4gl_build_csr[_sorted], items in
 *   ascending edge id).   _lens: row lengths len_out / len_in [E + B] (scan them into rp_out / rp_in [E + B + 1]) and
 *   o_node_ptr[B + 1] (= edge_ptr[g] + g).   _fill: col_out / col_in (global conjugate vertex ids, rows ascending) and
 *   o_vlabel[E + B] (label of the original edge, 1 if elabel == NULL; D: 0); edge2graph[E] = graph of every raw edge
 *   (dn4gl_segment_ids_i32 over edge_ptr).                                                                            */
int dn4gl_tu_conj_direct_lens(int32_t B, const int32_t *edge_ptr, const int32_t *src, const int32_t *dst,
                              const int32_t *out_ptr, const int32_t *in_ptr, int64_t E, int32_t *len_out,
                              int32_t *len_in, int32_t *o_node_ptr, void *stream);
int dn4gl_tu_conj_direct_fill(int32_t B, const int32_t *edge_ptr, const int32_t *edge2graph, const int32_t *src,
                              const int32_t *dst, const int32_t *elabel, const int32_t *out_ptr, const int32_t *out_eid,
                              const int32_t *in_ptr, const int32_t *in_eid, int64_t E, const int32_t *rp_out,
                              const int32_t *rp_in, int32_t *col_out, int32_t *col_in, int32_t *o_vlabel,
                              void *stream);

/* subgraph-isomorphism flavour, replaces convert_conjugate_graph, DGL branch (subgraph_isomorphism/utils/graph.py:
 * 77-175; igraph branch :177-267 is the same rule), called per graph by convert_to_conjugate (train.py:564-593).
 * Edges with equal eid merge into one conjugate vertex (numbered by ascending id, attributes of the first such edge);
 * candidate conjugate edges (e' -> e), e in edge order, e' ascending over the in-edges of src(e), are kept on the FIRST
 * occurrence of the key (eid[e'], vlabel[src e], eid[e]).  Three phases (two data-dependent sizes):
 *   _count: in_ptr = row_ptr of dn4gl_build_csr(key=dst).  id_bound > every eid.  Writes ev[E] (conjugate vertex of
 *           every edge, global numbering), cand_off[E+1], o_node_ptr[B+1].  Host then reads V' = o_node_ptr[B] and
 *           ncand = cand_off[E].  ws from dn4gl_sub_conj_workspace_bytes and must be kept untouched until _fill.
 *   _mark : table = table_slots 64-bit words (power of two >= 2 * ncand), keep_scan[ncand+1]; ws here is a SEPARATE
 *           scan workspace of dn4gl_scan_workspace_bytes(ncand + 1).  Writes o_edge_ptr[B+1]; E' = o_edge_ptr[B].
 *   _fill : o_src/o_dst[E'] (global conjugate vertex ids), o_v_origin[V'] (original edge of each conjugate vertex),
 *           o_e_shared[E'] (shared original vertex of each conjugate edge), in exactly the reference's order.
 * err_flag receives DN4GL_ELIMIT if an eid falls outside [0, id_bound).                                          */
size_t dn4gl_sub_conj_workspace_bytes(int32_t B, int64_t E, int32_t id_bound);
int dn4gl_sub_conj_count(int32_t B, const int32_t *edge_ptr, const int32_t *src, const int32_t *eid,
                         int64_t N, int64_t E, int32_t id_bound, const int32_t *in_ptr, int32_t *ev,
                         int32_t *cand_off, int32_t *o_node_ptr, void *ws, size_t ws_bytes,
                         int32_t *err_flag, void *stream);
int dn4gl_sub_conj_mark(int32_t B, const int32_t *edge_ptr, const int32_t *src, const int32_t *vlabel,
                        int64_t E, const int32_t *in_ptr, const int32_t *in_eid, const int32_t *ev,
                        const int32_t *cand_off, int64_t ncand, void *table, int64_t table_slots,
                        int32_t *keep_scan, int32_t *o_edge_ptr, void *ws, size_t ws_bytes, void *stream);
int dn4gl_sub_conj_fill(int32_t B, const int32_t *src, int64_t E, int32_t id_bound, const int32_t *in_ptr,
                        const int32_t *in_eid, const int32_t *ev, const int32_t *cand_off,
                        const int32_t *keep_scan, int32_t *o_src, int32_t *o_dst, int32_t *o_v_origin,
                        int32_t *o_e_shared, void *ws, size_t ws_bytes, void *stream);

/* ---- SURVEY.md 8(f) rank 3: remaining augmentation flags of subgraph_isomorphism/train.py --------------------- */
/* add_reversed_edges, GraphAdj branch (train.py:291-345): graph g's m edges are followed by their m reversals (v, u)
 * with id = max_ne + position-in-graph, label + max_nel, is_reversed = 1 (originals: 0).  Outputs hold 2E edges;
 * o_edge_ptr = 2 * edge_ptr.  Node arrays are unchanged.                                                            */
int dn4gl_sub_add_reversed(int32_t B, const int32_t *edge_ptr, const int32_t *src, const int32_t *dst,
                           const int32_t *eid, const int32_t *elabel, int64_t E, int32_t max_ne, int32_t max_nel,
                           int32_t *o_edge_ptr, int32_t *o_src, int32_t *o_dst, int32_t *o_eid,
                           int32_t *o_elabel, int32_t *o_e_is_reversed, void *stream);
/* remove_loops, GraphAdj branch (train.py:270-288): keep_scan[E+1] = exclusive scan of (src != dst); survivors[<=E] =
 * surviving edge indices in order (gather every edge column through it); o_edge_ptr[B+1]; E' = keep_scan[E].
 * ws: dn4gl_scan_workspace_bytes(E + 1).                                                                           */
int dn4gl_remove_loops_mark(int32_t B, const int32_t *edge_ptr, const int32_t *src, const int32_t *dst,
                            int64_t E, int32_t *keep_scan, int32_t *o_edge_ptr, int32_t *survivors, void *ws,
                            size_t ws_bytes, void *stream);
/* compute_largest_eigenvalues (utils/graph.py:41-71) per graph of the batch: node_eig[g] = max_e (out_deg[u] + in_deg[v]),
 * edge_eig[g] = max_e (in_deg[u] + out_deg[v]) over the graph's edges (0 for a graph without edges).                 */
int dn4gl_sub_eigen_bounds(int32_t B, const int32_t *edge_ptr, const int32_t *src, const int32_t *dst,
                           const int32_t *in_deg, const int32_t *out_deg, int32_t *node_eig, int32_t *edge_eig,
                           void *stream);

/* ---- SURVEY.md 8(f) rank 2: match-weight targets from ground-truth subisomorphisms ------------------------------ */
/* Batched compute_nodeseq_subisoweights (subgraph_isomorphism/dataset.py:54-61, called at :1491-1500): sample b owns
 * S_b subisomorphisms, each a row of np_b graph-LOCAL node ids, concatenated in values[total] with val_ptr[B+1] giving
 * each sample's first element.  weights[Ng] (zeroed here) += 1 per occurrence of a graph node.                         */
int dn4gl_subiso_node_weights(int32_t B, const int32_t *val_ptr, const int32_t *values, int64_t total,
                              const int32_t *g_node_ptr, int64_t Ng, int32_t *weights, void *stream);
/* Batched compute_edgeseq_subisoweights (dataset.py:64-108, called at :1502-1520): for every subisomorphism and every
 * pattern edge (u, v, l) whose run of consecutive equal (u, v) is the last one with that key (the reference's dict
 * semantics), every graph edge (map[u], map[v]) with label l gets +1.  work_ptr[B+1] = prefix sums of S_b * m_b
 * (m_b = pattern edges of sample b), total_work = work_ptr[B].  The graph side is given as its CSR by source whose
 * rows are sorted by (dst, edge id) (dn4gl_build_csr(key = src) then dn4gl_sort_csr_rows(primary = dst), i.e.
 * all_edges(order="srcdst")) plus dst / label in edge-id order.  active_ws: Ep int32 of scratch.  weights[Eg] zeroed here. */
int dn4gl_subiso_edge_weights(int32_t B, const int32_t *work_ptr, int64_t total_work, const int32_t *val_ptr,
                              const int32_t *values, const int32_t *p_node_ptr, const int32_t *p_edge_ptr,
                              const int32_t *p_src, const int32_t *p_dst, const int32_t *p_elabel, int64_t Ep,
                              int32_t *active_ws, const int32_t *g_node_ptr, const int32_t *g_out_ptr,
                              const int32_t *g_out_items, const int32_t *g_dst, const int32_t *g_elabel,
                              int64_t Eg, int32_t *weights, void *stream);

/* Batched get_conjugate_subisomorphisms (utils/graph.py:294-330) + the g_eid gather of convert_to_conjugate
 * (train.py:546-556, 577-587): conj[work_ptr[b] + s * m_b + q] = graph-local id of the edge that pattern edge slot q of
 * subisomorphism s maps to (slot q = q-th distinct (u, v) pair of the pattern in order of first appearance, label set =
 * last run with that pair; the last matching edge in (src, dst, id) order wins; unmatched slots and slots beyond the
 * number of distinct pairs give the first edge of that order, as the reference's zero-initialised matrix does).
 * Arguments as for dn4gl_subiso_edge_weights, plus g_edge_ptr[B+1]; needs at least one edge per graph with matches.     */
int dn4gl_subiso_conjugate(int32_t B, const int32_t *work_ptr, int64_t total_work, const int32_t *val_ptr,
                           const int32_t *values, const int32_t *p_node_ptr, const int32_t *p_edge_ptr,
                           const int32_t *p_src, const int32_t *p_dst, const int32_t *p_elabel, int64_t Ep,
                           int32_t *active_ws, const int32_t *g_node_ptr, const int32_t *g_edge_ptr,
                           const int32_t *g_out_ptr, const int32_t *g_out_items, const int32_t *g_dst,
                           const int32_t *g_elabel, int32_t *conj, void *stream);

/* The dummy column of add_dummy_nodes_edges (train.py:467-472), batched: row s of sample b (rows[b] rows of
 * np_b = (val_ptr[b+1] - val_ptr[b]) / rows[b] ids) is written at out[out_ptr[b] + s * (np_b + 1)] as its np_b ids
 * followed by n_b = g_node_ptr[b+1] - g_node_ptr[b], the graph's node count BEFORE augmentation (the graph-local id of
 * the dummy node dn4gl_sub_add_dummy appends last).  Samples with rows[b] = 0 write nothing.  out_ptr[B+1]: the output
 * offsets val_ptr[b] + sum_{b' < b} rows[b'] (from the caller's host size tables); out_total = out_ptr[B].          */
int dn4gl_subiso_append_dummy(int32_t B, const int32_t *val_ptr, const int32_t *values, const int32_t *rows,
                              const int32_t *g_node_ptr, const int32_t *out_ptr, int64_t out_total, int32_t *out,
                              void *stream);

/* The match terms of the counting models' bp_loss (train.py:776-813), node and edge kind in one launch each way
 * (csrc/match.cu).  Per kind: pred[B*L] fp32 left-padded, mask[B*L] (bool bytes, 1 = real), w[N] int32 flat weights of
 * the augmented graph batch with row offsets seg_ptr[B+1] (position (b, j) reads w[seg_ptr[b] + j - (L - len_b)] when
 * j >= L - len_b); pred = NULL leaves the kind out.  On masked and padded positions prediction and target count as 0.
 *   out[0] = (match_loss_w * sum crit(leaky(p, neg_slp) - w) + match_reg_w * sum crit(relu(p - pred_c[b]))) / B
 * over both kinds' B*L positions; crit 0 = MAE, 1 = MSE, 2 = SMSE (smooth L1, beta 1).  neg_slp / match_loss_w /
 * match_reg_w: device fp32 scalars.  Sums in double in an order fixed by B and the padded lengths; ws:
 * dn4gl_match_loss_workspace_bytes(B) bytes, 8-byte aligned; counter: one int32 that is 0 on entry (left 0).
 * The backward writes g_pred_v / g_pred_e (every position, masked and padded ones included) and g_pred_c[B] (the
 * per-graph sum of the regulariser's derivatives) for the upstream gradient g_out[0].                              */
size_t dn4gl_match_loss_workspace_bytes(int32_t B);
int dn4gl_match_loss_f32(int32_t B, const float *pred_c, const float *pred_v, const uint8_t *mask_v, const int32_t *w_v,
                         const int32_t *ptr_v, int32_t Lv, const float *pred_e, const uint8_t *mask_e,
                         const int32_t *w_e, const int32_t *ptr_e, int32_t Le, int32_t crit, const float *neg_slp,
                         const float *match_loss_w, const float *match_reg_w, float *out, void *ws, size_t ws_bytes,
                         int32_t *counter, void *stream);
int dn4gl_match_loss_bwd_f32(int32_t B, const float *g_out, const float *pred_c, const float *pred_v,
                             const uint8_t *mask_v, const int32_t *w_v, const int32_t *ptr_v, int32_t Lv,
                             const float *pred_e, const uint8_t *mask_e, const int32_t *w_e, const int32_t *ptr_e,
                             int32_t Le, int32_t crit, const float *neg_slp, const float *match_loss_w,
                             const float *match_reg_w, float *g_pred_v, float *g_pred_e, float *g_pred_c,
                             void *stream);

/* ---- a3: PyG read_tu_data canonicalisation ------------------------------------------------- */
/* remove_self_loops + coalesce [torch-geometric 2.0.2 read_tu_data, called from
 * graph_classification/graph_neural_networks/dataset.py:151]: given the edge list's endpoints
 * src[E], dst[E] (edge-id order) and its by-src CSR (row_ptr[N+1], items[E] = edge ids, from
 * dn4gl_build_csr(key=src)), sorts every row in place by (dst, edge id), drops self loops, merges
 * repeated (src,dst) pairs.  keep_scan[E+1] = exclusive scan of survivor flags in sorted order;
 * survivors are written compacted in (src,dst) order: o_src/o_dst/o_first[<=E] (o_first = first
 * original edge of each merged group).  E' = keep_scan[E].                                    */
size_t dn4gl_coalesce_workspace_bytes(int64_t N, int64_t E);
int dn4gl_coalesce(const int32_t *src, const int32_t *dst, int64_t N, int64_t E, const int32_t *row_ptr, int32_t *items,
                   int32_t *keep_scan, int32_t *o_src, int32_t *o_dst, int32_t *o_first,
                   void *ws, size_t ws_bytes, int32_t *err_flag, void *stream);

/* a[i] = b[i] = fill for i in [count[0], cap): pads a compacted list whose length only the device knows (dn4gl_coalesce's
 * keep_scan[E]) up to its host-known capacity with the index of a trash row, so that the CSR builds behind it need no
 * device->host read of the count.  b may be NULL.                                                                    */
int dn4gl_pad_tail_i32(const int32_t *count, int64_t cap, int32_t *a, int32_t *b, int32_t fill, void *stream);

/* ---- K1: sum aggregation -------------------------------------------------------------------- */
/* out[v,:] = self_scale * x[v,:] + sum_{p in [row_ptr[v], row_ptr[v+1])} x[col[p],:]
 * replaces torch_scatter.scatter(reduce='sum') under PyG GINConv.propagate (gconv.py:212) and
 * DGL update_all(copy, fn.sum) -> gspmm (rgin.py:159).  With the transposed CSR it is its own
 * backward.  x has n_src rows, out has N rows (x may be a different table than out: RGIN gathers
 * from the (N*R, D) per-relation table).  Rows listed in heavy_rows (degree > heavy threshold,
 * e.g. dummy nodes) are reduced by a whole CTA; pass heavy_rows = NULL to let the per-row path
 * handle everything.  self_scale != 0 requires n_src == N.  eps_dev (may be NULL): a device scalar;
 * when given, self_scale = 1 + *eps_dev is read by the kernel (GINConv(train_eps=True): eps is a
 * Parameter on the device, gconv.py:197, and reading it on the host would synchronise).        */
int dn4gl_spmm_sum_f32(const int32_t *row_ptr, const int32_t *col, const float *x, float *out,
                       int64_t N, int64_t n_src, int32_t D, float self_scale, const float *eps_dev,
                       const int32_t *heavy_rows, const int32_t *heavy_count, int32_t heavy_threshold,
                       void *stream);

/* K1, tiled variant for block-diagonal batches (n_src == N): a warp-specialised producer/consumer pipeline.  Rows are
 * cut into tiles of whole consecutive graphs (dn4gl_make_row_tiles over the per-graph row offsets seg_ptr[B+1]); a
 * producer lane streams every tile's feature rows, row_ptr slice and col slice into a ring of `stages` shared-memory
 * buffers with bulk asynchronous copies (cp.async.bulk + mbarrier), consumer warps resolve the neighbour indices
 * there and stream the output rows.  Same result contract as dn4gl_spmm_sum_f32 and correct for ANY CSR (indices
 * outside a staged window fall back to global loads); the tiling is a performance contract only.
 *
 * dn4gl_make_row_tiles: tile_desc[4*num_tiles] int32 = {r0, r1, e0, e1 | cut<<31} per tile, num_tiles >=
 *   ceil(N / window_rows); window_rows <= cap_rows - (largest graph) keeps every tile inside one stage (cap_rows / 2
 *   is always safe).  heavy_list[heavy_cap] / heavy_count[1] (optional, both or neither): rows with more than 64
 *   neighbours inside tiles that had to cut a graph longer than the window; the kernel reduces them CTA-wide.
 *   heavy_cap >= E / 64 + 1.  The tiling must be rebuilt when row_ptr / col change.  col may be NULL: the caller vouches
 *   that every column of a graph's rows lies inside that graph (block-diagonal by construction, e.g. the output of
 *   dn4gl_tu_conj_direct_fill) and the per-tile verification pass is skipped.
 * dn4gl_spmm_tiled_f32: smem_bytes = dynamic shared memory per CTA (16 KiB .. 220 KiB; <= 110 KiB lets two CTAs share
 *   an SM for D <= 128), stages in 1..4, nnz_per_row = col slots staged per row (about ceil(E/N) + 1), warps = 16, 24
 *   or 32 per CTA (one producer + 15 / 23 / 31 consumers; more than 16 only applies to D <= 128).  Tiles whose columns were verified to
 *   stay inside the tile (done by dn4gl_make_row_tiles) run an unchecked shared-memory-only loop.
 * row_ptr and col must be 16-byte aligned and their allocations padded to a multiple of 16 bytes (bulk copies move
 * whole 16-byte words; true for any cudaMalloc / torch allocation).                                                 */
int dn4gl_make_row_tiles(const int32_t *seg_ptr, int32_t B, int32_t window_rows, const int32_t *row_ptr,
                         const int32_t *col, int64_t N, int32_t *tile_desc, int32_t num_tiles, int32_t *heavy_list,
                         int32_t heavy_cap, int32_t *heavy_count, void *stream);
int32_t dn4gl_spmm_tiled_cap_rows(int32_t D, int32_t smem_bytes, int32_t stages, int32_t nnz_per_row);
int dn4gl_spmm_tiled_f32(const int32_t *row_ptr, const int32_t *col, const float *x, float *out, int64_t N,
                         int32_t D, float self_scale, const float *eps_dev, const int32_t *tile_desc, int32_t num_tiles,
                         const int32_t *heavy_list, const int32_t *heavy_count, int32_t heavy_cap,
                         int32_t smem_bytes, int32_t stages, int32_t nnz_per_row, int32_t warps, void *stream);

/* ---- K3: segment readout ------------------------------------------------------------------- */
/* out[b,:] = scale_b * sum_{v in [seg_ptr[b], seg_ptr[b+1]), mask[v]==0} x[v,:]
 * mode 0: sum (global_add_pool, gconv.py:176; SumPredictNet.agg_graph pred.py:215),
 * mode 1: mean over the segment length (global_mean_pool).  mask (uint8, 1 = skip row, e.g.
 * dummy nodes, basemodel.py:905-912) may be NULL.                                              */
int dn4gl_segment_sum_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *x, float *out,
                          int32_t B, int32_t D, int32_t mode, void *stream);
/* backward of the above: gx[v,:] = mask[v] ? 0 : scale_b * g[b(v),:]                            */
int dn4gl_segment_bcast_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *g, float *gx,
                            int32_t B, int64_t N, int32_t D, int32_t mode, void *stream);

/* loss[0] = -(1/B) sum_b logp[b, y[b]]: F.nll_loss(log_probs, y) with mean reduction, the classification criterion of
 * graph_neural_networks/main.py:41 (y: int64 class indices as torch carries them; no class weights, no ignore_index --
 * the reference uses neither).  One CTA, fixed reduction tree.  _bwd: g_logp[b, c] = (c == y[b]) ? -g[0] / B : 0.        */
int dn4gl_nll_mean_f32(const float *logp, const int64_t *y, int32_t B, int32_t C, float *loss, void *stream);
int dn4gl_nll_mean_bwd_f32(const float *g, const int64_t *y, int32_t B, int32_t C, float *g_logp, void *stream);

/* Jumping-knowledge class head of the GIN classifier, graph_neural_networks/models/gconv.py:205-214 (out += dropout(
 * Linear_l(pool(h_l))), then log_softmax; dropout p = 0):
 *   logp = log_softmax_c( sum_l pooled_l W_l^T + n_b bias_0 + sum_{l>=1} bias_l )
 * pooled / W / bias / g_pooled / dW / db are HOST arrays of L device pointers (pooled_l: B x D, W_l: C x D row-major,
 * bias_l: C).  seg_ptr (B + 1, the graphs' row ranges) selects the reference's sum-pooling form, where layer 0 pools
 * Linear_0(h) and its bias is therefore counted n_b = rows-of-graph-b times (gconv.py:210); NULL counts it once (mean
 * pooling).  L <= 16, C <= 32; _bwd additionally needs ((C + 8) L D + 10 C + 8) * 4 <= 48 KiB of shared memory
 * (DN4GL_EINVAL otherwise: the host composes the head from library GEMMs instead).  _bwd writes every g_pooled_l,
 * dW_l, db_l; partial sums are merged in a fixed order by the last CTA (counter: one zeroed int32, left at zero).        */
size_t dn4gl_jk_head_workspace_bytes(int32_t L, int32_t B, int32_t D, int32_t C);
int dn4gl_jk_head_fwd_f32(const float *const *pooled, const float *const *W, const float *const *bias, int32_t L,
                          int32_t B, int32_t D, int32_t C, const int32_t *seg_ptr, float *logp, void *stream);
int dn4gl_jk_head_bwd_f32(const float *g_logp, const float *logp, const float *const *pooled, const float *const *W,
                          int32_t L, int32_t B, int32_t D, int32_t C, const int32_t *seg_ptr,
                          float *const *g_pooled, float *const *dW, float *const *db, void *ws, size_t ws_bytes,
                          int32_t *counter, void *stream);

/* left-padded dense batchify, replaces split_and_batchify_graph_feats(pre_pad=True)
 * (subgraph_isomorphism/utils/dl.py:51-81): out[b, Lmax-len_b+i, :] = x[seg_ptr[b]+i, :] (0 on
 * pads and on rows with mask[v]=1); inverse gather for the backward.                          */
int dn4gl_pad_segments_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *x, float *out,
                           int32_t B, int32_t Lmax, int32_t D, void *stream);
int dn4gl_unpad_segments_f32(const int32_t *seg_ptr, const uint8_t *mask, const float *g, float *gx,
                             int32_t B, int32_t Lmax, int32_t D, int64_t N, void *stream);

/* label filter gate, replaces ScalarFilter on the padded label matrices
 * (models/filter.py:10-16, basemodel.py:830-847): gate[v] = 1 if label of graph node v occurs
 * among the labels of its pattern, or equals 0 while the pattern is shorter than Lp_max
 * (padding leak, SURVEY.md App. A-14).                                                        */
int dn4gl_label_filter_gate(const int32_t *g_ptr, const int32_t *g_label,
                            const int32_t *p_ptr, const int32_t *p_label,
                            int32_t B, int32_t Lp_max, int64_t Ng, float *gate, void *stream);

/* ---- K4 / K5: DMPNN ------------------------------------------------------------------------ */
/* node aggregation by linearity (dmpnn.py:111-127, reduce fn.sum :92):
 *   S[v, 0:D]  = sum_{e in in(v),  is_rev[e]} ef[e,:]      (multiplies W_out)
 *   S[v, D:2D] = sum_{e in in(v), !is_rev[e]} ef[e,:]      (multiplies -W_in)
 * in_ptr/in_eid: CSR by destination.  S is (N, 2D).                                            */
int dn4gl_dmp_node_agg_f32(const int32_t *in_ptr, const int32_t *in_eid, const uint8_t *is_rev,
                           const float *ef, float *S, int64_t N, int32_t D,
                           const int32_t *heavy_rows, const int32_t *heavy_count, int32_t heavy_threshold,
                           void *stream);
/* backward: gef[e,:] = is_rev[e] ? gS[dst[e], 0:D] : gS[dst[e], D:2D]                           */
int dn4gl_dmp_node_agg_bwd_f32(const int32_t *dst, const uint8_t *is_rev, const float *gS, float *gef,
                               int64_t E, int32_t D, void *stream);
/* edge message + self terms (dmpnn.py:112,120,123,126 and 142-149), PQ = h @ [W_dst | W_src]
 * (N, 2D), T = ef @ [W_eloop | W_src - W_dst] (E, 2D):
 *   msg_e = is_rev ? P[src]-Q[dst] : P[dst]-Q[src]
 *   out[e,:] = T[e,0:D] + 2*(1+log2(1+out_deg[dst[e]])) * T[e,D:2D] + msg_e + bias
 * bias may be NULL.                                                                            */
int dn4gl_dmp_edge_update_f32(const int32_t *src, const int32_t *dst, const uint8_t *is_rev,
                              const int32_t *out_deg, const float *PQ, const float *T,
                              const float *bias, float *out, int64_t E, int32_t D, void *stream);
/* backward wrt T: gT[e,0:D] = g[e,:], gT[e,D:2D] = c_e * g[e,:]                                 */
int dn4gl_dmp_edge_update_bwd_T_f32(const int32_t *dst, const int32_t *out_deg, const float *g,
                                    float *gT, int64_t E, int32_t D, void *stream);
/* backward wrt PQ (deterministic, per node over its in- and out-lists):
 *   gPQ[v,0:D]  =  sum_{e in in(v),!rev} g_e + sum_{e in out(v), rev} g_e
 *   gPQ[v,D:2D] = -sum_{e in in(v), rev} g_e - sum_{e in out(v),!rev} g_e                        */
int dn4gl_dmp_edge_update_bwd_PQ_f32(const int32_t *in_ptr, const int32_t *in_eid,
                                     const int32_t *out_ptr, const int32_t *out_eid,
                                     const uint8_t *is_rev, const float *g, float *gPQ,
                                     int64_t N, int32_t D, void *stream);

/* ---- CompGCN composition (SURVEY.md 8(f) rank 1) ------------------------------------------------------------ */
/* Replaces CompGCNLayer._comp_func + the edge normalisation inside _node_message_func
 * (subgraph_isomorphism/models/compgcn.py:214-240, norms :190-209) for comp_opt "sub" (op 0) and "mult" (op 1):
 *   C[e,:] = a[src e] * (h[src e,:] - ef[e,:])   |   a[src e] * h[src e,:] * ef[e,:]
 * src_scale = a (N floats) or NULL for a = 1.  The reduce fn.sum(msg) (compgcn.py:163) is dn4gl_dmp_node_agg_f32 on C
 * and the in/out weights are applied by one node-level GEMM on [S_rev | S_fwd] (linearity).  src[E]: source of every
 * edge in edge-id order; h (N x D), ef / C (E x D) fp32 row-major, D % 4 == 0.                                          */
int dn4gl_comp_edge_f32(const int32_t *src, const float *src_scale, const float *h, const float *ef, float *C,
                        int64_t E, int32_t D, int32_t op, void *stream);
/* gEF[e,:] = -a[src e] gC[e,:]  |  a[src e] gC[e,:] * h[src e,:]   (h may be NULL for op 0)                             */
int dn4gl_comp_edge_bwd_ef_f32(const int32_t *src, const float *src_scale, const float *h, const float *gC,
                               float *gEF, int64_t E, int32_t D, int32_t op, void *stream);
/* gH[u,:] = a[u] * sum_{e in out(u)} gC[e,:] (* ef[e,:] for op 1), out-list = CSR by source (dn4gl_build_csr(key=src)),
 * items in edge-id order: deterministic, no float atomics.  ef may be NULL for op 0.  D in {4,...,128,256}.              */
int dn4gl_comp_edge_bwd_h_f32(const int32_t *out_ptr, const int32_t *out_eid, const float *src_scale,
                              const float *ef, const float *gC, float *gH, int64_t N, int32_t D, int32_t op,
                              void *stream);

/* ---- dense helpers of the MLPs ----------------------------------------------------------------- */
/* C (Ka x Kb) = A^T B, colsum_A (Ka, may be NULL) = column sums of A; A (N x Ka), B (N x Kb) row-major.
 * The weight gradient of every nn.Linear on the path (dW = G^T X, db = colsum G: gconv.py:190-196 MLPs,
 * rgin.py:52 / dmpnn.py:47,55 MLPs) and of the raw-parameter matmuls (dW = X^T G: rgin.py:141, dmpnn.py:112-146),
 * written as a deterministic row reduction instead of a large-K library GEMM.
 * Limit: ceil(Ka/4) * ceil(Kb/4) <= 256 (e.g. 64 x 64); DN4GL_EINVAL otherwise (callers keep the library GEMM). */
size_t dn4gl_atb_workspace_bytes(int64_t N, int32_t Ka, int32_t Kb);
int dn4gl_atb_f32(const float *A, const float *B, float *C, float *colsum_A, int64_t N, int32_t Ka, int32_t Kb,
                  void *ws, size_t ws_bytes, void *stream);

/* ---- tensor-core stages of the per-node / per-edge MLPs (tcgen05, 3xTF32) --------------------- */
/* Replaces, on the layer's MLP (gconv.py:190-196 `Linear, BatchNorm1d, ReLU, Linear, BatchNorm1d, ReLU`;
 * rgin.py:52, dmpnn.py:47,55 `Linear, act, Linear`), the chain nn.Linear -> F.batch_norm -> activation and its
 * autograd backward (cuBLAS SGEMMs + ATen batch-norm / elementwise kernels in the reference's stack).
 *
 * A BatchNorm "record" over C channels is 4*C floats: mean[C], rstd[C], k[C] = gamma*rstd, beta[C]; applying it is
 * (x - mean) * k + beta.  Activations: */
#define DN4GL_ACT_NONE 0
#define DN4GL_ACT_RELU 1
#define DN4GL_ACT_LEAKY_RELU 2
/* 1 if (K inputs, M outputs) is inside the kernels' tile limits (currently K, M <= 64)               */
int32_t dn4gl_lin_supported(int32_t K, int32_t M);
size_t dn4gl_lin_workspace_bytes(int64_t N, int32_t K, int32_t M);
#define DN4GL_LIN_COUNTERS 64
/* Y (N x M) = act_in(bn_in(X)) W^T + bias.   X (N x K) row-major; in_bn NULL or the record (over K) of the previous
 * stage's BatchNorm; W (M x K) as nn.Linear stores it; bias NULL or (M).
 * If bn_out != NULL the per-channel batch statistics of Y (biased variance, eps) are reduced in a fixed order and
 * the record {mean, rstd, gamma*rstd, beta} (gamma / beta NULL = 1 / 0) is written to bn_out[4*M]; running_mean /
 * running_var (momentum, unbiased variance) and num_batches_tracked are updated in place when non-NULL -- the
 * training-mode semantics of nn.BatchNorm1d (at N = 1, which nn.BatchNorm1d refuses in training, running_var takes the
 * biased variance, 0).  ws: dn4gl_lin_workspace_bytes.  counters: DN4GL_LIN_COUNTERS int32 that are
 * 0 on entry and left 0 (arrival / ticket counters of the grid rendezvous that merges the per-CTA partials -- the stage
 * kernels are launched cooperatively; one array per stream that runs these stages concurrently).                      */
int dn4gl_lin_fwd_f32(const float *X, int64_t N, int32_t K, const float *in_bn, int32_t in_act, float in_slope,
                      const float *W, const float *bias, int32_t M, float *Y,
                      const float *gamma, const float *beta, float eps, float momentum, float *bn_out,
                      float *running_mean, float *running_var, int64_t *num_batches_tracked,
                      void *ws, size_t ws_bytes, int32_t *counters, void *stream);
/* Backward of one stage  Y = X' W^T + b,  X' = act_in(bn_in(X)):
 *   gY = G                                  (bn == NULL), or the BatchNorm(+ReLU) backward of the stage OUTPUT:
 *        gm = G * [bn(Y) > 0] (skipped when g_masked), gY = k * (gm - s1/N - xhat * s2/N), xhat = (Y - mean) * rstd,
 *        sums = {s1[M], s2[M]} = {sum gm, sum gm*xhat} (dn4gl_bn_bwd_sums_f32 or the sums_prev of the stage after);
 *   dW (M x K) = gY^T X',  db (M) = colsum gY   (either may be NULL);
 *   GX (N x K) = (gY W) * act_in'(bn_in(X))     (NULL: not needed), and when in_bn != NULL also
 *   sums_prev[2*K] = {sum GX, sum GX * xhat_in}: the batch sums the previous stage's backward needs, so the chain
 *   needs no separate reduction pass.  dgamma = s2, dbeta = s1 of the stage's own sums.
 * The upstream gradient is G[r] + Gseg[row2seg[r]]: G (N x M, may be NULL) is the gradient arriving row-wise (the next
 * layer's aggregation backward), Gseg (B x M, may be NULL, pre-scaled by 1/n_g for mean pooling) the gradient of the
 * per-graph readout of this stage's output (global_add_pool / global_mean_pool backward, gconv.py:213) -- the broadcast
 * row is added in the prologue instead of being materialised as an N x M tensor.  counters: as for dn4gl_lin_fwd_f32. */
int dn4gl_lin_bwd_f32(const float *G, const float *Gseg, const int32_t *row2seg, const float *Yout, int64_t N, int32_t M,
                      const float *bn, const float *sums, int32_t g_masked,
                      const float *W, int32_t K,
                      const float *X, const float *in_bn, int32_t in_act, float in_slope,
                      float *GX, float *sums_prev, float *dW, float *db,
                      void *ws, size_t ws_bytes, int32_t *counters, void *stream);
/* out = act(bn(Y))  (bn NULL = identity): the activation a stage hands to the aggregation / readout kernels      */
int dn4gl_bn_act_f32(const float *Y, int64_t N, int32_t M, const float *bn, int32_t act, float slope, float *out,
                     void *stream);
/* sums[2*M] = {sum_r gm, sum_r gm * xhat}, gm = G * act'(bn(Y)): the batch sums of a BatchNorm whose output
 * gradient G arrives from outside the MLP (aggregation / readout backward).  counters: DN4GL_LIN_COUNTERS zeroed int32,
 * left at zero (the per-CTA partials are merged inside the kernel after a grid rendezvous)                         */
size_t dn4gl_bn_bwd_sums_workspace_bytes(int64_t N, int32_t M);
int dn4gl_bn_bwd_sums_f32(const float *G, const float *Gseg, const int32_t *row2seg, const float *Y, int64_t N, int32_t M,
                          const float *bn, int32_t act, float slope, float *sums, void *ws, size_t ws_bytes,
                          int32_t *counters, void *stream);
/* Stand-alone training-mode BatchNorm1d for widths above the fused stages' (M <= 128; gconv.py:190-196 with main.py:174's
 * hidden 128): _stats writes the record {mean, rstd, gamma*rstd, beta} of Y's batch statistics to bn_out[4*M] (fixed-order
 * double-precision merge of per-CTA shifted sums) and updates running_mean / running_var / num_batches_tracked like
 * nn.BatchNorm1d (NULL = skip); dn4gl_bn_act_f32 applies it.  _bwd_apply: GX = gamma rstd (gm - s1 / N - xhat s2 / N) with
 * gm = G * act'(bn(Y)) and sums = {s1, s2} from dn4gl_bn_bwd_sums_f32 (d beta = s1, d gamma = s2).                      */
size_t dn4gl_bn_stats_workspace_bytes(int64_t N, int32_t M);
int dn4gl_bn_stats_f32(const float *Y, int64_t N, int32_t M, const float *gamma, const float *beta, float eps, float momentum,
                       float *running_mean, float *running_var, int64_t *num_batches_tracked, float *bn_out, void *ws,
                       size_t ws_bytes, void *stream);
int dn4gl_bn_bwd_apply_f32(const float *G, const float *Y, int64_t N, int32_t M, const float *bn, const float *sums, int32_t act,
                           float slope, float *GX, void *stream);
/* out = act(bn(Y)) and pooled[b,:] = sum (mode 0) / mean (mode 1) of out over rows [seg_ptr[b], seg_ptr[b+1]) in one pass
 * (the layer output handed to the next aggregation + its global_add_pool / global_mean_pool readout, gconv.py:213)   */
int dn4gl_bn_act_pool_f32(const float *Y, int64_t N, int32_t M, const float *bn, int32_t act, float slope, float *out,
                          const int32_t *seg_ptr, int32_t B, int32_t mode, float *pooled, void *stream);
/* out[i] = index of the contiguous segment holding row i (PyG's `batch` vector as int32)                             */
int dn4gl_segment_ids_i32(const int32_t *seg_ptr, int32_t B, int64_t N, int32_t *out, void *stream);

/* ---- optimizer step ---------------------------------------------------------------------------------------- */
/* ---- general fp32 GEMM on the tensor cores (3xTF32, csrc/gemm3x.cu) ----------------------------------------
 * C (N x M, leading dimension ldc) = A (N x K, leading dimension lda) * B (+ bias[M] if non-NULL), fp32 in and out.
 *   b_layout 0: B is an nn.Linear weight, (M x K) row-major with leading dimension ldb:  C = A B^T  -- the layers of
 *               rgin.py:52 / dmpnn.py:47,55 / pred.py and the data gradient of `x @ w`;
 *   b_layout 1: B is (K x M) row-major with leading dimension ldb:  C = A B  -- the relation-table, loop, P|Q and T
 *               products (rgin.py:137-154, dmpnn.py:111-156, rgconv.py:48-51) and the data gradient of nn.Linear.
 * Any N, K >= 1, M; any alignment (rows that are not 16-byte aligned take scalar loads / stores).  Every operand is
 * split hi + lo in tf32, hi*hi + hi*lo + lo*hi is formed per 32-wide chunk of K in tensor memory (lo products first) and
 * the chunks are added in fp32 registers with round-to-nearest: errors at the level of an fp32 FMA loop, not of a
 * single-pass TF32 GEMM.  ws: dn4gl_gemm_workspace_bytes(K, M) bytes, 16-byte aligned (the split, swizzled copy of B).  */
size_t dn4gl_gemm_workspace_bytes(int32_t K, int32_t M);
int dn4gl_gemm_f32(const float *A, int64_t N, int32_t K, int32_t lda, const float *B, int32_t ldb, int32_t b_layout,
                   int32_t M, const float *bias, float *C, int32_t ldc, void *ws, size_t ws_bytes, void *stream);

/* ---- data-parallel exchange (SURVEY.md 8(e); the reference is single-device) --------------------------------
 * One-shot all-reduce of the flat gradient bucket over NVLink peer memory, one node, world <= 8:
 *   bucket[i] <- sum_{s = 0 .. world-1} weight_s * bucket_s[i]      on every rank, added in rank order (every rank
 * computes the same bits).  bucket: this rank's n floats (n % 4 == 0, 16-byte aligned), updated in place.  exposed /
 * signals: HOST arrays of `world` device pointers -- entry `rank` is this rank's own exposed area (2 n floats) / signal
 * words (DN4GL_PEER_SIGNAL_WORDS int32, zeroed once at set-up, never reset afterwards), the others are peer mappings of
 * the other ranks' (CUDA IPC handles opened with dn4gl_ipc_open).  weight: this rank's weight (B_r / B for a
 * mean-reduced loss).  Every rank must issue the call the same number of times with the same n (it is a collective: block
 * b of a rank waits for block b of every other rank inside the kernel, bounded -- a missing peer traps).  Replaces
 * `flat *= weight; dist.all_reduce(flat)` of the pipelines; the library collective remains the fallback when the mappings
 * cannot be set up.                                                                                                */
#define DN4GL_PEER_SIGNAL_WORDS 2048
int dn4gl_ipc_open(const void *handle, void **base_out);   /* handle: the 64 bytes of a cudaIpcMemHandle_t; maps it for the
                                                               current device, peer access enabled on demand           */
int dn4gl_ipc_close(void *base);
int32_t dn4gl_peer_allreduce_grid(int64_t n);
int dn4gl_peer_allreduce_f32(float *bucket, int64_t n, float weight, float *const *exposed, int32_t *const *signals,
                             int32_t rank, int32_t world, void *stream);

/* One Adam / AdamW (optionally amsgrad) update over FLAT fp32 buffers of n elements -- replaces the per-tensor kernels
 * of torch.optim.Adam.step() (graph_neural_networks/main.py:43) and torch.optim.AdamW(amsgrad=True).step()
 * (subgraph_isomorphism/train.py:831-838), same update rule and operation order as torch's single-tensor path:
 *   [decoupled: p *= 1 - lr*wd | else g += wd*p];  m += (g - m)(1 - b1);  v = v*b2 + (1 - b2) g*g;
 *   [amsgrad: vmax = max(vmax, v)];  p -= lr / (1 - b1^t) * m / (sqrt(v | vmax) / sqrt(1 - b2^t) + eps),  t = step + 1.
 * hyper: 5 device floats {lr, beta1, beta2, eps, weight_decay}; step: 1 device float holding the number of updates done
 * so far, advanced by the kernel (so a captured CUDA graph replays with the right bias correction and the current lr);
 * max_exp_avg_sq NULL = no amsgrad; counter: one int32 that is 0 on entry (left 0).  All buffers 16-byte aligned.     */
int dn4gl_adam_f32(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *max_exp_avg_sq,
                   int64_t n, const float *hyper, float *step, int32_t decoupled, int32_t *counter, void *stream);

/* out[0] = sum_i a[i] * b[i] over n floats, fixed-order (the gradient of GINConv's trainable eps: sum(g_z * x)).
 * ws: dn4gl_dot_workspace_bytes; counter: one int32 that is 0 on entry (left 0).                                  */
size_t dn4gl_dot_workspace_bytes(int64_t n);
int dn4gl_dot_f32(const float *a, const float *b, int64_t n, float *out, void *ws, size_t ws_bytes, int32_t *counter,
                  void *stream);

/* ---- mini-batch assembly from a data set resident in HBM (datasets.py; replaces the host-side collation of PyG's
 * DataLoader and of GraphAdjDataset.batchify, subgraph_isomorphism/dataset.py:1604-1636) ----------------------------
 * Segmented gather of one level (nodes, edges, graphs, subisomorphism values) for all of its columns in one launch.
 * ptr_in[n_seg_in + 1]: the data set's item offsets of the level; idx[K]: the segments to take, each in [0, n_seg_in)
 * (the caller validates them: an index outside is never read and leaves its output items unwritten); ptr_out[K + 1]:
 * the batch's offsets (ptr_out[k+1] - ptr_out[k] = ptr_in[idx[k]+1] - ptr_in[idx[k]]).  col_in / col_out: HOST arrays of
 * ncols (1..8) device column pointers, col_words[c] (host) 4-byte words per item (1 for an int32 / float column, F for
 * an F-wide float attribute, 2 for int64).  For k < K and j below the segment's length, item ptr_out[k] + j of every
 * output column is item ptr_in[idx[k]] + j of its input column; in columns with col_rebase[c] != 0 (host) each int32
 * word also gets rebase_out[k] - rebase_in[idx[k]] added (device arrays; the node offsets on the edge level, so that
 * src / dst become batch-global node ids).  No allocation, no atomics, deterministic; K == 0 is a no-op.            */
int dn4gl_gather_segments(int32_t K, const int32_t *idx, const int32_t *ptr_in, int64_t n_seg_in,
                          const int32_t *ptr_out, const int32_t *rebase_in, const int32_t *rebase_out,
                          int32_t ncols, const void *const *col_in, void *const *col_out,
                          const int32_t *col_words, const int32_t *col_rebase, void *stream);

/* ---- evaluation over a held-out split (pipelines.py evaluate; the reference's eval_test, main.py:54, and evaluate,
 * subgraph_isomorphism/train.py:609-618) ----------------------------------------------------------------------------
 * Record kernels write one record per sample of a batch at positions pos0 .. pos0 + B - 1 of split-sized arrays.
 * dn4gl_eval_class_rows_f32: logp (B, C) row-major log-probabilities, y[B] int64 targets.  pred[p] = arg-max of the
 *   row as torch.max(dim=1) picks it (lowest index on ties; a NaN counts as the largest value, the first NaN wins);
 *   nll[p] = -logp[b, y[b]]; correct[p] = 1.f if pred == y else 0.f.  A y outside [0, C) contributes nll 0 and is never
 *   correct (as in dn4gl_nll_mean_f32).  A row holding a NaN gets nll = NaN and correct = 0, whatever its target.
 * dn4gl_eval_count_rows_f32: pred_c[B] fp32, counts[B] int64; with r = relu(pred_c), t = (float)count:
 *   pred[p] = pred_c[b]; err[3p .. 3p+2] = { |r - t|, (r - t)^2, smooth-L1(r - t, beta 1) } (F.l1_loss / F.mse_loss /
 *   F.smooth_l1_loss per element).
 * dn4gl_eval_reduce_f32: out[c] = sum_{i < n} v[i * k + c] in double for k (1..8) interleaved fp32 columns.  The order
 *   is fixed by n alone (tiles of 1024 rows summed by a fixed tree, tile partials merged in tile order by a fixed tree;
 *   csrc/eval.cu), not by the grid or the SM count.  ws: dn4gl_eval_reduce_workspace_bytes(n, k) bytes, 8-byte
 *   aligned; counter: one int32 that is 0 on entry (left 0).  n == 0 writes k zeros and reads nothing.              */
int dn4gl_eval_class_rows_f32(const float *logp, const int64_t *y, int32_t B, int32_t C, int64_t pos0, int32_t *pred,
                              float *nll, float *correct, void *stream);
int dn4gl_eval_count_rows_f32(const float *pred_c, const int64_t *counts, int32_t B, int64_t pos0, float *pred,
                              float *err, void *stream);
size_t dn4gl_eval_reduce_workspace_bytes(int64_t n, int32_t k);
int dn4gl_eval_reduce_f32(const float *v, int64_t n, int32_t k, double *out, void *ws, size_t ws_bytes,
                          int32_t *counter, void *stream);

/* ---- small fused elementwise helpers of the layers ------------------------------------------ */
/* gather rows: out[i,:] = x[idx[i],:] (idx int32, n rows)                                       */
int dn4gl_gather_rows_f32(const int32_t *idx, const float *x, float *out, int64_t n, int32_t D, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DN4GL_H */
