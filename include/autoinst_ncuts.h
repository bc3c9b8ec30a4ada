/*
 * autoinst_ncuts.h — C ABI of libautoinst_ncuts.so, the B200 (sm_100a) implementation of the
 * chunk-level normalized-cuts path of artonson/autoinst (reference: pipeline/ncuts/).
 *
 * The reference is pure Python and has no FFI; its boundary for this path is two imports
 * (pipeline/run_pipeline.py:14-17, pipeline/ncuts/ncuts_utils.py:22).  The entry points below are
 * what a ctypes binding inside those two modules calls (see INTEGRATION.md); each one names the
 * reference lines it replaces.
 *
 * Conventions
 *  - every function returns 0 on success or a negative ANCUTS_E* code; ancuts_last_error() gives a
 *    thread-local message for the last failure on the calling thread;
 *  - pointers named d_* are device pointers on the handle's device, h_* are host pointers;
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream); device-pointer entry
 *    points are asynchronous on it unless they return data through host pointers;
 *  - one handle per (device, host thread); a handle owns a growable device workspace.
 *  - dense matrices are row-major float32 with leading dimension ld (elements), ld % 4 == 0 and a
 *    16-byte aligned base.
 */
#ifndef AUTOINST_NCUTS_H
#define AUTOINST_NCUTS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ANCUTS_OK            0
#define ANCUTS_EINVAL       -1   /* bad argument */
#define ANCUTS_ECUDA        -2   /* CUDA runtime error (message holds cudaGetErrorString) */
#define ANCUTS_ENOMEM       -3   /* workspace allocation failed */
#define ANCUTS_ENOTCONV     -4   /* reserved; non-convergence is counted per call: ancuts_last_unconverged() */
#define ANCUTS_EUNSUPPORTED -5   /* e.g. beta != 0 (SAM term, ncuts_utils.py:115-123) */

#define ANCUTS_NUM_CUTS 10       /* normalized_cut.py:54 calls get_min_ncut(ev, D, w, 10) */

typedef struct ancuts_handle ancuts_handle;

/* Gains and thresholds of one run: pipeline/config.py:6-37 (alpha, theta, gamma, T) and
 * config.py:61,65 (SPLIT_LIM, PROXIMITY_THRESHOLD). */
typedef struct ancuts_params {
    double alpha;        /* spatial gain  (ncuts_utils.py:63-66);  0 -> term is the mask        */
    double theta;        /* TARL gain     (ncuts_utils.py:135-149); 0 -> term is the mask        */
    double gamma;        /* DINOv2 gain   (ncuts_utils.py:125-133); 0 -> term is the mask        */
    double proximity;    /* PROXIMITY_THRESHOLD, inclusive (ncuts_utils.py:61)                   */
    double T;            /* N-cut stopping threshold, strict '<' (normalized_cut.py:56)          */
    double split_lim;    /* size limit at the root (normalized_cut.py:39-40); children use 0.01  */
    int    tarl_dim;     /* 96  (0 when d_tarl is NULL) */
    int    dino_dim;     /* 384 (0 when d_dino is NULL) */
    int    lanczos_max_steps;   /* 0 -> default (1024) */
    int    lanczos_check_every; /* 0 -> default (16)   */
    double lanczos_tol;         /* 0 -> default (1e-10): residual <= tol * (theta1 - theta2) */
    int    affinity_impl;       /* 0 = exact CUDA-core tile kernel, 1 = tcgen05 Gram GEMM */
    int    lanczos_impl;        /* 0 = persistent cluster kernel for nodes <= 4096 points, grid-wide
                                   multi-launch path above; 1 = multi-launch path for every node */
} ancuts_params;

/* One row per recursion node that reached the eigensolver (debug / accounting; SURVEY.md §8d). */
typedef struct ancuts_node_stat {
    int32_t chunk;       /* chunk index within the call */
    int32_t n;           /* node size */
    int32_t steps;       /* Lanczos steps taken */
    int32_t converged;   /* 1 = residual test met or Krylov space exhausted */
    int32_t best_k;      /* index of the chosen threshold, -1 = none (allclose) */
    int32_t split;       /* 1 = mcut < T */
    int32_t level;       /* recursion level */
    int32_t n_side;      /* points on the mask side of the chosen cut */
    double  lambda2;     /* second smallest eigenvalue of the normalised Laplacian */
    double  mcut;        /* N-cut value of the chosen cut */
} ancuts_node_stat;

int         ancuts_version(void);
const char* ancuts_last_error(void);
int         ancuts_create(int device, ancuts_handle** out);
int         ancuts_destroy(ancuts_handle* h);
/* bytes of device workspace a segment call over these chunk sizes needs (for batch planning) */
int64_t     ancuts_segment_workspace_bytes(int num_chunks, const int32_t* h_chunk_n, int lanczos_max_steps);

/* Stage 1 — replaces ncuts_utils.py:60-66,125-133,135-156 (3x cdist + mask + exp + product).
 * d_points: n x 3 float64; d_tarl: n x tarl_dim float32 or NULL; d_dino: n x dino_dim float32 or NULL.
 * Writes the dense n x n float32 affinity (zeros outside the proximity mask, 1 on the diagonal)
 * and, if d_rowsum != NULL, float64 row sums. */
int ancuts_affinity_f32(ancuts_handle* h, int n, const double* d_points, const float* d_tarl,
                        const float* d_dino, const ancuts_params* p, float* d_W, int64_t ld,
                        double* d_rowsum, void* stream);

/* DINOv2 term over several cameras (the reference's CAM_IDS, ncuts_utils.py:125-133: exp(-gamma cdist(g_c, g_c)) multiplied
 * over the cameras c).  The ancuts_*_cams* entry points take d_dino / h_dino point-major: n x dino_cams x p->dino_dim float32,
 * row i = camera 0's dino_dim values, then camera 1's, ...; p->dino_dim is the width of ONE camera (a multiple of 4).  The term
 * is evaluated as exp(-gamma * S) with S = dd_0 + dd_1 + ... (float64, camera order), dd_c the Euclidean distance of the two
 * rows' camera-c slices; zero rows are not neutralised in any camera.  dino_cams >= 1; dino_cams = 1 gives exactly what the
 * entry point without _cams gives (which forwards here with dino_cams = 1).  dino_cams > 1 with affinity_impl = 1 (tensor-core
 * form) returns ANCUTS_EUNSUPPORTED. */
int ancuts_affinity_cams_f32(ancuts_handle* h, int n, const double* d_points, const float* d_tarl,
                             const float* d_dino, int dino_cams, const ancuts_params* p, float* d_W, int64_t ld,
                             double* d_rowsum, void* stream);

/* Stage 2 — replaces normalized_cut.py:38,42-47 (W = w + I, d = W.sum(0), D^-1/2 W D^-1/2).
 * d_deg[i] = 1 + sum_j w_ij (float64).  If d_M != NULL also writes M = D^-1/2 (w+I) D^-1/2 in
 * float32 (the pipeline itself applies the scaling inside the matvec and never materialises M). */
int ancuts_degree_normalize_f32(ancuts_handle* h, int n, const float* d_W, int64_t ld,
                                double* d_deg, float* d_M, int64_t ldm, void* stream);

/* Stage 3 — replaces normalized_cut.py:49-53 (eigsh(A, 2, sigma=1e-10) + argsort).
 * Nodes are diagonal blocks [off, off+n) of the dense matrix.  For each node writes the unit-norm
 * Fiedler vector with sum >= 0 into d_ev[off .. off+n), and per node lambda2 / steps / converged
 * to the host arrays.  Blocks until done. */
int ancuts_lanczos_fiedler_batched(ancuts_handle* h, int n_total, const float* d_W, int64_t ld,
                                   int num_nodes, const int32_t* h_node_off, const int32_t* h_node_n,
                                   const ancuts_params* p, double* d_ev, double* h_lambda2,
                                   int32_t* h_steps, int32_t* h_converged, void* stream);

/* Stage 4a — replaces get_min_ncut / ncut_cost / cut_cost (normalized_cut.py:4-34): all ten
 * threshold cuts from one pass over each block.  d_ev as produced by stage 3.
 * h_best_k[node] = -1 when min and max of ev are allclose; d_side[i] = 1 where ev > threshold
 * (the reference's mask) for the chosen cut, 0 elsewhere.  Blocks until done. */
int ancuts_ncut_scan_batched(ancuts_handle* h, int n_total, const float* d_W, int64_t ld,
                             int num_nodes, const int32_t* h_node_off, const int32_t* h_node_n,
                             const double* d_ev, int32_t* h_best_k, double* h_mcut,
                             double* h_costs /* num_nodes x 10 or NULL */, uint8_t* d_side, void* stream);

/* Stage 4b — replaces w[mask][:, mask], w[~mask][:, ~mask], labels[mask] (normalized_cut.py:57-58):
 * stable partition of every node (mask side first), each side further split into the connected
 * components of its sub-graph, blocks gathered into d_W_out.  d_perm_out[new position] = old
 * position; child ranges are returned through the host arrays (capacity n_total). Blocks. */
int ancuts_partition_batched(ancuts_handle* h, int n_total, const float* d_W_in, float* d_W_out,
                             int64_t ld, int num_nodes, const int32_t* h_node_off,
                             const int32_t* h_node_n, const uint8_t* d_side, int split_components,
                             int32_t* d_perm_out, int32_t* h_num_children, int32_t* h_child_off,
                             int32_t* h_child_n, void* stream);

/* Whole path on the device for a batch of chunks — replaces ncuts_utils.py:56-174 per chunk
 * (affinity -> remove_isolated_points (no-op) -> normalized_cut -> labels, :177-183).
 * Chunk c owns points [h_chunk_off[c], h_chunk_off[c+1]) of the concatenated inputs.
 * d_labels[i] = segment id of point i within its chunk (0 .. h_num_segments[c]-1).
 * h_stats/h_num_stats: optional per-node log (capacity stats_cap).  Blocks until done. */
int ancuts_segment_chunks(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off,
                          const double* d_points, const float* d_tarl, const float* d_dino,
                          const ancuts_params* p, int32_t* d_labels, int32_t* h_num_segments,
                          ancuts_node_stat* h_stats, int32_t stats_cap, int32_t* h_num_stats,
                          void* stream);

/* Same with HOST buffers (pinned memory recommended): copies inputs to the device, runs, copies
 * labels back.  This is the call ncuts_chunk() makes (ncuts_utils.py:28-204). */
int ancuts_segment_chunks_host(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off,
                               const double* h_points, const float* h_tarl, const float* h_dino,
                               const ancuts_params* p, int32_t* h_labels, int32_t* h_num_segments,
                               ancuts_node_stat* h_stats, int32_t stats_cap, int32_t* h_num_stats,
                               void* stream);

/* The two above with the DINOv2 input of several cameras (layout and term: ancuts_affinity_cams_f32).  The host form copies
 * each chunk's n_c x dino_cams x dino_dim floats as one piece. */
int ancuts_segment_chunks_cams(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off,
                               const double* d_points, const float* d_tarl, const float* d_dino, int dino_cams,
                               const ancuts_params* p, int32_t* d_labels, int32_t* h_num_segments,
                               ancuts_node_stat* h_stats, int32_t stats_cap, int32_t* h_num_stats,
                               void* stream);
int ancuts_segment_chunks_cams_host(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off,
                                    const double* h_points, const float* h_tarl, const float* h_dino, int dino_cams,
                                    const ancuts_params* p, int32_t* h_labels, int32_t* h_num_segments,
                                    ancuts_node_stat* h_stats, int32_t stats_cap, int32_t* h_num_stats,
                                    void* stream);

/* normalized_cut(w, num_points_orig, labels, T, split_lim) (normalized_cut.py:37) on a dense
 * float32 copy of w already on the device (n x n, unit diagonal, symmetric). Blocks. */
int ancuts_segment_dense_f32(ancuts_handle* h, int n, const float* d_W, int64_t ld,
                             int num_points_orig, const ancuts_params* p, int32_t* d_labels,
                             int32_t* h_num_segments, ancuts_node_stat* h_stats, int32_t stats_cap,
                             int32_t* h_num_stats, void* stream);

/* normalized_cut(w, num_points_orig, labels, T, split_lim) (normalized_cut.py:37-63) for a BATCH of sparse
 * affinity graphs in CSR form on the device -- the scipy CSR `w` that ncuts_utils.py:167-174 passes, or any
 * affinity a caller builds.  Graph c owns rows [h_graph_off[c], h_graph_off[c+1]) of one concatenated CSR
 * (h_graph_off[0] = 0): d_row_ptr has P + 1 global entry offsets (d_row_ptr[0] = 0, d_row_ptr[P] = nnz), d_col
 * the column LOCAL to the row's graph (0 .. n_c - 1), d_val the float32 value.  The CSR is read in place.
 * Each graph must be symmetric bit for bit (an absent entry counts as 0), have a unit diagonal (a stored diagonal
 * entry is exactly 1.0f, an absent one is taken as 1), strictly increasing columns per row and finite values; a
 * stored 0 is no edge.  A violation returns ANCUTS_EINVAL naming the graph, the row and the rule; no malformed
 * d_row_ptr / d_col makes any kernel read outside the arrays.  The result is the one ancuts_segment_dense_f32
 * gives on the densified graph.  h_num_points_orig: per-graph num_points_orig, or NULL for each graph's own
 * size.  Of p only T, split_lim and the lanczos_* fields are read.  d_labels, h_num_segments and the stats are
 * as in ancuts_segment_chunks (`chunk` of a record = graph index).  Blocks. */
int ancuts_segment_csr_f32(ancuts_handle* h, int num_graphs, const int64_t* h_graph_off,
                           const int64_t* d_row_ptr, const int32_t* d_col, const float* d_val, int64_t nnz,
                           const int32_t* h_num_points_orig, const ancuts_params* p, int32_t* d_labels,
                           int32_t* h_num_segments, ancuts_node_stat* h_stats, int32_t stats_cap,
                           int32_t* h_num_stats, void* stream);

/* "Next" row N1 — replaces kDTree_1NN_feature_reprojection (point_cloud_utils.py:144-174, called at
 * ncuts_utils.py:185-189): every query point (5 cm cloud) takes the label of its nearest source point
 * (0.35 m cloud).  d_source_label may be NULL (the source index is returned as label).  max_radius <= 0
 * disables the radius test; otherwise points farther than max_radius get no_label.  Asynchronous. */
int ancuts_nn_reproject(ancuts_handle* h, int num_query, const double* d_query, int num_source,
                        const double* d_source, const int32_t* d_source_label, double max_radius,
                        int32_t no_label, int32_t* d_out_label, int32_t* d_out_index, void* stream);

/* "Next" row N3 (TARL half) — replaces the per-point KD-tree loop of tarl_features_per_patch
 * (pipeline/utils/point_cloud/chunk_generation.py:205-258, called at ncuts_utils.py:135-141): every major point
 * takes the float64 mean of the feature rows of the scan points strictly closer than `radius`
 * (MAJOR_VOXEL_SIZE / 2, :212,249-252; Open3D's radius search keeps squared distance < radius^2); major points
 * without such a neighbour keep a zero row (:247,255-256).  Scan points take part only if strictly inside the
 * box (h_box_min, h_box_max) = center_position -/+ CHUNK_SIZE / 2 (:220-221,233-236); the two bounds are HOST
 * arrays of 3 doubles.  d_scan_points: num_scan x 3 float64 (already in the chunk frame, :228-231),
 * d_scan_feat: num_scan x feat_dim float32 (feat_dim <= 384), d_out: num_major x feat_dim float64,
 * d_out_count: neighbours per major point (may be NULL).  normalise != 0 divides each non-empty row by its
 * L2 norm (TARL_NORM, :253-254).  The workspace is the caller's (ancuts_feature_pool_workspace_bytes).
 * Asynchronous on `stream`; deterministic (fixed summation order). */
int64_t ancuts_feature_pool_workspace_bytes(int num_scan);
int ancuts_feature_pool(ancuts_handle* h, int num_major, const double* d_major, int num_scan,
                        const double* d_scan_points, const float* d_scan_feat, int feat_dim, double radius,
                        const double* h_box_min, const double* h_box_max, int normalise, double* d_out,
                        int32_t* d_out_count, void* d_workspace, int64_t workspace_bytes, void* stream);

/* "Next" row N3 (DINOv2 half) — replaces the per-view part of image_based_features_per_patch behind the visibility
 * bookkeeping (pipeline/utils/image/image_utils.py:264-346, called at ncuts_utils.py:81-110) and dinov2_mean (:363-371).
 * ancuts_dino_view_pixels, one call per view: every major point (d_major_cam, N x 3 float64, already in the view's camera
 * frame, :264) looks up its nearest visible chunk point (d_visible_cam, M x 3 float64, same frame, :262-263) and is kept
 * if that distance is strictly below max_dist (MAJOR_VOXEL_SIZE / 2, :271-276); kept points are projected with the 3 x 3
 * intrinsics h_K (row-major, HOST array): K p, division by the depth, np.round, inside the img_h x img_w image and depth > 0
 * (point_to_pixels.py:21-30); d_out_pixel[i] = int(map_h / img_h * row) * map_w + int(map_w / img_w * col) (:255-256,
 * 341-346) or -1.  ancuts_dino_mean: d_view_pixel is num_views x N (views the reference skips, :183-191,:212-214, hold -1
 * everywhere), h_feature_maps a HOST array of num_views device pointers to map_h x map_w x feat_dim float32 maps; a view
 * counts for a point if its looked-up feature vector has any non-zero entry; d_out (N x feat_dim float64) = the mean over
 * those views in view order, zero row if none; d_out_count their number (may be NULL).  Asynchronous on `stream`
 * (ancuts_dino_mean synchronises once to read the pointer table). */
int ancuts_dino_view_pixels(ancuts_handle* h, int num_major, const double* d_major_cam, int num_visible,
                            const double* d_visible_cam, double max_dist, const double* h_K, int img_h, int img_w,
                            int map_h, int map_w, int32_t* d_out_pixel, void* stream);
int ancuts_dino_mean(ancuts_handle* h, int num_major, int num_views, const int32_t* d_view_pixel,
                     const float* const* h_feature_maps, int feat_dim, double* d_out, int32_t* d_out_count, void* stream);

/* "Next" row N2 — replaces merge_chunks_unite_instances2 (pipeline/utils/point_cloud/point_cloud_utils.py:387-491; caller
 * pipeline/run_pipeline.py:197-199): the chunk labelings of one map, chunks in file-name order, are united into one map
 * labeling.  Chunk c owns points [h_chunk_off[c], h_chunk_off[c+1]) of d_points (P x 3 float64) and d_labels (P int32,
 * 0 = background / "black", :428; every other value names an instance and must not be negative).  Per new chunk:
 * crop of the merge so far to the cube h_centers[c] +/- crop_half_side (20.0, inclusive, :405-417; the centre is the mean
 * of the chunk's points, :397-403, computed by the caller with the reference's own expression), per-instance bounding
 * boxes (:447-448), points of every new instance inside them (:452-455), union = number of DISTINCT SCALAR coordinate
 * values of both instances (np.unique without axis, :457), iou > min_iou (0.01, :459), every new instance keeps the
 * cropped instance with the largest iou in (id1, id2) ascending order with strict replacement (:465-477), recolour
 * (:479-481), append and drop exact-coordinate duplicates keeping the first occurrence (:488-489).
 * d_out_labels[P]: label of every slot after the association; d_out_index: indices of the surviving points in order
 * (capacity P; may be NULL); *h_num_kept their number.  Blocks until done. */
int ancuts_merge_chunks(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const double* d_points,
                        const int32_t* d_labels, const double* h_centers, double crop_half_side, double min_iou,
                        int32_t* d_out_labels, int64_t* d_out_index, int64_t* h_num_kept, void* stream);

/* Glue of run_pipeline.py:216-218 for integer labels: per-chunk segment ids (0 .. n_c - 1, as the segment calls write
 * them) -> labels unique across the map, ((c + 1) << id_shift) + r + 1 with r = rank of the segment by first occurrence
 * in the chunk's point order (the reference's colours are random; its greedy rules depend on the order of the label
 * values, so both sides of a comparison need the same, labeling-independent numbering; SURVEY.md Appendix B). */
int ancuts_map_labels(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const int32_t* d_seg_labels,
                      int id_shift, int32_t* d_out_labels, void* stream);

/* remove_semantics(labels, preds, threshold) (point_cloud_utils.py:253-287; caller run_pipeline.py:223): a predicted
 * label with more than `threshold` (0.8) of its points on ground-truth background (gt == 0) becomes 0.  Asynchronous. */
int ancuts_remove_semantics(ancuts_handle* h, int64_t n, const int32_t* d_gt_labels, const int32_t* d_pred_labels,
                            double threshold, int32_t* d_out_labels, void* stream);

/* "Next" row N4 — Metrics(...).update_stats(all_labels, pred_labels, gt_labels) of a fresh Metrics object for one map
 * (pipeline/metrics/metrics_class.py:137-179): filter_labels (:302-309, fewer than min_points points -> 0) on both
 * prediction arrays, IoU table of the co-occurring (pred, gt) pairs (:296-300), greedy first-unused-GT matching in
 * np.unique order at IoU 0.5 for P / R / F1 (:61-117,315-340) and at the 11 overlaps of :40 for AP with constant
 * confidence (:181-235, np.trapz with the sentinels), and the association term of modified_LSTQ.py:23-80 on all_labels.
 * h_out (21 doubles): [0..6] p, r, f1, ap, ap0.25, ap0.5, S_assoc (the keys of sequence_stats, :262-269);
 * [7..9] true positives, n_pred, n_gt at IoU 0.5; [10..20] AP per overlap.  Labels must not be negative.  Blocks. */
int ancuts_instance_metrics(ancuts_handle* h, int64_t n, const int32_t* d_all_labels, const int32_t* d_pred_labels,
                            const int32_t* d_gt_labels, int min_points, double* h_out, void* stream);

/* Eigensolver nodes of the handle's last segment call (ancuts_segment_chunks / _host / _dense_f32) that stopped at
 * lanczos_max_steps without meeting the residual test.  Their cut used the unconverged Ritz vector; the reference's
 * eigsh (normalized_cut.py:49) raises ArpackNoConvergence in that situation, so callers must look at this count
 * (the Python drop-in raises, the array-level API warns). */
int ancuts_last_unconverged(ancuts_handle* h);

/* Alternative implementations behind the same results (each one parity-tested; 0 = the default).  Option 0 is retired
 * (it selected a dense affinity form of the segment path); setting it returns ANCUTS_EINVAL.
 *   ANCUTS_OPT_PAIR_SEARCH   0 cell-sorted tile sweep, all chunks of the call in one launch, tile pairs pruned by their boxes,
 *                             1 shuffled 64 x 64 tile sweep over the whole upper triangle, one launch per chunk
 *   ANCUTS_OPT_MATVEC         0 the cluster's row slices compressed (CSR) into shared memory once per node; a node whose
 *                               slices do not fit falls back, inside the kernel, to the dense form,
 *                             1 dense blocks streamed from HBM every Lanczos step (the north-star form; bench.py measures
 *                               its roofline)
 *   ANCUTS_OPT_CLUSTER_MAP    0 built-in; otherwise six decimal digits (1, 2, 4 or 8 each) = CTAs per node for the size bins
 *                             <= 320, 512, 640, 1024, 2048, 4096 points (tuning)
 *   ANCUTS_OPT_FUSED_CUT      0 a cluster kernel that holds its node as CSR slices also takes the node's cut decision (sign,
 *                               thresholds, buckets, N-cut scan, decision, side flags, component unions) in its epilogue,
 *                             1 the cut always runs as its own kernels after the eigensolver
 *   ANCUTS_OPT_NODE_FORM      0 recursion nodes of the segment path kept as CSR (built from the pair queue, children
 *                               compacted from the parent's rows); a node's dense block is written only for the nodes that
 *                               read dense W (slices that do not fit, nodes above 4096 points or past the cluster kernel's
 *                               step limit),
 *                             1 every node as a dense block in HBM (zeroed, scattered and gathered on every level).
 *                             Calls with a dense matvec, separate cut kernels, the grid-wide Lanczos path, the shuffled
 *                             pair search, caller-supplied graphs or an overflowed pair queue take form 1 */
#define ANCUTS_OPT_PAIR_SEARCH   1
#define ANCUTS_OPT_MATVEC        2
#define ANCUTS_OPT_CLUSTER_MAP   3
#define ANCUTS_OPT_FUSED_CUT     4
#define ANCUTS_OPT_NODE_FORM     5
#define ANCUTS_OPT_COUNT         6
int ancuts_set_option(ancuts_handle* h, int option, int value);

/* Shared-memory sparse matvec form (ANCUTS_OPT_MATVEC = 0), last segment call: out2[0] = sum over the nodes it ran of
 * Lanczos steps x stored entries (what the sparse lower bound of SURVEY.md §8d multiplies by 8 bytes), out2[1] = entries. */
int ancuts_last_sparse_accounting(ancuts_handle* h, double* out2);
/* Persistent Lanczos kernel, last segment call: out2[0] = Lanczos steps of the nodes it ran, out2[1] = steps among them
 * that took the full Gram-Schmidt pass (partial re-orthogonalisation, DESIGN.md §4.3). */
int ancuts_last_reorth_accounting(ancuts_handle* h, double* out2);

/* Counter for bench.py (`gpu_launches`): kernels launched by this handle since the last reset. */
int64_t ancuts_launch_count(ancuts_handle* h, int reset);
/* Accounting of the last segment call: algorithmic bytes (SURVEY.md §8d) and event-timed
 * milliseconds per stage: [0]=affinity [1]=degree [2]=matvec [3]=reorth [4]=scan [5]=cc+partition */
int ancuts_last_accounting(ancuts_handle* h, double* bytes6, double* ms6, int64_t* launches6);
/* CUDA-event timing of the library's own launches, summed per stage and read back with
 * ancuts_last_accounting: 0 = off, 1 = every launch, 2 = only the matvec launches (dominant kernel) */
int ancuts_set_stage_timing(ancuts_handle* h, int on);
/* Per-level trace of the last segment call in timing mode 2 (tools/level_profile.py): rows of 16 doubles
 * [0] active nodes, [1] nodes above the cluster kernel's size limit, [2] ms of the concurrent cluster
 * kernels of the level, [3..8] nodes per size bin, [9..14] cluster size used per bin.  Returns the row count. */
int ancuts_last_levels(ancuts_handle* h, double* out, int cap_rows);
/* Debug (handle created with ANCUTS_PHASES=1 in the environment): cycles spent by the persistent Lanczos kernel per
 * phase, [cluster size 1,2,4,8][basis write, matvec, alpha + three-term pass with norm and z push, multisection of the check,
 * dots of the full Gram-Schmidt pass, its update + norm, norm exchange + omega recurrence, rest of the check]. */
int ancuts_debug_phases(ancuts_handle* h, double* out32, int reset);

#ifdef __cplusplus
}
#endif
#endif /* AUTOINST_NCUTS_H */
