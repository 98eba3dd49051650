/*
 * shotfpfh_b200 — C ABI of the B200 (sm_100a) hot path of aubin-tchoi/shot-fpfh:
 * fixed-radius neighbour search -> SHOT / FPFH descriptors -> descriptor nearest-neighbour matching.
 *
 * The reference is pure Python and has no FFI of its own (SURVEY.md §8b); the entry points below are what a
 * binding for its hot-path functions has to call. Each one names the reference code it replaces (paths relative
 * to the reference repository). INTEGRATION.md shows the ctypes stubs a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C: pointers, sizes, an opaque grid handle; no C++ or torch types, no exceptions across the boundary;
 *   - every function returns SF_OK (0) or an SF_ERR_* code; sf_last_error() gives the text (thread-local);
 *   - pointers named *_dev are DEVICE pointers on the current CUDA device, `stream` is a cudaStream_t passed as
 *     void* (NULL = default stream); work is enqueued on that stream and the call returns without
 *     synchronising, except where a host result is produced (documented per function);
 *   - coordinates, normals, radii are float64 exactly as the reference's NumPy arrays (row-major (n,3));
 *   - neighbour lists are CSR: int64 offsets[q + 1], int32 entries;
 *   - "cell-sorted position" = index into the grid's internal cell-ordered copy of the cloud (better locality
 *     for the descriptor kernels); sf_grid_permutation maps it from/to original point indices.
 * There is no CPU fallback anywhere behind this ABI.
 */
#ifndef SHOTFPFH_B200_H
#define SHOTFPFH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SF_ABI_VERSION 15

#define SF_OK 0
#define SF_ERR_CUDA 1     /* a CUDA runtime call or kernel launch failed */
#define SF_ERR_ARG 2      /* invalid argument */
#define SF_ERR_CAPACITY 3 /* a fixed capacity (descriptor length, k, shared memory) was exceeded */

#define SF_SHOT_LEN 352 /* 11 cosine x 8 azimuth x 2 elevation x 2 radial bins (shot.py:197) */

typedef struct sf_grid sf_grid;

const char* sf_last_error(void);
int sf_abi_version(void);

/* ------------------------------------------------------------------------------------------------------------
 * G — spatial index.  Replaces `KDTree(points)` (sklearn; shot_parallelization.py:167, fpfh.py:26, shot.py:340).
 * ---------------------------------------------------------------------------------------------------------- */
int sf_grid_create(sf_grid** out);
int sf_grid_destroy(sf_grid* grid);

/* Builds (or rebuilds, reusing its buffers) the uniform grid over `n` points for searches of radius <= `radius`.
 * xyz_dev, normals_dev: float64 (n,3); normals_dev may be NULL when only neighbour search is needed.
 * Synchronises `stream` once (the bounding box is needed on the host to size the cell table). */
int sf_grid_build(sf_grid* grid, const double* xyz_dev, const double* normals_dev, int64_t n, double radius,
                  void* stream);
int sf_grid_info(const sf_grid* grid, int64_t* n, int64_t* ncells, double* cell_edge, int32_t* dims3);
/* The same build inside a bounding box the CALLER gives (lo3, hi3: host float64), without a bounding-box pass and
 * without synchronising: the cells are exactly those of any other cloud built in that box with that radius — a cell
 * with the same points in it yields the same candidate runs. For a rank of a spatially partitioned job (a slab of the
 * cloud plus the cells around it, in the geometry of the whole cloud: shot_fpfh_b200/distributed.py; the reference has
 * no counterpart, it builds one KDTree of everything, shot_parallelization.py:167). Every point is checked against the
 * box on the device: sf_grid_poll reports 1 when one lay outside (the build is then memory-safe but wrong).
 * sf_grid_geometry: the cell edge and table dimensions sf_grid_build / _in_box derive from a box and a radius. */
int sf_grid_build_in_box(sf_grid* grid, const double* xyz_dev, const double* normals_dev, int64_t n, double radius,
                         const double* lo3, const double* hi3, void* stream);
int sf_grid_geometry(const double* lo3, const double* hi3, double radius, double* cell_edge, int32_t* dims3,
                     int64_t* ncells);
/* Calls without host synchronisation, for a caller that repeats the same work on one handle (a loop over time steps,
 * blocks of queries, a benchmark). `mode` bit 0: sf_grid_build on the same number of points and the same radius as the
 * handle's last synchronising build assumes that build's box (for rebuilding the SAME cloud); bit 1: sf_shot_single_scale
 * sizes its neighbour list from its last synchronising call on this cloud instead of reading the size back. Both assumptions are CHECKED ON THE DEVICE: when one
 * fails the kernels of these calls do nothing, and sf_grid_poll — to be called after synchronising the stream, before
 * the results are used — reports a non-zero status (1: a point outside the assumed box, 2: neighbour list too small)
 * and returns the handle to synchronising calls; the caller then simply repeats its calls. The calls copy nothing
 * back: sf_grid_poll reads the device-side flag itself (a synchronous 4-byte copy). */
int sf_grid_set_speculative(sf_grid* grid, int32_t mode);
int sf_grid_poll(sf_grid* grid, int32_t* status);
/* Copies perm[n] (cell-sorted position -> original index) and/or its inverse into caller buffers (NULL = skip). */
int sf_grid_permutation(const sf_grid* grid, int32_t* perm_out_dev, int32_t* inv_perm_out_dev, void* stream);
/* Copies the grid's cell-sorted arrays into caller buffers (NULL = skip): pts (n,4) float64 (xyz, original index as
 * int64 bits), nrm (n,4) float64, xyzc (n,4) float32 (cell-relative xyz, cell bits), nrm32 (n,4) float32 and
 * cell_start[ncells + 1] int32. nrm / nrm32 only for a grid built with normals. */
int sf_grid_arrays(const sf_grid* grid, double* pts_out_dev, double* nrm_out_dev, float* xyzc_out_dev,
                   float* nrm32_out_dev, int32_t* cell_start_out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * G — fixed-radius search.  Replaces `KDTree.query_radius(X, r[, return_distance=True])`
 * (shot_parallelization.py:167-169, fpfh.py:28-30). Predicate: ((dx*dx + dy*dy) + dz*dz) <= r*r in float64,
 * inclusive, the query point itself included when it belongs to the cloud — sklearn's, bit for bit.
 * queries_dev == NULL means "the cloud's own points at cell-sorted positions [self_first, self_first + nq)" (the
 * FPFH case; a sub-range is what one rank of a multi-GPU job searches); self_first is ignored otherwise.
 * ---------------------------------------------------------------------------------------------------------- */
/* Pass 1: offsets_dev[0..nq] (exclusive prefix of the neighbour counts). When total_host != NULL the total is
 * copied to the host and `stream` is synchronised. */
int sf_radius_count(sf_grid* grid, const double* queries_dev, int64_t self_first, int64_t nq, double radius,
                    int64_t* offsets_dev, int64_t* total_host, void* stream);
/* Pass 2: any of the three outputs may be NULL. nbr_sorted_dev: cell-sorted positions (what the descriptor
 * kernels consume); nbr_index_dev: original point indices (what query_radius returns, in grid-walk order);
 * dist_dev: float64 sqrt of the reduced distance (what return_distance=True returns). */
int sf_radius_fill(sf_grid* grid, const double* queries_dev, int64_t self_first, int64_t nq, double radius,
                   const int64_t* offsets_dev, int32_t* nbr_sorted_dev, int32_t* nbr_index_dev, double* dist_dev,
                   void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * G3 — support reducer.  Replaces `grid_subsampling(points, voxel_size)` (core/subsampling.py:5-39) where the SHOT
 * drivers call it on the support cloud (shot_parallelization.py:157-161, :210-214, :273-277).
 * picked_dev: int32[n] capacity; the first *count_host entries receive, in lexicographic voxel order, the index of
 * the point closest to each occupied voxel's barycentre (first on ties, members in ascending index order).
 * members_dev (optional, same capacity): the number of points of each of those voxels — what
 * `select_keypoints_with_density_threshold` thresholds (keypoint_selection.py:75-80, :109-111).
 * Synchronises `stream` (the count is a host result).
 * ---------------------------------------------------------------------------------------------------------- */
int sf_voxel_subsample(const double* xyz_dev, int64_t n, double voxel_size, int32_t* picked_dev, int32_t* members_dev,
                       int64_t* count_host, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * N — PCA normals ("next" row: upstream of the hot path).  Replaces `compute_normals`
 * (descriptors/pca_based_descriptors.py:29-59), which get_data runs on every cloud (helpers/io_ply.py:259-301).
 * ---------------------------------------------------------------------------------------------------------- */
/* k nearest neighbours, replaces `KDTree(cloud).query(queries, k, return_distance=False)` (:46). For every query
 * whose status is not 1: if at least k cloud points lie within `reach` (<= the grid's cell edge) the k nearest
 * (ORIGINAL point indices, nearest first) are written to nbr_index_dev[q*k ..] and status_dev[q] = 1; otherwise
 * status_dev[q] = 0 (too few: retry with a larger reach) or 2 (more than 512 within reach: retry with a smaller
 * one). status_dev must be zero-initialised by the caller before the first attempt. */
int sf_knn(sf_grid* grid, const double* queries_dev, int64_t nq, int32_t k, double reach, int32_t* nbr_index_dev,
           int32_t* status_dev, void* stream);
/* normal = eigenvector of the smallest eigenvalue of the neighbourhood's covariance about its barycentre
 * (`pca(...)[1][:, 0]`, :15-26, :51), LAPACK's sign; flipped when its dot product with pre_normals_dev[q] is
 * negative (:53-57; pre_normals_dev may be NULL). xyz_dev: the cloud, float64 (n,3); neighbourhoods are ORIGINAL
 * point indices, CSR (offsets_dev != NULL) or fixed_k entries per query (offsets_dev == NULL).
 * normals_dev: float64 (nq,3); NaN for an empty neighbourhood, as NumPy gives. */
int sf_pca_normals(const double* xyz_dev, int64_t nq, const int64_t* offsets_dev, int32_t fixed_k,
                   const int32_t* nbr_index_dev, const double* pre_normals_dev, double* normals_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * K — salient keypoints (no counterpart in the reference). ISS, Intrinsic Shape Signatures (Zhong 2009), as Open3D
 * defines it, with the covariance accumulated about the point; oracle/iss_oracle.py is the specification. Both calls
 * take a grid built (sf_grid_build, normals not needed) for max(salient radius, non-max radius); each radius must be
 * positive and within the grid's cell edge. Neighbourhoods use the fixed-radius predicate above.
 * ---------------------------------------------------------------------------------------------------------- */
/* saliency_dev: float64[n] per CELL-SORTED position: s_i = e3 of the covariance of the points within salient_radius
 * (about their barycentre) where that neighbourhood holds >= min_neighbors points and e2/e1 < gamma_21 and
 * e3/e2 < gamma_32 (e3 <= e2 <= e1, np.linalg.eigh's values), else 0. counts_dev (int32[n], the neighbourhood sizes)
 * and eigvals_dev (float64 (n,3), ascending) may be NULL. min_neighbors >= 1, finite gammas.
 * An empty handle (n = 0) writes nothing. No synchronisation. */
int sf_iss_saliency(sf_grid* grid, double salient_radius, int32_t min_neighbors, double gamma_21, double gamma_32,
                    double* saliency_dev, int32_t* counts_dev, double* eigvals_dev, void* stream);
/* Non-maximum suppression: point i is a keypoint iff s_i > 0, at least min_neighbors points lie within
 * non_max_radius of it, and none of them has a larger saliency (ties keep both). keypoints_dev: int32[n] capacity;
 * the first *count_host entries receive the keypoints' ORIGINAL indices in ascending order. Synchronises `stream`
 * (the count is a host result); *count_host = 0 for an empty handle. */
int sf_iss_select(sf_grid* grid, const double* saliency_dev, double non_max_radius, int32_t min_neighbors,
                  int32_t* keypoints_dev, int64_t* count_host, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * O — consistent normal orientation (no counterpart in the reference). Hoppe et al. 1992: signs propagated along the
 * minimum spanning forest of the k-NN graph; oracle/orientation_oracle.py is the specification. Every entry j != i of
 * point i's list is an undirected edge {i, j} (found from both ends, it is one edge) with
 * d = (n_i.x*n_j.x + n_i.y*n_j.y) + n_i.z*n_j.z (float64, no FMA), weight 1 - |d|, flip bit d < 0, and the unique key
 * (weight, min(i, j), max(i, j)). A point's sign relative to another point of its tree is the XOR of the flip bits on
 * the tree path between them. In each tree the member with the lowest index keeps its input sign; with towards_host
 * (3 float64, a viewpoint t) each tree instead takes the sign under which more of its members have n . (t - p) > 0
 * than < 0 (ties: the lowest-index rule).
 * ---------------------------------------------------------------------------------------------------------- */
/* xyz_dev, normals_dev: float64 (n,3); nbr_index_dev: int32 (n, k_stride) ORIGINAL point indices (the lists of
 * sf_knn with k + 1: self entries are skipped, an index outside [0, n) is an error); towards_host may be NULL.
 * out_dev: float64 (n,3), the input normals with some negated (may not alias normals_dev). *n_trees_host = number of
 * trees of the forest. Borůvka rounds with parity labels on the device; synchronises `stream` once per round and once
 * per pointer-jumping step (O(log n) rounds). */
int sf_orient_normals(const double* xyz_dev, const double* normals_dev, int64_t n, const int32_t* nbr_index_dev,
                      int32_t k_stride, const double* towards_host, double* out_dev, int64_t* n_trees_host,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * S — SHOT.
 * ---------------------------------------------------------------------------------------------------------- */
/* Local reference frames. Replaces `get_local_rf` (shot.py:16-48) fanned out by
 * `ShotMultiprocessor.compute_local_rf` (shot_parallelization.py:46-84). lrf_dev: float64 (nq,3,3), columns
 * [x y z]; identity for an empty neighbourhood. */
int sf_shot_lrf(sf_grid* grid, const double* queries_dev, int64_t nq, double radius, const int64_t* offsets_dev,
                const int32_t* nbr_sorted_dev, double* lrf_dev, void* stream);
/* Descriptors. Replaces `compute_single_shot_descriptor` (shot.py:175-306) fanned out by
 * `ShotMultiprocessor.compute_descriptor` (shot_parallelization.py:86-133), including the reference's
 * last-writer-wins binning. out_dev: (nq,352), float64 when out_is_f64 else float32. */
int sf_shot_descriptor(sf_grid* grid, const double* queries_dev, int64_t nq, double radius,
                       const int64_t* offsets_dev, const int32_t* nbr_sorted_dev, const double* lrf_dev,
                       int32_t min_neighborhood_size, int32_t normalize, void* out_dev, int32_t out_is_f64,
                       void* stream);

/* The whole single-scale driver in one call: replaces `compute_descriptor_single_scale` (shot_parallelization.py:
 * 135-183) after the grid is built — query_radius, compute_local_rf and compute_descriptor on the same neighbourhoods.
 * Same results as sf_radius_* + sf_shot_lrf + sf_shot_descriptor, but the neighbour list stays an internal (padded)
 * temporary: ONE pass over the candidate cells finds the neighbours and accumulates the frame's moments, and the sign
 * votes run inside the descriptor kernel. lrf_out_dev (nq,3,3) and pairs_host (number of neighbour pairs found) are
 * optional. Synchronises `stream` once (to size the temporary) unless the handle is in speculative mode (above). */
int sf_shot_single_scale(sf_grid* grid, const double* queries_dev, int64_t nq, double radius,
                         int32_t min_neighborhood_size, int32_t normalize, void* out_dev, int32_t out_is_f64,
                         double* lrf_out_dev, int64_t* pairs_host, void* stream);

/* Both descriptor entry points run the float32-filtered kernel first (csrc/shot.cu::shot_fast_kernel: decisions from
 * cell-relative float32 coordinates with proven margins) and hand the queries it cannot decide — more than 128
 * neighbours, a decision inside its margin, two competitors closer than float32 orders — to the float64 kernel.
 * Number of queries handed over in the last sf_shot_single_scale call that asked for `pairs_host` (measurement). */
int sf_shot_last_deferred(int64_t* deferred);

/* Measurement hook: with profiling enabled, the fused drivers (sf_shot_single_scale, sf_fpfh_cloud) record CUDA
 * events on their stream around their three stages; sf_profile_read waits for the last call and returns the
 * durations in milliseconds: search + moments, eigen-decomposition, sign votes + descriptor for SHOT;
 * search + weights, SPFH, FPFH for FPFH. */
int sf_profile_enable(int32_t enable);
int sf_profile_read(float* ms_out3);

/* ------------------------------------------------------------------------------------------------------------
 * P — FPFH.  Replaces `compute_fpfh_descriptor` (fpfh.py:16-117).
 * ---------------------------------------------------------------------------------------------------------- */
/* Stage 1 (fpfh.py:38-90): SPFH of the cloud points at cell-sorted positions [first, first + count), rows written
 * in that order to spfh_dev (count, width). offsets/nbr_sorted: the CSR of sf_radius_* called with
 * queries_dev == NULL on the same range. edges_host: float64 (3, n_bins + 1) histogram edges
 * (np.linspace(lo, hi, n_bins + 1) for alpha, phi, theta). width = 3*n_bins (decorrelated) or n_bins^3. */
int sf_spfh(sf_grid* grid, int64_t first, int64_t count, const int64_t* offsets_dev, const int32_t* nbr_sorted_dev,
            int32_t n_bins, int32_t decorrelated, const double* edges_host, float* spfh_dev, void* stream);
/* Stage 2 (fpfh.py:97-116) on keypoints given as ORIGINAL point indices. spfh_dev: the SPFH rows of the WHOLE
 * cloud in cell-sorted order. The CSR (with its distances) is either the self-search of the whole cloud
 * (csr_by_keypoint = 0: row = cell-sorted position of the keypoint) or a search around the keypoints'
 * coordinates (csr_by_keypoint = 1: row q belongs to keypoint q). */
int sf_fpfh(sf_grid* grid, const int64_t* offsets_dev, const int32_t* nbr_sorted_dev, const double* dist_dev,
            int32_t csr_by_keypoint, const float* spfh_dev, int32_t width, const int64_t* keypoint_index_dev,
            int64_t nq, void* out_dev, int32_t out_is_f64, void* stream);

/* The fused driver of one cloud, what `compute_fpfh_descriptor` does between its KDTree and its return
 * (fpfh.py:26-117): search around EVERY cloud point, SPFH of every point, FPFH of the keypoints (original point
 * indices). The neighbour list is an internal, padded temporary written by ONE pass over the candidate cells,
 * together with the float32 weights 1/d of fpfh.py:112-114. edges_host as for sf_spfh. pairs_host (optional):
 * number of neighbour pairs found (the "mean neighbourhood size" the reference logs). Synchronises `stream` once. */
int sf_fpfh_cloud(sf_grid* grid, double radius, int32_t n_bins, int32_t decorrelated, const double* edges_host,
                  const int64_t* keypoint_index_dev, int64_t nq, void* out_dev, int32_t out_is_f64, int64_t* pairs_host,
                  void* stream);

/* sf_fpfh_cloud by BLOCKS of the cell-sorted cloud, for one block per GPU (north_star: "FPFH ... query-sharded at
 * 1/2/4/8 B200"; SURVEY.md 8e: SPFH by blocks, ONE all-gather of the SPFH rows, FPFH by blocks). The caller owns the
 * temporaries and does the all-gather between the second and the third call:
 *   sf_fpfh_block_begin  cand_offsets_dev[count + 1]: padded list offsets of the cell-sorted points
 *                        [first, first + count); *total_host = list capacity to allocate (synchronises `stream`)
 *   sf_fpfh_block_spfh   ONE scan of the candidate cells writes nbr_dev / weights_dev [total] (cell-sorted positions,
 *                        float32 1/d) and counts_dev[count], then the block's SPFH rows spfh_block_dev
 *                        [count x stride] floats, stride = sf_fpfh_row_stride(width) (rows padded to 16 bytes)
 *   sf_fpfh_block_rows   FPFH rows of keypoint_index_dev[nq] — original point indices whose cell-sorted position
 *                        lies in the block — from the block's lists and the SPFH rows of the WHOLE cloud
 *                        spfh_all_dev [n x stride] (cell-sorted order: the concatenation of the blocks' rows)
 * first = 0, count = n reproduces sf_fpfh_cloud bit for bit. */
int sf_fpfh_row_stride(int32_t width, int32_t* stride_out);
int sf_fpfh_block_begin(sf_grid* grid, double radius, int64_t first, int64_t count, int64_t* cand_offsets_dev,
                        int64_t* total_host, void* stream);
int sf_fpfh_block_spfh(sf_grid* grid, double radius, int32_t n_bins, int32_t decorrelated, const double* edges_host,
                       int64_t first, int64_t count, const int64_t* cand_offsets_dev, int32_t* nbr_dev,
                       float* weights_dev, int32_t* counts_dev, float* spfh_block_dev, int64_t* pairs_host, void* stream);
int sf_fpfh_block_rows(sf_grid* grid, int64_t first, int64_t count, const int64_t* cand_offsets_dev,
                       const int32_t* counts_dev, const int32_t* nbr_dev, const float* weights_dev,
                       const float* spfh_all_dev, int32_t width, const int64_t* keypoint_index_dev, int64_t nq,
                       void* out_dev, int32_t out_is_f64, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * M — descriptor matching.  Replaces `cdist(...).argmin(axis=1)` in `basic_matching` (matching.py:162-169),
 * `match_descriptors` (matching.py:43-52) and the ratio test `double_matching_with_rejects` (matching.py:172-221).
 * ---------------------------------------------------------------------------------------------------------- */
/* Rows with at least one non-zero entry (matching.py:43-44): ascending row ids into rows_dev[0..count).
 * absmax_host (optional): the largest |x| of the whole array, from the same pass (the common scale of the float16
 * operands; NaN or infinity when the array holds one). Synchronises `stream`. */
int sf_nonempty_rows(const double* desc_dev, int64_t n, int32_t width, int64_t* rows_dev, int64_t* count_host,
                     double* absmax_host, void* stream);
/* Gathers rows `rows_dev` of a float64 matrix into the GEMM operand format: float16 (count, width_padded)
 * scaled by `scale`, plus the float32 squared norms of the ROUNDED rows. width_padded is a multiple of 64. */
int sf_match_pack(const double* desc_dev, int32_t width, const int64_t* rows_dev, int64_t count, double scale,
                  void* packed_dev, int32_t width_padded, float* sqnorm_dev, void* stream);
/* Shortlist: for each of the qa packed query rows, the k packed target rows with the smallest
 * |b|^2 - 2 a.b (tensor-core GEMM, float16 operands, float32 accumulation). idx_dev: int32 (qa,k) positions in
 * the packed target set plus `b_index_offset`; score_dev: float32 (qa,k), ascending. k <= 16.
 * use_tensor_cores = 0 selects the plain CUDA-core kernel (used to cross-check the tcgen05 kernel). */
int sf_match_topk(const void* a_packed_dev, int64_t qa, const void* b_packed_dev, const float* b_sqnorm_dev,
                  int64_t qb, int32_t width_padded, int32_t k, int32_t b_index_offset, float* score_dev,
                  int32_t* idx_dev, int32_t use_tensor_cores, void* stream);
/* k-way merge of `parts` shortlists laid out (parts, qa, k) into (qa, k) (the step after the all-gather when the
 * target set is sharded across GPUs). */
int sf_topk_merge(const float* score_dev, const int32_t* idx_dev, int32_t parts, int64_t qa, int32_t k,
                  float* score_out_dev, int32_t* idx_out_dev, void* stream);
/* Merge of the EXACT per-shard results of a target set sharded across GPUs (shot_fpfh_b200/distributed.py; replaces
 * matching.py:164-169's argmin over the whole set): packed_dev (parts, q, 3) float64 = (d1, global index of the
 * nearest target, d2) per shard in ascending order of target indices -> nearest (lowest index on ties), d1, and the
 * second smallest distance over all shards. */
int sf_nearest_merge(const double* packed_dev, int32_t parts, int64_t q, int64_t* nn_dev, double* d1_dev,
                     double* d2_dev, void* stream);
/* Certificate of the float16 shortlist (csrc/match.cu::certify_kernel): flags_dev[q] = 1 when the exact nearest
 * (want_second: second-nearest) distance of query q from sf_match_rerank is NOT provably below the distance to every
 * target outside its k-entry shortlist — bound from the k-th shortlist score, the float16 rounding of the operands and
 * the float32 accumulation. score_dev: (qa, k) of sf_match_topk; a_sqnorm_dev: squared norms of the packed query rows
 * (sf_match_pack); b_norm_max: largest norm of a packed target row; scale: the packing scale.
 * Replaces nothing in the reference: it is what makes `cdist(...).argmin()` (matching.py:164-168) provable here. */
int sf_match_certify(const float* score_dev, int32_t k, const float* a_sqnorm_dev, const double* d1_dev,
                     const double* d2_dev, int64_t qa, double scale, double b_norm_max, int32_t width, int64_t qb,
                     int32_t want_second, uint8_t* flags_dev, void* stream);
/* The exhaustive redo of all flagged queries in ONE pass over the targets: limit_dev[i] = an upper bound on the wanted
 * distance of flagged query which_dev[i] (its exact nearest / second-nearest distance from the re-rank); every target at
 * most that far is listed — the pass runs in float32 on the rows multiplied by `scale` (a power of two that brings every
 * |entry| below 1: sf_match_pack's) with a proven slack, norm_bound = an upper bound on |a| + |b| over the SCALED rows,
 * so it may list a few more — and the list goes to cand16_dev (n_which, 16), -1 padded, for sf_match_rerank,
 * which decides in float64. cand16_dev[i][0] = -2 marks a query with more than 16 listed targets: those take
 * sf_match_exhaustive_topk. */
int sf_match_exhaustive(const double* a_dev, const int64_t* rows_a_dev, const int64_t* which_dev, int64_t n_which,
                        const double* limit_dev, const double* b_dev, const int64_t* rows_b_dev, int64_t qb, int32_t width,
                        double scale, double norm_bound, int32_t* cand16_dev, void* stream);
/* Exhaustive float64 shortlist of the flagged queries which_dev[0..n_which) (positions in rows_a): the k (8 or 16)
 * nearest targets by float64 distance, lowest index on ties, written into their rows of cand_dev (qa, k); the caller
 * re-ranks those rows with sf_match_rerank. */
int sf_match_exhaustive_topk(const double* a_dev, const int64_t* rows_a_dev, const int64_t* which_dev, int64_t n_which,
                             const double* b_dev, const int64_t* rows_b_dev, int64_t qb, int32_t width, int32_t k,
                             int32_t* cand_dev, void* stream);
/* Exact re-rank: float64 `sqrt(sum((a-b)^2))` accumulated sequentially (what scipy's cdist computes) between each
 * query row and its k candidates; nn_dev = candidate with the smallest distance (lowest index on ties),
 * d1_dev / d2_dev = smallest and second smallest distance (d2 = +inf when k == 1 or a single candidate).
 * rows_a/rows_b map packed positions to rows of the float64 matrices. nn_dev holds PACKED positions of b. */
int sf_match_rerank(const double* a_desc_dev, const int64_t* rows_a_dev, int64_t qa, const double* b_desc_dev,
                    const int64_t* rows_b_dev, int32_t width, const int32_t* cand_idx_dev, int32_t k,
                    int32_t* nn_dev, double* d1_dev, double* d2_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Registration stages downstream of the matcher (SURVEY.md 8f row 4): their data-parallel part.
 * ---------------------------------------------------------------------------------------------------------- */
/* RANSAC (`ransac_on_matches`, matching/ransac.py:55-62): for each of the n_draws candidate transforms
 * (transforms_dev: (n_draws, 12) = rotation row-major then translation) the number of matches i with
 * || R a_i + t - b_i || <= threshold; a_dev / b_dev: the matched scan / reference keypoints, float64 (m,3). */
int sf_ransac_count_inliers(const double* a_dev, const double* b_dev, int64_t m, const double* transforms_dev,
                            int64_t n_draws, double threshold, int32_t* counts_dev, void* stream);
/* Adaptive RANSAC on the m matches (a_dev, b_dev: matched scan / reference keypoints, float64 (m,3), 3 <= m < 2^32);
 * oracle/adaptive_ransac_oracle.py is the specification. Draw d picks three distinct matches from splitmix64 of
 * seed * 0x9E3779B97F4A7C15 + 3d + s; a draw survives when every edge length of the triple agrees between the two
 * clouds within edge_similarity (in (0, 1]), is fitted by Kabsch (eigh3 of H^T H; rejected when degenerate) and is
 * valid when its own three pairs are inliers (|| R a + t - b || <= threshold, the predicate of
 * sf_ransac_count_inliers). Draws run in batches of 2^20 (the last truncated to max_draws, in [1, 2^32 - 1]) until
 * max_draws or until k 2^20 log1p(-(c/m)^3) <= log(1 - confidence) for the best count c. The winner is the valid draw
 * with the most inliers, the lowest draw on ties. Outputs: transform_host[12] (rotation row-major, translation), its
 * draw and count (-1 and 0 if no draw was valid), the draws run, the valid draws over all batches, and
 * inlier_mask_dev (uint8[m]) = the winner's inliers. Two host synchronisations per batch; synchronises `stream`. */
int sf_ransac_adaptive(const double* a_dev, const double* b_dev, int64_t m, double threshold, double edge_similarity,
                       uint64_t seed, int64_t max_draws, double confidence, double* transform_host,
                       int64_t* best_draw_host, int64_t* best_count_host, int64_t* draws_used_host, int64_t* valid_host,
                       uint8_t* inlier_mask_dev, void* stream);
/* One batch of the above, draws [first_draw, first_draw + n_draws) with n_draws <= 2^20, with what it produces:
 * survivors_dev = the draws that pass the edge check, valid_draws_dev / transforms_dev (12 doubles each) / counts_dev =
 * the valid draws, their transforms and inlier counts (each list in no particular order; buffers of n_draws entries).
 * n_host[2] = {survivors, valid}. Synchronises `stream`. */
int sf_ransac_adaptive_batch(const double* a_dev, const double* b_dev, int64_t m, double threshold,
                             double edge_similarity, uint64_t seed, int64_t first_draw, int64_t n_draws,
                             uint32_t* survivors_dev, uint32_t* valid_draws_dev, double* transforms_dev,
                             int32_t* counts_dev, int64_t* n_host, void* stream);
/* One ICP point-to-plane iteration (`icp_point_to_plane`, icp.py:157-182 with `solver_point_to_plane`,
 * core/solvers.py:34-48) on a grid built over the REFERENCE cloud with its normals and radius >= d_max: the scan
 * points are moved by transform_host (12 doubles, as above), each one's nearest reference point is found
 * (`KDTree.query`), pairs farther than d_max are dropped, and sums_host[29] receives, over the remaining pairs
 * (p, q, n = normal of q), with g = [p x n, n] and h = (q - p).n: the 21 entries g_i g_j (i <= j, row order), the 6
 * entries g_i h, sum |(p - q).n| and the number of pairs. nearest_dev (optional, int32[n_scan]): original index of
 * the nearest reference point, -1 where none is within d_max. Synchronises `stream`. */
int sf_icp_plane_step(sf_grid* ref_grid, const double* scan_dev, int64_t n_scan, const double* transform_host,
                      double d_max, double* sums_host, int32_t* nearest_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Result transport. The reference returns dense float64 rows on the host (shot_parallelization.py:183); a SHOT row
 * is ~86 % zeros and the kernels' values are float32, so the rows cross PCIe compacted and the dense float64
 * array is rebuilt by host threads (float64(float32 x) is exact: the array equals a dense float64 copy).
 * ---------------------------------------------------------------------------------------------------------- */
/* Device: non-zero entries of dense float32 rows (n_rows, width <= 65536), row by row, ascending columns.
 * _count writes offsets_dev[0..n_rows] (exclusive prefix of the per-row counts) and the total to *total_host
 * (synchronises `stream`); _fill writes cols_dev / vals_dev [0, total). */
int sf_rows_compact_count(const float* dense_dev, int64_t n_rows, int32_t width, int64_t* offsets_dev,
                          int64_t* total_host, void* stream);
int sf_rows_compact_fill(const float* dense_dev, int64_t n_rows, int32_t width, const int64_t* offsets_dev,
                         uint16_t* cols_dev, float* vals_dev, void* stream);
/* Host (all pointers are HOST memory; a persistent pool of up to `threads` threads). sf_host_expand_rows_begin
 * starts writing the dense rows dst[r * width + c] (zeros, and vals[i] at c = cols[i] for the entries
 * i in [offsets[r], offsets[r+1]) of row r; width <= 4096) and returns at once, so that one block of rows is
 * rebuilt while the next is computed and copied; a second call first waits for the previous one. sf_host_wait blocks until
 * everything started has finished and reports a malformed input. The buffers must stay valid until then. */
int sf_host_expand_rows_begin(const int64_t* offsets_host, const uint16_t* cols_host, const float* vals_host,
                              int64_t n_rows, int32_t width, double* dst_host, int32_t threads);
/* Host helpers of the same transport: parallel copy of pageable caller memory into a page-locked staging buffer by the
 * pool (completed by sf_host_wait), and a huge-page hint for a freshly allocated result buffer. */
int sf_host_copy_begin(const void* src_host, void* dst_host, int64_t bytes, int32_t threads);
int sf_host_advise_huge(void* ptr_host, int64_t bytes);
/* dst[i] = (double)src[i] for i in [0, n) by the same pool (started, not awaited: the float32 rows of one block are
 * widened into the float64 result the reference API returns while the next block crosses PCIe; a float32 D2H copy
 * plus this costs less than copying float64). Jobs run in the order they were started; sf_host_wait awaits all. */
int sf_host_widen_begin(const float* src_host, int64_t n, double* dst_host, int32_t threads);
int sf_host_wait(void);

#ifdef __cplusplus
}
#endif
#endif /* SHOTFPFH_B200_H */
