/*
 * pcc/search.h -- C ABI of the B200-native neighbour-search engine (libpcc_search.so).
 *
 * This is the drop-in boundary for PointCloudComparator's one data-parallel hot path: the batched
 * kNN / radius queries behind pcl::search::Search<PointT> and the per-query reductions its
 * consumers apply.  Every entry point cites the reference interface it replaces
 * (file:line in adr-arroyo/PointCloudComparator; "[up]" = the un-vendored PCL 1.7 unit it calls).
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns 0 on success, < 0 on error
 *     (pcc_last_error() gives the message for the calling thread).
 *   - `mem`: PCC_HOST  = every pointer argument is host memory; the call copies in/out and
 *                        returns after the results are complete (synchronous, like PCL).
 *            PCC_DEVICE = every pointer argument is device memory on the index's GPU; work is
 *                        enqueued on `stream` (a cudaStream_t, NULL = default stream).  Calls that
 *                        return a host scalar (counts) synchronise that stream.
 *   - points are rows of `stride_bytes` bytes whose first 12 bytes are float x, y, z
 *     (pcl::PointXYZ = 16, pcl::PointXYZRGB / PointXYZI / PointNormal = 32, packed xyz = 12).
 *   - neighbour order is (fp32 squared distance, original index); d2 = ((dx*dx + dy*dy) + dz*dz)
 *     with no FMA contraction (FLANN L2_Simple [up]).
 *   - there is no CPU fallback: every call fails loudly if no CUDA device is usable.
 */
#ifndef PCC_SEARCH_H_
#define PCC_SEARCH_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCC_HOST 0
#define PCC_DEVICE 1

#define PCC_OK 0
#define PCC_ERR_INVALID (-1)
#define PCC_ERR_CUDA (-2)
#define PCC_ERR_STATE (-3)

#define PCC_MAX_K 512

typedef struct pcc_index pcc_index;

const char *pcc_last_error(void);
int pcc_version(void);
/* number of CUDA kernels this library has launched in the calling process (bench.py "gpu_launches") */
int64_t pcc_launch_count(void);

/* pcl::search::KdTree<PointT> construction (src/segmentation.cpp:120-121,169-171,232-234). */
int pcc_create(int device, pcc_index **out);
void pcc_destroy(pcc_index *idx);

/* Search::setInputCloud(cloud, indices) (src/segmentation.cpp:122; implicit in every consumer) ->
 * KdTreeFLANN::setInputCloud [up]: non-finite points are skipped, original indices are kept.
 * `indices` may be NULL (= all n points), else n_idx row numbers into pts.
 * cell_hint > 0 fixes the grid cell edge (use the radius for radius-only workloads);
 * cell_hint <= 0 chooses it from the measured occupancy for k = k_hint (<= 0 -> 16). */
int pcc_build(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const int32_t *indices, int64_t n_idx,
              float cell_hint, int k_hint, int mem, void *stream);
int64_t pcc_size(const pcc_index *idx);   /* number of indexed (finite) points */
/* grid description for logs / DESIGN.md: out[0..2] dims, out[3] cell edge, out[4] mean points per non-empty cell */
int pcc_grid_info(const pcc_index *idx, double out[5]);

/* Search::nearestKSearch, batched overload (src/segmentation.cpp:239-240 k=50, :263,271 k=100, :190 k=100;
 * src/comparator.cpp:1525-1527 k=51, :1096,1099 k=1).  q == NULL means "the indexed cloud itself"
 * (nq is then ignored, one row per INPUT point in original order; rows of skipped points are empty).
 * Rows have stride k; entries past *k_eff = min(k, pcc_size) and rows of non-finite queries hold (-1, +inf). */
int pcc_knn(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int k, int32_t *out_idx, float *out_d2,
            int *k_eff, int mem, void *stream);
/* RegionGrowingRGB::findPointNeighbours (src/segmentation.cpp:190) on every cluster of a concatenated cloud in one call.  Cluster c is
 * rows [cloud_offsets[c], cloud_offsets[c+1]) of pts; cloud_offsets (HOST, n_clouds + 1 entries, n_clouds <= 2^24) starts at 0, ends at
 * n and never decreases, empty clusters allowed; 1 <= k <= PCC_MAX_K.  Row i of out_idx / out_d2 (stride k, input order) is, bit for
 * bit, row i - cloud_offsets[c] of pcc_knn(q == NULL, k) on cluster c alone: cluster-LOCAL indices, (d2, index) order, entries past
 * min(k, finite points of c) and rows of non-finite points (-1, +inf).  k_eff (HOST, n_clouds) gets min(k, finite points) per cluster.
 * Host round trips do not depend on n_clouds.  `idx` is the workspace: after a call with n > 0 it indexes the concatenated input
 * (k_hint = k); with n = 0 it is untouched. */
int pcc_knn_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const int64_t *cloud_offsets, int64_t n_clouds, int k,
                    int32_t *out_idx, float *out_d2, int32_t *k_eff, int mem, void *stream);

/* Search::radiusSearch, batched overload (src/segmentation.cpp:126,131 r=0.05; src/comparator.cpp:631,655,666 r=0.03/0.05).
 * KdTreeFLANN::radiusSearch [up]: d2 < float(radius*radius) strictly; max_nn = 0 means unlimited, else the max_nn
 * smallest (d2, idx).  CSR in two calls: count fills offsets[nq+1] and *total; fill writes the rows
 * ((d2, idx)-sorted when `sorted`, unspecified order otherwise). */
int pcc_radius_count(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, unsigned max_nn,
                     int64_t *offsets, int64_t *total, int mem, void *stream);
int pcc_radius_fill(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, unsigned max_nn, int sorted,
                    const int64_t *offsets, int32_t *out_idx, float *out_d2, int mem, void *stream);

/* StatisticalOutlierRemoval::applyFilterIndices first pass (src/comparator.cpp:1523-1527,1537-1541) [up]:
 * out_mean[i] = float(sum_{j=1..mean_k} sqrt(double(d2_j)) / mean_k) over the (mean_k+1)-NN of query i
 * (j = 0, the query itself, is dropped); 0 for non-finite queries.  Fused: the neighbour lists never reach HBM. */
int pcc_knn_mean_dist(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int mean_k, float *out_mean,
                      int mem, void *stream);
/* second pass: mean / stddev (n-1) / threshold = mean + std_mul*stddev in double over n distances with
 * n_valid valid ones; keep[i] = distances[i] <= threshold.  stats[0..2] = mean, stddev, threshold (host). */
int pcc_sor_threshold(pcc_index *idx, const float *distances, int64_t n, int64_t n_valid, double std_mul, double stats[3],
                      uint8_t *keep, int64_t *kept, int mem, void *stream);

/* NormalEstimation::computeFeature (src/segmentation.cpp:236-240 k=50; src/comparator.cpp:628-635,764-771 r=0.03) [up]:
 * computeMeanAndCovarianceMatrix (fp32 single pass, neighbour order) -> pcl::eigen33 smallest eigenpair ->
 * flipNormalTowardsViewpoint.  out[nq*4] = nx, ny, nz, curvature; NaN when < 3 neighbours. */
int pcc_normals_knn(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int k, const float viewpoint[3], float *out,
                    int mem, void *stream);
int pcc_normals_radius(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, const float viewpoint[3],
                       float *out, int mem, void *stream);

/* IntensityGradientEstimation::computeFeature (src/comparator.cpp:649-656, r = 0.03) [up]. intensity[n_input]: one float per INPUT
 * row of the indexed cloud (original order). normals4[rows*4]: the query's (nx, ny, nz, curvature) as pcc_normals_* writes them,
 * rows = nq, or n_input when q == NULL. out[rows*4] = gx, gy, gz, 0; NaN with < 3 neighbours and for skipped (non-finite) rows.
 * Per query over its (d2, idx)-sorted radius row: fp32 centroid and mean intensity (true divisions), A = sum (p-c)(p-c)^T and
 * b = sum (p-c)(I-mean) in row order (non-finite intensities skipped), x = Eigen 3.3 colPivHouseholderQr(A).solve(b) -- rank-
 * deficient A (planar neighbourhoods) solves over the nonzero pivots only -- and gradient = (I - n n^T) x. */
int pcc_intensity_gradient(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, const float *intensity,
                           const float *normals4, float *out, int mem, void *stream);
/* RIFTEstimation::computeFeature (src/comparator.cpp:659-673, r = 0.05, 4 x 8 bins) [up]. gradient4[n_input*4] per INPUT row of the
 * indexed cloud. out[rows * nd*ng] in PCL's histogram order; NaN row without neighbours. nd*ng <= 32 (Histogram<32>), else PCC_ERR_INVALID.
 * PCL's histogram order is gradient bin outer, distance bin inner: out[row*nd*ng + g*nd + d].  The query point is both the search
 * centre and p0; each histogram is normalised to unit Frobenius norm (an all-zero one stays zero). */
int pcc_rift(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, const float *gradient4,
             int n_distance_bins, int n_gradient_bins, float *out, int mem, void *stream);
/* processRIFT (src/comparator.cpp:590-684) on every cluster of a concatenated cloud in one call: per cluster, pcc_normals_radius
 * (viewpoint 0) -> drop the rows with a non-finite normal -> pcc_intensity_gradient and pcc_rift on the remaining points -> drop the
 * rows with a non-finite bin, bit for bit as those calls on the cluster alone.  Cluster c is rows [cloud_offsets[c],
 * cloud_offsets[c+1]) of pts (rows of stride_bytes with x, y, z first); intensity[n] is one float per row (rgbToIntensity).
 * cloud_offsets (HOST, n_clouds + 1 entries, n_clouds <= 2^24) starts at 0, ends at n and never decreases, empty clusters allowed;
 * radii finite and >= 0, 1 <= nd*ng <= 32.  out_desc gets the surviving descriptors (nd*ng floats each, PCL's bin order) in
 * (cluster, row) order and out_rows their cluster-LOCAL row numbers, at most `cap` rows; desc_offsets (HOST, n_clouds + 1) always
 * gets the full layout, desc_offsets[n_clouds] = total (cap = 0 only counts).  Host round trips do not depend on n_clouds.
 * `idx` is the workspace: after a call with n > 0 it indexes the concatenated input (cell max(radii)); with n = 0 it is untouched. */
int pcc_rift_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const float *intensity, const int64_t *cloud_offsets,
                     int64_t n_clouds, double normal_radius, double gradient_radius, double rift_radius, int n_distance_bins, int n_gradient_bins,
                     float *out_desc, int32_t *out_rows, int64_t cap, int64_t *desc_offsets, int mem, void *stream);

/* SIFTKeypoint<PointXYZRGB, PointWithScale> (src/comparator.cpp:449-465: min_scale 0.005, 5 octaves, 5 scales per octave,
 * min_contrast 0.001) [up].  DESIGN.md section 2 records the reading of PCL's sift_keypoint.hpp these restate.
 *
 * computeScaleSpace over the indexed cloud itself: values[n_input] = one field value per INPUT row (SIFTKeypointFieldSelector);
 * scales[n_scales] (HOST array in either memory mode, positive and ascending, 2 <= n_scales <= 16) is one octave's scale table.
 * sigma^2 = powf(scale, 2.0f) and the cutoff 9 sigma^2 are formed on the host; each point's (d2, idx)-sorted radius row at
 * max_radius = 3.0f * scales[n_scales-1] is walked once: scale s sums w = expf((-0.5f d2) / sigma_s^2) over the neighbours with
 * d2 <= 9 sigma_s^2, response_s = sum(value w) / sum(w).  out[n_input * (n_scales-1)] row-major, dog[:, s-1] = response_s -
 * response_{s-1}; rows of skipped (non-finite) inputs are NaN.  expf is the fp64-evaluated restatement of pcc_device.cuh
 * (sift_expf), which may differ from a libm expf by one ulp. */
int pcc_sift_dog(pcc_index *idx, const float *values, const float *scales, int n_scales, float *out, int mem, void *stream);
/* findScaleSpaceExtrema: dog[n_input * n_cols] row-major over the indexed cloud (1 <= n_cols <= 15).  Per point the min and max of
 * every column over its min(25, pcc_size) nearest points (pcc_knn, q == NULL; ties by (d2, index)); the point is a keypoint at
 * column c in 1..n_cols-2 when |v| >= min_contrast and (v == min[c] && v < min[c-1] && v < min[c+1]) or else (v == max[c] &&
 * v > max[c-1] && v > max[c+1]).  (out_row, out_col) in (row, column) order; *n_found is always the full count, at most `cap`
 * entries are written. */
int pcc_sift_extrema(pcc_index *idx, const float *dog, int n_cols, float min_contrast, int32_t *out_row, int32_t *out_col, int64_t cap,
                     int64_t *n_found, int mem, void *stream);
/* detectKeypoints: the octave loop over pts[n] (rows of stride_bytes >= 16 with x, y, z first and the packed 0x00RRGGBB colour word at
 * rgb_offset_bytes -- pcl::PointXYZRGB: stride 32, offset 16).  scale = min_scale; per octave: VoxelGrid(leaf = scale, rgb averaged)
 * of the previous octave's cloud (the input for the first), stop below 25 points, index the result, scales[i] = scale *
 * powf(2.0f, (1.0f * i - 1.0f) / nr_scales_per_octave) for i < nr_scales_per_octave + 3, pcc_sift_dog on the field values
 * float(299 r + 587 g + 114 b) / 1000.0f, pcc_sift_extrema, then scale *= 2.  out4 rows = (x, y, z, scales[column]) in (octave,
 * point, column) order; *n_keypoints is the full count, at most `cap` rows are written.  nr_scales_per_octave <= 13.
 * `idx` is the workspace: the call rebuilds it per octave and leaves it indexing the last octave's grid. */
int pcc_sift_keypoints(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, float min_scale, int nr_octaves,
                       int nr_scales_per_octave, float min_contrast, float *out4, int64_t cap, int64_t *n_keypoints, int mem, void *stream);
/* pcc_sift_keypoints, then pcc_first_within, on every cluster of a concatenated cloud in one call (processRIFTwithSIFT's per-cluster
 * processSift + snap, src/comparator.cpp:435-469, 696-713).  Cluster c is rows [cloud_offsets[c], cloud_offsets[c+1]) of pts (row
 * layout as pcc_sift_keypoints); cloud_offsets (HOST, n_clouds + 1 entries) starts at 0, ends at n and never decreases, empty clusters
 * allowed.  out4 gets every cluster's pcc_sift_keypoints rows, bit for bit, concatenated in cluster order -- (cluster, octave, point,
 * column) order, at most `cap` rows; kp_offsets (HOST, n_clouds + 1) always gets the full layout, kp_offsets[n_clouds] = total.
 * snap (may be NULL) gets one int32 per written row: the cluster-LOCAL row of the lowest-index point of the keypoint's own cluster
 * with sqrt(double d^2) < snap_threshold, or -1.  The octave loop runs once for the batch; a cluster leaves it at the first octave
 * whose VoxelGrid result has fewer than 25 points.  Host round trips depend on the octave count, not on n_clouds (<= 2^24).
 * `idx` is the workspace: after the call it indexes the concatenated input (cell snap_threshold) when snap is non-NULL and a row was
 * written, else the union of the clusters' last octave clouds. */
int pcc_sift_keypoints_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, const int64_t *cloud_offsets,
                               int64_t n_clouds, float min_scale, int nr_octaves, int nr_scales_per_octave, float min_contrast, double snap_threshold,
                               float *out4, int32_t *snap, int64_t cap, int64_t *kp_offsets, int mem, void *stream);

/* CorrespondenceEstimation::determineCorrespondences + the sums TransformationEstimationSVD needs
 * (src/comparator.cpp:1091-1096) [up].  Each source point is first moved by the row-major 4x4 `T_apply`
 * (IterativeClosestPoint::transformCloud arithmetic; NULL = identity) IN PLACE when `src_inout` is device
 * memory, then matched to its nearest indexed (target) point.  sums[16] (host, double): 0-2 sum src, 3-5 sum tgt,
 * 6-14 sum tgt_a*src_b row-major, 15 sum d2; *count = correspondences.  corr_idx / corr_d2 may be NULL. */
int pcc_icp_step(pcc_index *idx, void *src_inout, int64_t ns, int stride_bytes, const float *T_apply, double sums[16],
                 int64_t *count, int32_t *corr_idx, float *corr_d2, int mem, void *stream);
/* IterativeClosestPoint::align + hasConverged + getFitnessScore as configured at src/comparator.cpp:1089-1110
 * (max_iter iterations, transformation epsilon 0, no rejectors).  src is host or device per `mem`; T16 row-major. */
int pcc_icp_align(pcc_index *idx, const void *src, int64_t ns, int stride_bytes, int max_iter, float T16[16], int *converged,
                  double *fitness, int *iterations, int mem, void *stream);
/* Umeyama (no scaling) from the 16 sums of pcc_icp_step; host-only O(1) helper used by pcc_icp_align. */
int pcc_umeyama_from_sums(const double sums[16], int64_t count, float T16[16]);

/* EuclideanClusterExtraction::extract over the indexed cloud (src/segmentation.cpp:125-131) [up]:
 * connected components of {d2 < float(tol*tol)}, kept when min_size <= size <= max_size, ordered by size
 * descending (ties: smallest member index).  labels[n_input] = cluster rank or -1; sizes[<= sizes_cap]. */
int pcc_euclidean_labels(pcc_index *idx, double tolerance, int64_t min_size, int64_t max_size, int32_t *labels,
                         int64_t *n_clusters, int64_t *sizes, int64_t sizes_cap, int mem, void *stream);

/* Sharded clustering for query-sharded multi-GPU runs (SURVEY.md section 8e).  Forests are uint32[pcc_size] arrays over
 * SORTED positions in device memory (the grid is replicated, so positions mean the same on every rank):
 *   pcc_ece_init        parent[i] = i
 *   pcc_ece_link_range  hook the radius-graph edges whose query endpoint is in [begin, end) (this rank's shard)
 *   pcc_ece_absorb      unite i with other[i] for every i (other = the element-wise MIN all-reduce of the ranks' compressed
 *                       forests), then compress so parent[i] = root = smallest member; repeat until the all-reduce is a fix-point
 *   pcc_ece_finish      sizes, size filter, PCL ordering, labels[n_input] in ORIGINAL row order (device pointers) */
int pcc_ece_init(pcc_index *idx, uint32_t *parent, void *stream);
int pcc_ece_link_range(pcc_index *idx, double tolerance, int64_t begin, int64_t end, uint32_t *parent, void *stream);
int pcc_ece_absorb(pcc_index *idx, const uint32_t *other, uint32_t *parent, void *stream);
int pcc_ece_finish(pcc_index *idx, uint32_t *parent, int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters, int64_t *sizes,
                   int64_t sizes_cap, void *stream);

/* SIFT keypoint -> first cloud point within `thr` in index order (src/comparator.cpp:696-713):
 * out[i] = lowest original index with sqrt(double(dx)^2+double(dy)^2+double(dz)^2) < thr, or -1. */
int pcc_first_within(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double thr, int32_t *out, int mem, void *stream);

/* pcl::VoxelGrid<PointT>::applyFilter [up] as the reference calls it before every segmentation search
 * (src/segmentation.cpp:69-74, 223-228; leaf 0.025): one centroid per occupied voxel, output ordered by voxel index
 * (x fastest), downsample_all_data semantics for PointXYZRGB (x, y, z averaged in fp32; r, g, b averaged and truncated,
 * packed at rgb_offset_bytes, -1 = no colour field).  `out` has room for n rows of stride_bytes; *n_out rows are written.
 * `idx` only provides the device and scratch buffers (it does not need to be built).  Points of a voxel are summed in
 * ascending row order (PCL's std::sort leaves that order unspecified). */
int pcc_voxel_grid(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, const float leaf[3],
                   int min_points_per_voxel, void *out, int64_t *n_out, int mem, void *stream);

/* RegionGrowing::extract minus findPointNeighbours (src/segmentation.cpp:249-271) [up]: the sequential smooth-region grow over
 * the N x k neighbour table built by pcc_knn(q == NULL) and the normals of pcc_normals_knn (rows nx, ny, nz, curvature).
 * HOST pointers only (the algorithm is order-dependent and runs on the host).  labels[i] = cluster number in creation
 * order among the clusters with min_size <= size <= max_size, or -1. */
int pcc_region_growing(const int32_t *neighbours, int64_t n, int k, const float *normals4, float smoothness_rad, float curvature_threshold,
                       int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters);

/* RegionGrowingRGB::extract minus findPointNeighbours (color_growing_segmentation, src/segmentation.cpp:161-216, run on both clouds of
 * every matched cluster pair at src/comparator.cpp:1457-1460, which then compares the cluster COUNTS) [up]: colour grow over the
 * N x k table of pcc_knn(q == NULL, k = 100) and its squared distances, segment neighbours, merge by mean colour, fold small regions,
 * size filter.  HOST pointers (sequential, order-dependent).  rgba = one packed 0x00RRGGBB word per point (PCL's PointXYZRGB::rgba),
 * rgba_stride_bytes apart.  Reference configuration: distance 10, point colour 6, region colour 5, min size 200, max INT_MAX;
 * grow_neighbours = 30 (RegionGrowing::neighbour_number_, which the reference never sets: growRegion only walks the first 30 of
 * the 100 neighbours).  labels[i] = cluster number in PCL's order, or -1. */
int pcc_region_growing_rgb(const int32_t *neighbours, const float *sqr_distances, int64_t n, int k, const uint32_t *rgba, int rgba_stride_bytes,
                           float distance_threshold, float point_color_threshold, float region_color_threshold, int grow_neighbours,
                           int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters);
/* color_growing_segmentation on every cluster of a concatenated cloud in one call: pcc_knn_batched, then pcc_region_growing_rgb on each
 * cluster's slice of the table (stride k, cluster-LOCAL indices), one cluster after another on the host.  pts and cloud_offsets as
 * pcc_knn_batched; the packed 0x00RRGGBB colour word sits at rgb_offset_bytes of every row (pcl::PointXYZRGB: stride 32, offset 16).
 * labels (HOST, n) gets each point's cluster-LOCAL label in PCL's order, or -1; n_clusters (HOST, n_clouds) each cluster's count -- for
 * every cluster what pcc_knn(q == NULL, k) + pcc_region_growing_rgb give on that cluster alone.  The reference only segments a cloud of
 * more than 10 points (src/segmentation.cpp:167); that test stays with the caller.  `idx` as pcc_knn_batched. */
int pcc_region_growing_rgb_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, const int64_t *cloud_offsets,
                                   int64_t n_clouds, int k, float distance_threshold, float point_color_threshold, float region_color_threshold,
                                   int grow_neighbours, int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters, int mem, void *stream);

/* matchRIFTFeaturesKnn (src/comparator.cpp:560-588): KdTreeFLANN<Histogram<32>> over `ref`, nearestKSearch(k = 1) for every row
 * of `qry` [up].  Exact brute force in descriptor space: d2 accumulated sequentially over the first `dim` floats of a row (fp32, no
 * FMA), ties to the lowest index, reference rows that are non-finite in those floats skipped, such queries get (-1, +inf).  The
 * caller applies the reference's acceptance test (d2 < 0.05f).  Rows are stride_floats floats apart (32 for RIFT32).
 * dim = 3 is REFERENCE-EXACT: the reference neither registers Histogram<32> nor sets a point representation, so PCL 1.7's
 * DefaultPointRepresentation clamps the tree to the first 3 floats [up]; dim = 32 compares all bins (what the author intended). */
int pcc_descriptor_nn(pcc_index *workspace, const float *ref, int64_t n_ref, const float *qry, int64_t n_qry, int dim, int stride_floats,
                      int32_t *out_idx, float *out_d2, int mem, void *stream);

/* Multi-GPU plumbing (query sharding with a replicated grid, SURVEY.md section 8e): the built index is four flat device
 * arrays that a host layer can broadcast with NCCL and adopt on the other ranks.
 * meta[16] (host doubles): n_indexed, n_input, nx, ny, nz, origin xyz, cell, inv_cell, mean occupancy, n_cells.
 * ptrs[2] (device): float4 sorted points [n_indexed], uint32 cell_start [n_cells+1]. */
int pcc_export(const pcc_index *idx, double meta[16], void *ptrs[2]);
int pcc_adopt(pcc_index *idx, const double meta[16], void *stream);   /* allocates; then fill via pcc_export ptrs */

/* One process per GPU (SURVEY.md section 8e): `nccl_comm` is the caller's ncclComm_t over the ranks (not owned, must outlive the
 * index; NULL detaches).  libnccl.so.2 is resolved with dlopen at this call -- the copy the process already loaded is the one
 * used, so the communicator must come from it; libpcc_search has no link-time NCCL dependency.  After this call:
 *   pcc_broadcast_index  the grid built on `root` (pcc_build) is adopted by every other rank: 16 doubles of description, then the
 *                        sorted float4 points and the cell table straight into place (ncclBroadcast over NVLink)
 *   pcc_gather           all-gather of per-shard result rows (DEVICE pointers).  Every rank passes its n_local rows of row_bytes
 *                        bytes (a multiple of 4); `out` receives all n_total rows on every rank -- in ORIGINAL row order when
 *                        `local_rows` (the original row number of each local row) is given, else concatenated in rank order
 *   pcc_icp_align        `src` is this rank's shard of the source cloud; the 16 sums + count of every pass are all-reduced
 *                        (17 doubles, ncclAllReduce), so every rank returns the same transform, iteration count and fitness
 *   pcc_allreduce_f64    the same sum over n device doubles, for a consumer that drives pcc_icp_step itself
 * Queries shard by construction (they are independent given the replicated grid): each rank simply calls pcc_knn / pcc_radius_* /
 * pcc_normals_* / pcc_knn_mean_dist on its own rows; Euclidean clustering shards through pcc_ece_* below. */
int pcc_comm_init(pcc_index *idx, void *nccl_comm, int rank, int world);
int pcc_comm_info(const pcc_index *idx, int *rank, int *world);
int pcc_broadcast_index(pcc_index *idx, int root, void *stream);
int pcc_gather(pcc_index *idx, const void *local, int64_t n_local, int row_bytes, const int32_t *local_rows, void *out, int64_t n_total, void *stream);
int pcc_allreduce_f64(pcc_index *idx, double *device_buf, int n, void *stream);

/* time of the last query's dominant kernel in ms (CUDA events on the launch stream), < 0 if not recorded.
 * Recording is enabled with pcc_set_timing(idx, 1) and adds two events per call. */
int pcc_set_timing(pcc_index *idx, int enable);
double pcc_last_kernel_ms(const pcc_index *idx);

#ifdef __cplusplus
}
#endif
#endif /* PCC_SEARCH_H_ */
