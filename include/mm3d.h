/* mm3d.h — C ABI of libmm3d.so, the B200-native registration hot path of map_merge_3d.
 *
 * The reference (hrnr/map-merge, package map_merge_3d) has no FFI or plugin layer:
 * its drop-in boundary is the static library `map_merging`
 * (map_merge_3d/CMakeLists.txt:67-74) and the three public headers under
 * map_merge_3d/include/map_merge_3d/.  Each entry point below names the reference
 * function it stands in for (file:line under /root/reference/map_merge_3d).  The
 * C++ shim in include/map_merge_3d/ re-creates the reference signatures on top of
 * this ABI; INTEGRATION.md shows how a maintainer would bind it.
 *
 * Conventions
 *   points      float[n][4]  = x, y, z, rgba bits (pcl::PointXYZRGB::rgba = a<<24|r<<16|g<<8|b)
 *   normals     float[n][4]  = nx, ny, nz, curvature (pcl::Normal)
 *   descriptors float[k][dim]
 *   transforms  float[16] COLUMN-major, i.e. Eigen::Matrix4f::data()
 *   status      0 = ok, <0 = error (text from mm3d_last_error), >0 = in-band result documented per call
 *   outputs returned through T** are allocated by the library; release with mm3d_free.
 *   All pointers are HOST pointers unless a name ends in _dev.
 * There is no CPU fallback: every call fails with MM3D_ERR_CUDA when no sm_100-class
 * device is usable.
 */
#ifndef MM3D_H_
#define MM3D_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mm3d_ctx mm3d_ctx;
typedef struct mm3d_maps mm3d_maps;         /* raw clouds resident in HBM */
typedef struct mm3d_features mm3d_features; /* per-map registration inputs resident in HBM */

enum { MM3D_OK = 0, MM3D_ERR = -1, MM3D_ERR_CUDA = -2, MM3D_ERR_ARG = -3, MM3D_ERR_UNSUPPORTED = -4 };

/* enum values follow the reference's declaration order
 * (features.h:20-24 Descriptor, features.h:49 Keypoint, matching.h:103 EstimationMethod) */
enum { MM3D_DESC_PFH = 0, MM3D_DESC_PFHRGB = 1, MM3D_DESC_FPFH = 2, MM3D_DESC_RSD = 3, MM3D_DESC_SHOT = 4, MM3D_DESC_SC3D = 5 };
enum { MM3D_KP_SIFT = 0, MM3D_KP_HARRIS = 1 };
enum { MM3D_EST_MATCHING = 0, MM3D_EST_SAC_IA = 1 };

/* MapMergingParams (include/map_merge_3d/map_merging.h:28-44), all 16 fields already resolved. */
typedef struct mm3d_params {
  double resolution;
  double descriptor_radius;
  int32_t outliers_min_neighbours;
  double normal_radius;
  int32_t keypoint_type;
  double keypoint_threshold;
  int32_t descriptor_type;
  int32_t estimation_method;
  int32_t refine_transform;
  double inlier_threshold;
  double max_correspondence_distance;
  int32_t max_iterations;
  uint64_t matching_k;
  double transform_epsilon;
  double confidence_threshold;
  double output_resolution;
} mm3d_params;

/* Defaults of MapMergingParams (map_merging.h:29-44): dependent values frozen at resolution 0.1. */
void mm3d_params_default(mm3d_params* p);

/* cuda_stream: a cudaStream_t to run on (e.g. the caller's current stream), or NULL for a private one. */
int mm3d_create(mm3d_ctx** ctx, int device, void* cuda_stream);
void mm3d_destroy(mm3d_ctx* ctx);
const char* mm3d_last_error(mm3d_ctx* ctx);
void mm3d_free(void* p);
/* Per-kernel device timing: between begin and end every kernel launch is bracketed by a CUDA event pair on the
 * launching stream.  *json (mm3d_free) = [{"kernel", "launches", "ms", "algorithmic_bytes", "ms_annotated"}, ...]. */
int mm3d_profile_begin(mm3d_ctx* ctx);
int mm3d_profile_end(mm3d_ctx* ctx, char** json);
/* Tensor-core k-NN bookkeeping since the context was created: out[0] = query rows processed, out[1] = early
 * flushes (a row's candidate list filled up with ties and was evaluated exactly before the last tile), out[2] = columns that
 * went through the exact FP32 distance. */
int mm3d_knn_stats(mm3d_ctx* ctx, uint64_t* out);
/* kernels launched through this context so far */
long long mm3d_kernel_launches(mm3d_ctx* ctx);

/* ---- high-level interface ------------------------------------------------ */

/* estimateMapsTransforms (src/map_merging.cpp:188-275).  out_transforms has room for n_maps
 * matrices; *n_out = number written (0 for no maps, 1 = identity for one map, else
 * numberOfNodesInEstimates, src/graph.cpp:7-15).  A NULL cloud pointer is an empty cloud. */
int mm3d_estimate_maps_transforms(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, const mm3d_params* params,
                                  float* out_transforms, int* n_out);

/* composeMaps (src/map_merging.cpp:277-305).  Returns 1 with *out = NULL for empty input (the
 * reference returns nullptr), MM3D_ERR_ARG when n_maps != n_transforms (the reference throws). */
int mm3d_compose_maps(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, int n_transforms,
                      const float* transforms, double resolution, float** out, uint64_t* n_out);

/* ---- the high-level calls on points in the caller's own record layout ------------------------------------------------
 * The records are converted to (and for outputs from) the packed layout on the GPU, so a caller that holds, for example,
 * a std::vector<pcl::PointXYZRGB> hands it over as it is.  Input in the packed layout {16, 0, 4, 8, 12, NULL} is copied
 * straight from the caller's buffer; any other layout goes through pinned staging slots of the context (host threads copy
 * the records in, the device converts them).  Fields move as 32-bit words, so NaN payloads, infinities and -0.0 arrive
 * bit for bit. */

/* Where the fields of one point sit in a caller's array of records.  All offsets and point_step are byte counts and
 * multiples of 4; each field is 4 bytes (float32 x, y, z; the 32-bit rgba word) and lies inside the record. */
typedef struct mm3d_layout {
  uint32_t point_step;                 /* bytes from one point to the next (16 = the packed layout, 32 = pcl::PointXYZRGB) */
  int32_t offset_x, offset_y, offset_z, offset_rgba;
  const void* record_template;         /* outputs only: point_step bytes that every output record starts from; NULL = zeros */
} mm3d_layout;
/* A layout is malformed (MM3D_ERR_ARG, nothing launched) when it is NULL, point_step < 16, point_step > MM3D_LAYOUT_MAX_STEP
 * or not a multiple of 4, or an offset is negative, not a multiple of 4 or puts its field past the end of the record. */
#define MM3D_LAYOUT_MAX_STEP 65536

/* mm3d_estimate_maps_transforms on records in `layout` */
int mm3d_estimate_maps_transforms_layout(mm3d_ctx* ctx, int n_maps, const void* const* clouds, const uint64_t* n_points,
                                         const mm3d_layout* layout, const mm3d_params* params, float* out_transforms, int* n_out);
/* mm3d_compose_maps on records in `in_layout`; *out = n_out records in `out_layout` (mm3d_free) */
int mm3d_compose_maps_layout(mm3d_ctx* ctx, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout* in_layout,
                             int n_transforms, const float* transforms, double resolution, const mm3d_layout* out_layout, void** out,
                             uint64_t* n_out);
/* mm3d_maps_upload on records in `layout` */
int mm3d_maps_upload_layout(mm3d_ctx* ctx, int n_maps, const void* const* clouds, const uint64_t* n_points, const mm3d_layout* layout,
                            mm3d_maps** maps);

/* ---- map set: resident maps that re-estimate only what changed (csrc/mapset.cu) ---------------------------------------
 * An ordered list of slots, one per robot.  Each slot keeps its raw cloud on the device, the features computed from it and,
 * for every pair, the last registration result.  It serves the reference's ROS node pattern (map_merge_node): each map
 * callback replaces one slot, and the estimation and compositing timers run over all slots.
 *
 * Contract: after any sequence of updates and parameter changes, mm3d_mapset_estimate returns bit for bit what
 * mm3d_estimate_maps_transforms returns on the slots' current clouds in slot order (n_out, empty slots and SAC_IA
 * included), and mm3d_mapset_compose returns bit for bit what mm3d_compose_maps_layout returns.  Caching skips work; it
 * never changes a result.
 *   - A map's features are recomputed when its cloud changed (bitwise, after conversion to the packed layout).
 *   - A pair is registered again when either of its maps changed.  Under MM3D_EST_SAC_IA it is also registered again
 *     when the offset at which its draws start in the C rand() stream moved, because an earlier source map's keypoints
 *     changed.
 *   - Any field of mm3d_params that differs from the previous estimate recomputes everything.
 *   - Cached state is committed only when a call succeeds; after an error the next estimate redoes what was pending.
 * A malformed layout, a negative or repeated slot index, a NULL pointer where one is required, or a ctx other than the
 * one the set was created on returns MM3D_ERR_ARG, launches nothing and leaves the set unchanged.
 * A set is used by one thread at a time, like a context, and is freed before its context.  On an mm3d_create_multi context
 * it runs on the first device. */
typedef struct mm3d_mapset mm3d_mapset;
/* a set with no slots */
int mm3d_mapset_create(mm3d_ctx* ctx, mm3d_mapset** set);
/* Replace the clouds of n slots (records in `layout`; a NULL cloud or 0 points is an empty cloud).  A slot index at or past
 * the current count grows the set; slots in between are empty.  changed (optional, n ints): 1 when the slot's cloud differs
 * from the resident one, bit for bit after conversion to the packed layout, or the call created the slot.  An unchanged
 * slot keeps its resident cloud and everything computed from it. */
int mm3d_mapset_update(mm3d_ctx* ctx, mm3d_mapset* set, int n, const int32_t* slots, const void* const* clouds, const uint64_t* n_points,
                       const mm3d_layout* layout, int32_t* changed);
/* number of slots (0 for NULL) */
int mm3d_mapset_size(const mm3d_mapset* set);
/* mm3d_estimate_maps_transforms over the slots; out_transforms has room for mm3d_mapset_size matrices.
 * work (optional, 3 ints): maps whose features were computed, pairs registered, pairs reused.  With nothing changed since
 * the previous estimate and the same params, no kernel is launched. */
int mm3d_mapset_estimate(mm3d_ctx* ctx, mm3d_mapset* set, const mm3d_params* params, float* out_transforms, int* n_out, int32_t* work);
/* mm3d_compose_maps_layout over the slots' resident clouds: 1 with *out = NULL when the set has no slots, MM3D_ERR_ARG when
 * n_transforms differs from the slot count; *out = n_out records in out_layout (mm3d_free). */
int mm3d_mapset_compose(mm3d_ctx* ctx, const mm3d_mapset* set, int n_transforms, const float* transforms, double resolution,
                        const mm3d_layout* out_layout, void** out, uint64_t* n_out);
void mm3d_mapset_free(mm3d_mapset* set);

/* ---- low-level interface (features.h / matching.h) ------------------------ */
/* index_leaf: voxel size the cloud was built with (MapMergingParams::resolution); 0 picks
 * radius / 8 (descriptor-style radii) or radius / 6 (normal-style radii), the reference's
 * default ratios.  It only affects speed and the float summation order, never the result set. */

/* downSample (src/features.cpp:17-27) */
int mm3d_downsample(mm3d_ctx* ctx, const float* pts, uint64_t n, double resolution, float** out, uint64_t* n_out);
/* removeOutliers (src/features.cpp:31-43); counts (optional, n ints) = neighbours found per input point */
int mm3d_remove_outliers(mm3d_ctx* ctx, const float* pts, uint64_t n, double radius, int min_neighbours, double index_leaf, float** out,
                         uint64_t* n_out, int32_t* counts);
/* computeSurfaceNormals (src/features.cpp:168-179) */
int mm3d_normals(mm3d_ctx* ctx, const float* pts, uint64_t n, double radius, double index_leaf, float** normals);
/* detectKeypoints (src/features.cpp:85-96); dog0 (optional) receives octave-0 DoG values, n0 x 5 */
int mm3d_keypoints(mm3d_ctx* ctx, const float* pts, uint64_t n, const float* normals, int type, double threshold, double radius,
                   double resolution, float** keypoints, uint64_t* n_keypoints, float** dog0, uint64_t* n_dog0);
/* computeLocalDescriptors (src/features.cpp:152-166); keypoints are filtered like the reference
 * does (features.cpp:119-141): *keypoints_out / *n_out hold the survivors.  spfh (optional) = n x 33. */
int mm3d_descriptors(mm3d_ctx* ctx, const float* pts, uint64_t n, const float* normals, const float* keypoints, uint64_t n_keypoints,
                     int type, double radius, double index_leaf, float** keypoints_out, uint64_t* n_out, float** descriptors, int* dim,
                     float** spfh);
/* findFeatureCorrespondences (src/matching.cpp:96-108): pairs = int32[nc][2] (source, target) */
int mm3d_match(mm3d_ctx* ctx, const float* desc_src, uint64_t n_src, const float* desc_tgt, uint64_t n_tgt, int dim, uint64_t k,
               int32_t** pairs, float** distances, uint64_t* n_corr);
/* the k-nearest-neighbour search inside findFeatureCorrespondences (src/matching.cpp:45-60, pcl::search::KdTree<DescriptorT>::
 * nearestKSearch under flann::L2_Simple): for every row of a, the k nearest rows of b sorted by (distance, index);
 * idx = int32[na][k], dist = float[na][k] (squared L2), k is clamped to nb; unused slots hold -1 / 0. */
int mm3d_knn(mm3d_ctx* ctx, const float* a, uint64_t na, const float* b, uint64_t nb, int dim, uint64_t k, int32_t* idx, float* dist);
/* Test hook of the tensor-core k-NN (33-dimensional descriptors, k <= 5): the same search as mm3d_knn through the tcgen05
 * filter, plus what the filter saw — acc = float[na][nb] raw accumulators (1 - ES) ||b'||^2 - 2 a'.b', the centred squared
 * norms of both sides and ES.  tests/test_full_size_gpu.py checks the filter's error bound with it on BASELINE-sized data. */
int mm3d_knn_tc_audit(mm3d_ctx* ctx, const float* a, uint64_t na, const float* b, uint64_t nb, int dim, uint64_t k, int32_t* idx, float* dist,
                      float* acc, float* norm_a, float* norm_b, float* err_store);
/* estimateTransformFromCorrespondences (src/matching.cpp:110-140); inliers = positions in pairs.
 * dbg (optional, 2 ints) = RANSAC iterations, best inlier count; dbg_d (optional) = sample distance threshold */
int mm3d_ransac(mm3d_ctx* ctx, const float* kp_src, uint64_t n_src, const float* kp_tgt, uint64_t n_tgt, const int32_t* pairs,
                uint64_t n_corr, double inlier_threshold, float* transform, int32_t** inliers, uint64_t* n_inliers, int32_t* dbg,
                double* dbg_d, float* best_model);
/* estimateTransformFromDescriptorsSets (src/matching.cpp:176-194, pcl::SampleConsensusInitialAlignment).
 * rand_calls (optional, in/out): how many C rand() calls the process has made before / after this call — the reference
 * draws from the never-seeded global rand() stream, so the n-th call of a process differs from the first. */
int mm3d_sac_ia(mm3d_ctx* ctx, const float* kp_src, uint64_t n_src, const float* desc_src, const float* kp_tgt, uint64_t n_tgt,
                const float* desc_tgt, int dim, double min_sample_distance, double max_correspondence_distance, int max_iterations,
                uint64_t* rand_calls, float* transform, float** errors, uint64_t* n_errors);
/* estimateTransformICP (src/matching.cpp:196-221); dbg (optional, 2 ints) = iterations, converged;
 * sums (optional) = per-iteration fixed-point reductions, n_sums x 17 int64 */
int mm3d_icp(mm3d_ctx* ctx, const float* src, uint64_t n_src, const float* tgt, uint64_t n_tgt, const float* initial_guess,
             double max_correspondence_distance, double outlier_rejection_threshold, int max_iterations, double transformation_epsilon,
             double index_leaf, float* transform, int32_t* dbg, long long** sums, uint64_t* n_sums);
/* transformScore (src/matching.cpp:259-268) */
int mm3d_score(mm3d_ctx* ctx, const float* src, uint64_t n_src, const float* tgt, uint64_t n_tgt, const float* transform,
               double max_distance, double index_leaf, double* score);
/* computeGlobalTransforms (src/map_merging.cpp:153-186) on the host: st = int32[n][2] (source, target).
 * With nodes = max index + 1: out has room for nodes matrices.  Optional outputs for parity with src/graph.cpp:
 * in_component n_pairs ints, tree_edges 4 x nodes ints (every tree edge is listed from both ends), centers nodes ints (a node without edges has eccentricity 0, so every
 * isolated node below the max index is reported as a centre). */
int mm3d_global_transforms(int n_pairs, const int32_t* st, const float* transforms, const double* confidences, double confidence_threshold,
                           float* out, int* n_out, int* reference_frame, int32_t* in_component, int32_t* tree_edges, int* n_tree_edges,
                           int32_t* centers, int* n_centers);

/* ---- resident interface (inputs already in HBM; what bench.py and the multi-GPU driver use) -- */

/* Copies the clouds to the device once (mm3d_maps_upload_layout takes other record layouts). */
int mm3d_maps_upload(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, mm3d_maps** maps);
void mm3d_maps_free(mm3d_maps* maps);

/* Per-map feature pipeline (src/map_merging.cpp:212-242) for maps [first, first+count). */
int mm3d_features_compute(mm3d_ctx* ctx, const mm3d_maps* maps, int first, int count, const mm3d_params* params, mm3d_features** out);
int mm3d_features_count(const mm3d_features* f);
/* per map: n_points (after downSample+removeOutliers), n_keypoints, descriptor dim */
int mm3d_features_sizes(const mm3d_features* f, int32_t* n_points, int32_t* n_keypoints, int32_t* dim);
/* device-to-device copies out of / into a feature set (NCCL allgather staging) */
int mm3d_features_export_dev(mm3d_ctx* ctx, const mm3d_features* f, int map, void* points_dev, void* keypoints_dev, void* descriptors_dev);
int mm3d_features_import_dev(mm3d_ctx* ctx, int n_maps, const int32_t* n_points, const void* const* points_dev, const int32_t* n_keypoints,
                             const void* const* keypoints_dev, const void* const* descriptors_dev, int dim, mm3d_features** out);
/* host copies (parity tests) */
int mm3d_features_export_host(mm3d_ctx* ctx, const mm3d_features* f, int map, float* points, float* keypoints, float* descriptors);
void mm3d_features_free(mm3d_features* f);

/* Pair loop (src/map_merging.cpp:256-269) over an explicit pair list ij = int32[n_pairs][2].
 * transforms = n_pairs x 16 (column-major), confidences = n_pairs (1 / transformScore),
 * stats (optional) = int32[n_pairs][4]: correspondences, RANSAC inliers, ICP iterations, ICP converged. */
int mm3d_register_pairs(mm3d_ctx* ctx, const mm3d_features* f, int n_pairs, const int32_t* ij, const mm3d_params* params, float* transforms,
                        double* confidences, int32_t* stats);

/* composeMaps (src/map_merging.cpp:277-305) sharded over ranks.  Per rank: begin (transform + concatenate its maps, local
 * bounding box) -> all-reduce the box -> histogram of global voxel keys over n_buckets key ranges (returns 1 when
 * pcl::VoxelGrid's overflow guard fires: the result is then the plain concatenation) -> all-reduce, pick splitters
 * (splitters[r] <= bucket < splitters[r+1] goes to rank r) -> partition (stable; points_dev receives the points grouped by
 * destination rank) -> all-to-all -> mm3d_downsample_dev on the received points.  Concatenating the ranks' outputs in rank
 * order gives exactly mm3d_compose_maps' output.  begin returns MM3D_ERR_ARG when n_maps != n_transforms (the reference throws). */
typedef struct mm3d_shard mm3d_shard;
int mm3d_compose_shard_begin(mm3d_ctx* ctx, int n_maps, const float* const* clouds, const uint64_t* n_points, int n_transforms,
                             const float* transforms, float* bbox, mm3d_shard** shard);
int mm3d_compose_shard_size(const mm3d_shard* shard, uint64_t* n);
int mm3d_compose_shard_histogram(mm3d_ctx* ctx, const mm3d_shard* shard, const float* global_bbox, double resolution, int n_buckets,
                                 uint64_t* hist);
int mm3d_compose_shard_partition(mm3d_ctx* ctx, const mm3d_shard* shard, const float* global_bbox, double resolution, int n_buckets, int n_ranks,
                                 const int32_t* splitters, uint64_t* send_counts, void* points_dev);
/* the rank's transformed, concatenated points (what the reference's output holds when the overflow guard fires) */
int mm3d_compose_shard_points(mm3d_ctx* ctx, const mm3d_shard* shard, float** out, uint64_t* n_out);
void mm3d_shard_free(mm3d_shard* shard);
/* downSample of a device-resident cloud (points_dev = n x 4 floats in HBM); the result is returned on the host */
int mm3d_downsample_dev(mm3d_ctx* ctx, const void* points_dev, uint64_t n, double resolution, float** out, uint64_t* n_out);

/* Whole path on resident clouds; stage_ms (optional, 10 floats) = device time per stage in the order
 * downsampling, removing outliers, normals, keypoints, descriptors, correspondences, initial alignment,
 * ICP, scoring, graph(host). */
int mm3d_estimate_resident(mm3d_ctx* ctx, const mm3d_maps* maps, const mm3d_params* params, float* out_transforms, int* n_out,
                           float* stage_ms);

/* ---- multi-GPU interface (csrc/dist.cu) -------------------------------------------------------------
 * estimateMapsTransforms (src/map_merging.cpp:188-275) and composeMaps (:277-305) with the maps spread over several
 * GPUs: rank r owns the contiguous block of maps mm3d_dist_block(r, world, n_maps) for the per-map stages, features are
 * exchanged with NCCL, the row-major pair list is dealt out by mm3d_dist_plan, results come back in the reference's pair
 * order.  The transforms are bit-identical to a single-GPU run.  Two ways to form the ranks: */

/* (1) one process, several GPUs: devices = CUDA device ordinals (NULL / 0 = every visible device).  The returned context
 * works with every call of this header; mm3d_estimate_maps_transforms and mm3d_compose_maps fan out over all its devices
 * (one host thread per device, NCCL between them), the other calls run on the first device. */
int mm3d_create_multi(mm3d_ctx** ctx, const int* devices, int n_devices);
/* devices behind a context (1 for mm3d_create) */
int mm3d_device_count(const mm3d_ctx* ctx);

/* (2) one process per GPU: rank 0 fills id (MM3D_COMM_ID_BYTES bytes, an ncclUniqueId) and hands it to every rank through
 * the launcher's own channel; every rank then creates its communicator on its context's device (collective call). */
#define MM3D_COMM_ID_BYTES 128
typedef struct mm3d_comm mm3d_comm;
int mm3d_comm_id(void* id);
int mm3d_comm_create(mm3d_ctx* ctx, int rank, int world, const void* id, mm3d_comm** comm);
void mm3d_comm_destroy(mm3d_comm* comm);
int mm3d_comm_rank(const mm3d_comm* comm);
int mm3d_comm_size(const mm3d_comm* comm);

/* the block of maps a rank owns: [first, first + count) */
int mm3d_dist_block(int rank, int world, int n_maps, int* first, int* count);
/* the pair list (row-major i < j over maps that have keypoints, src/map_merging.cpp:246-254) and the rank that registers
 * each pair (longest-processing-time-first on an estimated cost; deterministic, host only).  pairs = int32[n][2] and owner =
 * int32[n] have room for n_maps (n_maps - 1) / 2 entries; either may be NULL. */
int mm3d_dist_plan(int n_maps, const int32_t* n_points, const int32_t* n_keypoints, int dim, int world, int32_t* pairs, int32_t* owner,
                   int* n_pairs);

/* estimateMapsTransforms, collective over comm (comm = NULL: single rank).  clouds / n_points describe ALL n_maps maps; a
 * rank reads only the host buffers of its own block, the other entries may be NULL.  Every rank receives all transforms. */
int mm3d_estimate_maps_transforms_dist(mm3d_ctx* ctx, mm3d_comm* comm, int n_maps, const float* const* clouds, const uint64_t* n_points,
                                       const mm3d_params* params, float* out_transforms, int* n_out);
/* the same on resident clouds: local_maps = this rank's block (mm3d_maps_upload of exactly those maps).  phase_ms (optional,
 * 5 floats; synchronises between phases, diagnostic only) = features, feature exchange, pair registration, result exchange, graph. */
int mm3d_estimate_resident_dist(mm3d_ctx* ctx, mm3d_comm* comm, int n_maps, const mm3d_maps* local_maps, const mm3d_params* params,
                                float* out_transforms, int* n_out, float* phase_ms);
/* composeMaps, collective over comm: clouds / transforms = this rank's n_local maps (rank order = map order).  *out = this
 * rank's slice of the composed map (mm3d_free); the slices concatenated in rank order are exactly mm3d_compose_maps' output. */
int mm3d_compose_maps_dist(mm3d_ctx* ctx, mm3d_comm* comm, int n_local, const float* const* clouds, const uint64_t* n_points,
                           int n_transforms, const float* transforms, double resolution, float** out, uint64_t* n_out);
int mm3d_compose_resident_dist(mm3d_ctx* ctx, mm3d_comm* comm, const mm3d_maps* local_maps, int n_transforms, const float* transforms,
                               double resolution, float** out, uint64_t* n_out);

#ifdef __cplusplus
}
#endif
#endif /* MM3D_H_ */
