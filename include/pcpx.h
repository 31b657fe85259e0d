/*
 * pcpx — C ABI of the B200-native neighbourhood engine (libpcpx.so).
 *
 * This is the drop-in boundary for the ONE data-parallel hot path of
 * Q-Minh/point-cloud-processing (pcp): batched k-nearest-neighbour and radius search,
 * tangent-plane PCA normal estimation and the density outlier filter.  pcp itself is a
 * header-only C++17 template library with no FFI, so every entry point below cites the
 * reference interface it replaces (paths relative to the reference's include/pcp/), and
 * include/pcpx/ holds the C++17 headers that keep pcp's own call signatures on top of it.
 *
 * Conventions
 *   - every function returns 0 on success and a negative pcpx_status otherwise; it never
 *     throws and never falls back to a CPU path.  pcpx_last_error() gives the message of
 *     the last failure on the calling thread.
 *   - plain pointers and sizes only.  Every data pointer may be a HOST pointer (pageable or
 *     pinned) or a DEVICE pointer of the index's GPU; the library detects which
 *     (cudaPointerGetAttributes) and stages host buffers itself.  Device pointers let a
 *     caller keep clouds and results resident in HBM.
 *   - points are fp32 xyz, `stride_bytes` apart (12 for std::vector<pcp::point_t>,
 *     common/points/point.hpp:85).
 *   - indices are ORIGINAL positions in the indexed range (what
 *     `view.point() - cloud.data()` is for a pcp::point_view_t element).
 *   - an index is immutable after creation and may be queried from several host threads AT ONCE:
 *     every kNN / radius / normals / mean-distance / density-filter call borrows its own CUDA
 *     stream and temporaries, so calls from different threads overlap on the device (the reference's
 *     const member functions are re-entrant the same way); pcpx_last_timings is last-writer-wins.
 */
#ifndef PCPX_H
#define PCPX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCPX_VERSION 100

typedef enum pcpx_status
{
    PCPX_OK                = 0,
    PCPX_ERR_INVALID_ARG   = -1,
    PCPX_ERR_CUDA          = -2,
    PCPX_ERR_NO_DEVICE     = -3,
    PCPX_ERR_OUT_OF_MEMORY = -4,
    PCPX_ERR_UNSUPPORTED   = -5
} pcpx_status;

#define PCPX_NO_NEIGHBOUR 0xFFFFFFFFu /* padding value in kNN index rows */

typedef struct pcpx_index pcpx_index; /* opaque: the GPU-resident spatial index */

/*
 * Index parameters.  Replaces pcp::octree_parameters_t (octree/linked_octree_node.hpp:31-40)
 * and pcp::kdtree::construction_params_t (kdtree/linked_kdtree.hpp:26-33): tree shape does
 * not change the result of an exact search, so node_capacity / max_depth have no
 * counterpart; the one structure-dependent behaviour that survives is the root voxel grid:
 * with use_voxel_grid != 0, points outside [voxel_min, voxel_max] (inclusive,
 * common/axis_aligned_bounding_box.hpp:111-124) are NOT indexed, as
 * basic_linked_octree_node_t::insert rejects them (octree/linked_octree_node.hpp:174).
 * Zero-initialise for defaults.
 */
typedef struct pcpx_index_params
{
    int32_t device;         /* CUDA device ordinal; -1 = current device */
    int32_t use_voxel_grid; /* 0 = auto bounding box (octree/linked_octree.hpp:103-121) */
    float voxel_min[3];
    float voxel_max[3];
    uint32_t max_level;  /* finest grid level (cells per axis = 2^level); 0 = auto */
    uint32_t min_cell_occupancy; /* finest stored level keeps mean occupancy >= this; 0 = auto */
    /* Several GPUs behind one handle (replicated index, queries sharded): n_devices >= 2 builds
     * the SAME index on every listed device (devices[0] is the primary and takes the place of
     * `device`; the cloud reaches the others by peer copy when xyz is device memory) and every
     * kNN-shaped call with k <= 32 — pcpx_knn, pcpx_estimate_normals, pcpx_estimate_tangent_planes,
     * pcpx_mean_knn_distance — is answered by all of them at once: device i takes the i-th
     * contiguous share of the tile list (queries == NULL) or of the Morton-sorted queries; the
     * primary reads the replicas' answers over NVLink and scatters them to the caller's rows
     * (peer access is required in both directions: PCPX_ERR_UNSUPPORTED without it).  Results are bit-identical to a one-device
     * index.  Every other call runs on the primary alone.  0 or 1: one device.
     * (Clouds too large for one GPU are cut into slabs with halo strips one level up:
     * point-cloud-processing_b200/sharding.py over torch.distributed, pcpx_extract_bands.) */
    uint32_t n_devices;
    int32_t devices[8];
    uint32_t shard_mode; /* PCPX_SHARD_REPLICATED (0, the only mode inside the library);
                            PCPX_SHARD_SLAB returns PCPX_ERR_UNSUPPORTED: slabs are one process
                            per GPU (sharding.py + pcpx_extract_bands) */
    uint32_t reserved[6];
} pcpx_index_params;

#define PCPX_SHARD_REPLICATED 0u
#define PCPX_SHARD_SLAB 1u

/* Facts about a built index (all filled by pcpx_index_info). */
typedef struct pcpx_index_info
{
    uint64_t n_input;   /* points handed to pcpx_index_create */
    uint64_t n_indexed; /* points actually indexed == octree.size() (octree/linked_octree.hpp:127) */
    float bbox_min[3];  /* root voxel: pcp::bounding_box (common/axis_aligned_bounding_box.hpp:214-251) */
    float bbox_max[3];  /*   or the user's voxel grid */
    uint32_t code_bits;    /* Morton bits sorted on */
    uint32_t finest_level; /* finest level with a cell table */
    uint64_t n_cells;      /* cells over all stored levels */
    uint64_t device_bytes; /* HBM held by the index */
    int32_t device;
    float build_ms; /* device time of the build (CUDA events) */
    uint32_t n_devices; /* devices that hold a replica of the index (1: the primary only) */
} pcpx_index_info;

/* ---- lifecycle -------------------------------------------------------------------------- */

int pcpx_device_count(void);
const char* pcpx_last_error(void);

/*
 * Build the index on the GPU: bbox reduce -> quantise + Morton encode -> radix sort ->
 * per-level cell tables -> float4 SoA reorder; nothing is built on the host.
 * Replaces basic_linked_octree_t's range constructors (octree/linked_octree.hpp:83-121) and
 * basic_linked_kdtree_t's constructor (kdtree/linked_kdtree.hpp:100-135).
 * n == 0 is valid (every query then returns nothing).
 */
int pcpx_index_create(
    const float* xyz,
    size_t n,
    size_t stride_bytes,
    const pcpx_index_params* params /* may be NULL */,
    pcpx_index** out_index);

void pcpx_index_destroy(pcpx_index* index);
int pcpx_index_info_get(const pcpx_index* index, pcpx_index_info* out_info);
/* The root voxel alone: pcp::bounding_box of the cloud (common/axis_aligned_bounding_box.hpp:
 * 214-251) or the user's voxel grid — what basic_linked_octree_t::voxel_grid() returns. */
int pcpx_index_bbox(const pcpx_index* index, float out_min[3], float out_max[3]);

/* ---- queries ----------------------------------------------------------------------------
 * `queries`: nq points (fp32 xyz, query_stride_bytes apart), or NULL for "the indexed cloud's
 * own points, in their original order" (then nq must equal n_input; points that were not
 * indexed because of the voxel grid are still valid query targets).
 */

/*
 * Batched exact kNN.  Replaces basic_linked_octree_t::nearest_neighbours
 * (octree/linked_octree.hpp:245-254 -> octree/linked_octree_node.hpp:453-570) and
 * basic_linked_kdtree_t::nearest_neighbours (kdtree/linked_kdtree.hpp:200-263).
 *   - row i of out_idx (k entries) = the neighbours of query i nearest -> furthest, ordered by
 *     (fp32 squared distance, original index); rows shorter than k are padded with
 *     PCPX_NO_NEIGHBOUR (out_d2 with +inf); out_count[i] = number of valid entries.
 *   - distance = ((dx*dx) + (dy*dy)) + (dz*dz) in fp32 without FMA (common/norm.hpp:102-112).
 *   - a point is excluded iff |dx| < eps && |dy| < eps && |dz| < eps in fp32
 *     (common/vector3d_queries.hpp:31-35,48-64 applied at octree/linked_octree_node.hpp:540),
 *     which also drops foreign near-duplicates; eps is cast to float like the reference does.
 *   - k == 0 -> nothing is written, returns PCPX_OK (octree/linked_octree_node.hpp:464).
 *   - k <= 32 runs the register-list kernels, 32 < k <= 256 an exact heap kernel (slower per
 *     neighbour); larger k returns PCPX_ERR_UNSUPPORTED.
 * out_d2 and out_count may be NULL.
 */
int pcpx_knn(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    uint32_t k,
    double eps,
    uint32_t* out_idx,
    float* out_d2,
    uint32_t* out_count);

/*
 * Sphere range search, count only.  Replaces `range_search(sphere).size()`
 * (octree/linked_octree.hpp:264-276 -> octree/linked_octree_node.hpp:581-614,
 * kdtree/linked_kdtree.hpp:270-316) with predicate pcp::sphere_t::contains
 * (common/sphere.hpp:27-35): fl(d2) <= fl(r*r).  The query point itself is counted when it is
 * an indexed point.  radii != NULL gives one radius per query, else `radius` is used.
 * Note: the reference prunes with d2 <= r (common/intersections.hpp:101) and can therefore
 * MISS in-range points when r > 1; this library always returns the exact set.
 */
int pcpx_radius_count(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    const float* radii,
    float radius,
    uint32_t* out_count);

/*
 * Sphere range search, CSR lists.  out_offsets has nq + 1 entries.  `out_idx_device` is a set
 * of flags: PCPX_RADIUS_DEVICE (1) leaves *out_idx in device memory of the index's GPU instead
 * of HOST memory (free with pcpx_free either way); PCPX_RADIUS_SORTED (2) sorts every query's
 * list ascending by original index.  Without it the order within a query is the index's
 * traversal order (deterministic, unspecified — as in the reference, whose order is the tree's
 * DFS).
 */
#define PCPX_RADIUS_DEVICE 1
#define PCPX_RADIUS_SORTED 2
int pcpx_radius_search(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    const float* radii,
    float radius,
    uint64_t* out_offsets,
    uint32_t** out_idx,
    int out_idx_device);

/*
 * Axis-aligned box range search.  Replaces range_search(axis_aligned_bounding_box_t)
 * (octree/linked_octree.hpp:264-276 -> octree/linked_octree_node.hpp:581-614) and
 * range_search(kd_axis_aligned_bounding_box_t) (kdtree/linked_kdtree.hpp:270-316), with predicate
 * axis_aligned_bounding_box_t::contains (common/axis_aligned_bounding_box.hpp:99-149).
 *   - boxes: nb records of 6 fp32 {min x, min y, min z, max x, max y, max z}, box_stride_bytes
 *     (>= 24, a multiple of 4) apart, in host or device memory.
 *   - box b's result: the indexed points p with min <= p <= max on all three axes, compared in
 *     fp32 (inclusive on both ends); points a voxel grid left out of the index are in no box.
 *   - a box with a NaN bound or min > max on some axis is empty; +-inf bounds are valid.
 * pcpx_box_count: out_count (nb entries) = the size of every box's result.
 */
int pcpx_box_count(
    const pcpx_index* index,
    const float* boxes,
    size_t nb,
    size_t box_stride_bytes,
    uint32_t* out_count);

/*
 * Box range search, CSR lists (out_offsets: nb + 1 entries), flags as pcpx_radius_search:
 * PCPX_RADIUS_DEVICE leaves *out_idx in device memory, PCPX_RADIUS_SORTED sorts every list
 * ascending by original index; without it a list is in the index's traversal order
 * (deterministic, unspecified).  Free *out_idx with pcpx_free.  Runs on the primary device of a
 * multi-device index.
 */
int pcpx_box_search(
    const pcpx_index* index,
    const float* boxes,
    size_t nb,
    size_t box_stride_bytes,
    uint64_t* out_offsets,
    uint32_t** out_idx,
    int flags);

void pcpx_free(void* p, int is_device);

/*
 * Fused kNN -> 3x3 scatter matrix -> symmetric eigensolve -> normal.  Replaces
 * pcp::algorithm::estimate_normals (algorithm/estimate_normals.hpp:50-93,116-164) driven by a
 * kNN map over the index, with pcp::estimate_normal (common/normals/normal_estimation.hpp:32-78)
 * as the per-neighbourhood body and default_normal_transform (algorithm/common.hpp:31-34):
 * fp32 mean, centred UN-normalised scatter, unit eigenvector of the smallest eigenvalue.
 * The sign is not canonical (the reference returns whatever Eigen does): compare with |dot|.
 * Neighbourhoods with fewer than 3 points have no defined plane; the result is (0,0,1).
 * out_normals: nq x 3 fp32.
 */
int pcpx_estimate_normals(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    uint32_t k,
    double eps,
    float* out_normals);

/*
 * As pcpx_estimate_normals, and also writes the neighbourhood centroid: the tangent plane
 * (point, normal) of pcp::algorithm::estimate_tangent_planes
 * (algorithm/estimate_tangent_planes.hpp:82-94).  out_points: nq x 3 fp32.
 */
int pcpx_estimate_tangent_planes(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    uint32_t k,
    double eps,
    float* out_points,
    float* out_normals);

/*
 * Fused ball -> 3x3 scatter matrix -> symmetric eigensolve -> normal, in one device pass with
 * no per-neighbour data in memory.  Replaces pcp::algorithm::estimate_normals
 * (algorithm/estimate_normals.hpp:50-93,116-164) driven by a sphere range-search map,
 * `[&](auto const& p) { return octree.range_search(sphere_t{p, r}, point_view); }`
 * (octree/linked_octree.hpp:264-276, predicate common/sphere.hpp:27-35), with
 * pcp::estimate_normal (common/normals/normal_estimation.hpp:32-78) as the per-ball body.
 *   - the ball of query i is exactly the set pcpx_radius_search returns for it: the indexed
 *     points with fl(d2) <= fl(r*r), the query itself included when it is an indexed point;
 *     points a voxel grid left out of the index are in no ball but are valid queries.
 *   - radii != NULL gives one radius per query, else `radius` is used.
 *   - per ball: fp32 mean, centred UN-normalised scatter, unit eigenvector of the smallest
 *     eigenvalue.  The sign is not canonical: compare with |dot|.  A ball of 0 or 1 points (zero
 *     scatter) gives (0,0,1).
 *   - out_count (nq entries, may be NULL) = the ball's size, equal to pcpx_radius_count.
 * Note: the reference prunes with d2 <= r (common/intersections.hpp:101) and can therefore
 * MISS in-range points when r > 1; this library always uses the exact ball.
 * out_normals: nq x 3 fp32.  Runs on the primary device of a multi-device index.
 */
int pcpx_estimate_normals_radius(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    const float* radii,
    float radius,
    float* out_normals,
    uint32_t* out_count);

/*
 * As pcpx_estimate_normals_radius, and also writes the ball's centroid: the tangent plane
 * (point, normal) of pcp::algorithm::estimate_tangent_planes
 * (algorithm/estimate_tangent_planes.hpp:82-94) with a sphere range-search map.  An empty ball
 * gives a NaN centroid, normal (0,0,1) and count 0.  out_points: nq x 3 fp32.
 */
int pcpx_estimate_tangent_planes_radius(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    const float* radii,
    float radius,
    float* out_points,
    float* out_normals,
    uint32_t* out_count);

/*
 * PCA normal of caller-supplied neighbourhoods (CSR: neighbourhood i = points
 * nbr_xyz[offsets[i] .. offsets[i + 1]), packed fp32 xyz).  This is pcp::estimate_normal
 * (common/normals/normal_estimation.hpp:32-78) batched on the GPU; it serves
 * pcp::algorithm::estimate_normals when the KnnMap is an arbitrary user callable whose
 * neighbourhoods the host has already gathered.  out_normals: n x 3 fp32; device = CUDA ordinal
 * (-1 = current).  Host or device pointers.
 */
int pcpx_normals_from_neighbourhoods(
    const float* nbr_xyz,
    const uint64_t* offsets,
    size_t n,
    int device,
    float* out_normals);

/*
 * Mean distance to the k nearest neighbours of every indexed point.  Replaces
 * pcp::algorithm::average_distances_to_neighbors / average_distance_to_neighbors
 * (algorithm/average_distance_to_neighbors.hpp:39-113): per point the sequential fp32 sum of
 * sqrt(d2) nearest -> furthest divided by the neighbour count (bit-exact); *out_mean is the
 * mean of those values accumulated in fp64 by a fixed-shape tree (the reference's fp32
 * std::reduce order is unspecified).  out_per_point (n_input entries) and out_mean may be NULL.
 */
int pcpx_mean_knn_distance(
    const pcpx_index* index,
    uint32_t k,
    double eps,
    float* out_per_point,
    double* out_mean);

/*
 * Density outlier filter: keep point i iff |{j : d2(p_i, p_j) <= radius^2}| >= threshold, the
 * count including p_i itself.  Replaces the remove_if of
 * examples/filter_point_cloud_noise_by_density.cpp:81-91 evaluated on the immutable input.
 * out_keep_mask: n_input bytes (1 = kept), may be NULL.  out_xyz: kept points, packed xyz in
 * original relative order (std::remove_if is stable), capacity n_input*3 floats, may be NULL.
 * out_n: number kept.
 */
int pcpx_density_filter(
    const pcpx_index* index,
    float radius,
    uint32_t threshold,
    uint8_t* out_keep_mask,
    float* out_xyz,
    size_t* out_n);

/*
 * Density-based clustering (DBSCAN) of the indexed points, a pcpx extension: the reference has
 * no clustering.  With min_points <= 1 it is Euclidean clustering, the connected components of
 * the radius graph.
 *   - N(p) is exactly the ball pcpx_radius_search returns for p with queries = the cloud: the
 *     indexed q with fl(d2(p, q)) <= fl(radius * radius), d2 computed without FMA, p included.
 *     d2 is symmetric bit for bit (negating dx does not change dx * dx), so q in N(p) <=> p in
 *     N(q).
 *   - p is core iff |N(p)| >= min_points: exactly the points pcpx_density_filter(radius,
 *     min_points) keeps.  With min_points 0 or 1 every indexed point is core.
 *   - clusters are the connected components of the graph on the core points with an edge p - q
 *     iff q in N(p), numbered 0 .. C-1 in ascending order of the smallest original index among
 *     their core points (the order of scipy.sparse.csgraph.connected_components).
 *   - a non-core point with a core point in N(p) takes the label of the core q in N(p) with the
 *     smallest (fl(d2), original index); every other point is PCPX_NOISE, including the points a
 *     voxel grid left out of the index.
 * The labels are unique under these rules: identical bytes whatever the scheduling, for host or
 * device output, one or several replicas and concurrent calls.
 * out_labels: n_input entries, host or device.  *out_n_clusters (host, may be NULL) = C.  A NaN
 * radius is PCPX_ERR_INVALID_ARG; every other radius means what it means for
 * pcpx_radius_search.  Runs on the primary device of a multi-device index.
 */
#define PCPX_NOISE 0xFFFFFFFFu
int pcpx_cluster_by_density(
    const pcpx_index* index,
    float radius,
    uint32_t min_points,
    uint32_t* out_labels,
    uint64_t* out_n_clusters);

/* ---- rigid registration (a pcpx extension: the reference has none) ------------------------- */

/*
 * Bounded nearest neighbour of transformed queries: the correspondence search of ICP.
 *   - transformed query: with a row-major 4x4 rigid `transform` T = [R | t], query i is first
 *     mapped to y_i, each component computed in fp64 as ((R[a][0]*x + R[a][1]*y) + R[a][2]*z)
 *     + t[a] without FMA, then rounded once to fp32.  NULL means identity: the query is used as is.
 *   - out_idx[i] = the indexed point q with the smallest (fl(d2), original index) among those with
 *     fl(d2(y_i, q)) <= fl(max_distance * max_distance), d2 the no-FMA fp32 distance of
 *     pcpx_knn; out_d2[i] (may be NULL) = that d2.
 *   - no such point (also for a query with a non-finite coordinate, and for points a voxel grid
 *     left out of the index): PCPX_NO_NEIGHBOUR and +inf.
 *   - so the result equals the row of pcpx_knn(k = 1, eps = 0) whenever that row's d2 passes the
 *     bound.
 *   - max_distance must be finite and > 0 (else PCPX_ERR_INVALID_ARG); r > 1 is exact, as for
 *     pcpx_radius_search.
 * Host or device buffers, strided queries.  Runs on the primary device of a multi-device index.
 */
int pcpx_nearest_within(
    const pcpx_index* index,
    const float* queries,
    size_t nq,
    size_t query_stride_bytes,
    const double transform[16] /* may be NULL */,
    float max_distance,
    uint32_t* out_idx,
    float* out_d2 /* may be NULL */);

/*
 * Iterative closest point: the rigid transform that registers `source` to the indexed target.
 *   - target_normals: n_input rows in original order (what pcpx_estimate_normals(queries = NULL)
 *     writes), normal_stride_bytes apart; required for point-to-plane, ignored for
 *     point-to-point.  The sign of a normal does not matter.  A pair whose target normal has a
 *     non-finite component is not a correspondence.
 *   - iteration it, from T_0 = init (NULL = identity):
 *       1. the pairs (y_i, q_i) are those of pcpx_nearest_within(source, T_it, max_distance);
 *       2. sums in fp64 about c, the centre of the target's root voxel (pcpx_index_bbox):
 *          point-to-plane A = sum J^T J, b = sum J^T r with J = [(y - c) x n, n],
 *          r = (y - q) . n; point-to-point sum (y - c), sum (q - c), sum (y - c)(q - c)^T and
 *          the count; both sum d2;
 *       3. fewer than 6 (plane) or 3 (point) pairs: stop, PCPX_ICP_TOO_FEW;
 *       4. solve on the host in fp64: point-to-plane x = (omega, v) = -A^+ b, A^+ the
 *          pseudo-inverse of a cyclic-Jacobi eigendecomposition (fixed sweep order) without the
 *          eigenvalues <= 1e-12 * lambda_max, so a motion the pairs do not constrain (a plane
 *          sliding in itself) is zero; point-to-point Horn's quaternion method (the same Jacobi
 *          on the 4x4 matrix), never a reflection;
 *       5. T_it+1 = (y -> R(omega)(y - c) + c + v) o T_it, R by Rodrigues' formula in fp64;
 *       6. |omega| <= rotation_tolerance and |v| <= translation_tolerance: stop,
 *          PCPX_ICP_CONVERGED; after max_iterations updates: PCPX_ICP_MAX_ITERATIONS.
 *   - out_transform = the last T.  out_result and out_correspondences (ns entries, host or
 *     device, may be NULL: the original index of every source point's pair, or
 *     PCPX_NO_NEIGHBOUR) describe that T: one more correspondence pass runs after the loop.
 *     rmse = sqrt(sum d2 / n_correspondences) in fp64, NaN without pairs; fitness =
 *     n_correspondences / ns.
 *   - PCPX_ERR_INVALID_ARG: a NaN, infinite or <= 0 max_distance, an unknown metric,
 *     point-to-plane without normals, params or out_transform NULL.
 *   - ns == 0 or an empty index: out_transform = init, 0 correspondences, rmse NaN.
 *   - the bytes of the transform, the result and the correspondences depend on the inputs alone:
 *     host or device buffers, strided input, repeated and concurrent calls and multi-device
 *     handles give the same.  Runs on the primary device.
 *   - pcpx_last_timings covers the whole call; kernel_launches counts every launch.
 */
#define PCPX_ICP_POINT_TO_PLANE 0u
#define PCPX_ICP_POINT_TO_POINT 1u
#define PCPX_ICP_CONVERGED 0u
#define PCPX_ICP_MAX_ITERATIONS 1u
#define PCPX_ICP_TOO_FEW 2u
typedef struct pcpx_icp_params
{
    uint32_t metric;               /* PCPX_ICP_* */
    uint32_t max_iterations;       /* 0 = 30 */
    float max_distance;            /* correspondence bound, required: finite, > 0 */
    double rotation_tolerance;     /* rad; 0 = 1e-6 */
    double translation_tolerance;  /* 0 = 1e-6 x the diagonal of the target's root voxel */
    uint32_t reserved[8];
} pcpx_icp_params;
typedef struct pcpx_icp_result
{
    uint32_t iterations;        /* updates applied */
    uint32_t stop_reason;       /* PCPX_ICP_CONVERGED / _MAX_ITERATIONS / _TOO_FEW */
    uint64_t n_correspondences;
    double fitness;             /* n_correspondences / ns */
    double rmse;                /* sqrt(sum d2 / n_correspondences), NaN if none */
} pcpx_icp_result;
int pcpx_icp(
    const pcpx_index* target,
    const float* target_normals,
    size_t normal_stride_bytes,
    const float* source,
    size_t ns,
    size_t source_stride_bytes,
    const pcpx_icp_params* params,
    const double init[16] /* NULL = identity */,
    double out_transform[16],
    pcpx_icp_result* out_result /* may be NULL */,
    uint32_t* out_correspondences /* ns entries, may be NULL */);

/* ---- radius-search callers: smoothing and resampling (SURVEY.md 8f rank 3) ---------------- */

/*
 * Bilateral filter of the points.  Replaces pcp::algorithm::bilateral_filter_points
 * (algorithm/bilateral_filter.hpp:301-421; per point bilateral::detail::compute_pi, :47-100):
 * `iterations` (the reference's params.K) times, every point moves to the weighted mean of its
 * projections onto the tangent planes (p_j, n_j) of the points within 2*sigmaf, weights
 * gaussian(sigmaf, |s - p_j|) * gaussian(sigmag, |proj_j(s) - s|); the index is rebuilt on the
 * moved points each iteration, the normals stay those handed in.  fp32 as in the reference;
 * neighbours are summed in index order, not kd-tree order, so results agree to rounding
 * (tests: 1e-5 of the cloud extent).  xyz / normals / out_xyz: n rows, host or device; out_xyz
 * packed (12 B rows).  out_device_ms (may be NULL): device time of the whole call.
 */
int pcpx_bilateral_filter_points(
    const float* xyz,
    size_t n,
    size_t stride_bytes,
    const float* normals,
    size_t normal_stride_bytes,
    double sigmaf,
    double sigmag,
    uint32_t iterations,
    int device,
    float* out_xyz,
    float* out_device_ms);

/*
 * Bilateral "normal improvement".  Replaces pcp::algorithm::bilateral_filter_normals
 * (algorithm/bilateral_filter.hpp:452-575; per point bilateral::detail::compute_ni, :113-267):
 * the points stay fixed (one index), and `iterations` times every normal is mapped through the
 * Jacobian of the bilateral filter at its point and renormalised.  Formula restated verbatim,
 * including the sign convention of the reference's projection Jacobian.
 */
int pcpx_bilateral_filter_normals(
    const float* xyz,
    size_t n,
    size_t stride_bytes,
    const float* normals,
    size_t normal_stride_bytes,
    double sigmaf,
    double sigmag,
    uint32_t iterations,
    int device,
    float* out_normals,
    float* out_device_ms);

/*
 * WLOP / LOP resampling.  Replaces pcp::algorithm::wlop::wlop (algorithm/wlop.hpp:278-438).
 * n_out points (params.I) are drawn from the cloud and moved `iterations` (params.k) times by
 * the local-median attraction of the cloud plus the mutual repulsion (mu) of the resampled
 * points, both with support radius h; uniform != 0 applies the WLOP density weights v_j, w_i
 * (:371-401), 0 gives plain LOP.  The reference draws the start set with std::random_device
 * (:346-358), which cannot be reproduced: pass it as initial_idx (n_out indices into xyz, host
 * or device), or NULL for the last n_out entries of a std::mt19937(seed) shuffle of 0..n-1.
 * out_xyz: n_out packed rows in the order of initial_idx.
 */
int pcpx_wlop(
    const float* xyz,
    size_t n,
    size_t stride_bytes,
    const uint32_t* initial_idx,
    size_t n_out,
    double mu,
    double h,
    uint32_t iterations,
    int uniform,
    uint32_t seed,
    int device,
    float* out_xyz,
    float* out_device_ms);

/* ---- normal orientation (SURVEY.md 8f rank 4) ---------------------------------------------- */

/*
 * Orient a normal field consistently.  Replaces pcp::algorithm::propagate_normal_orientations
 * (algorithm/estimate_normals.hpp:187-302) with a k-nearest-neighbour KnnMap over the indexed
 * cloud: the directed kNN graph (graph/knn_adjacency_list.hpp:117-156) is searched breadth
 * first (graph/search.hpp:41-85) from the first point of maximal z, whose normal becomes
 * (0, 0, 1); every other reached normal is negated iff its inner product with the final normal
 * of the vertex that reached it is < 0 and not within 1e-5 of 0.  Unreached points keep their
 * normals.  The result is bit-identical to the reference's sequential search: the queue order
 * is reproduced exactly (see csrc/orient.cu).
 *
 * edge_order: the reference walks the out-edges of a vertex in the order its
 * std::unordered_multimap yields equal keys (graph/directed_adjacency_list.hpp:79-83,183),
 * which is the standard library's choice.  PCPX_EDGES_FURTHEST_FIRST is what libstdc++ does
 * (reverse insertion order; verified against the reference compiled with g++ 13);
 * PCPX_EDGES_NEAREST_FIRST is insertion order.
 *
 * normals: n_input x 3 packed floats in input order, host or device, updated in place.
 * out_levels / out_reached (may be NULL): BFS depth and number of vertices reached.
 */
#define PCPX_EDGES_FURTHEST_FIRST 0
#define PCPX_EDGES_NEAREST_FIRST 1

int pcpx_orient_normals(
    const pcpx_index* index,
    uint32_t k,
    double eps,
    int edge_order,
    float* normals,
    uint32_t* out_levels,
    uint64_t* out_reached);

/*
 * The same search over a caller-supplied directed graph (any KnnMap of the reference's
 * signature): vertex i has the out-edges neighbours[i*k .. i*k+k) in insertion order,
 * PCPX_NO_NEIGHBOUR marking unused slots.  xyz (n rows) only selects the root.
 */
int pcpx_orient_normals_graph(
    const float* xyz,
    size_t n,
    size_t stride_bytes,
    const uint32_t* neighbours,
    uint32_t k,
    int edge_order,
    int device,
    float* normals,
    uint32_t* out_levels,
    uint64_t* out_reached);

/* ---- multi-GPU plumbing (SURVEY.md 8e) ---------------------------------------------------- */

/*
 * Cut the two boundary strips of a slab out of a device-resident cloud: rows whose coordinate
 * `axis` is < below go to out_below, rows with coordinate > above to out_above, both in input
 * order (an ordered compaction, so the assembled local cloud is reproducible).  These are the
 * strips a rank sends to its neighbours across the two inner faces of its slab
 * (point-cloud-processing_b200/sharding.py: exchange_halo).  xyz / out_*: DEVICE memory; out_*
 * hold `capacity` packed rows each, rows beyond the capacity are counted but not written.
 * counts[0..1] (host or device memory) receive the two strip sizes.  cuda_stream: the
 * cudaStream_t to run on (NULL = the legacy default stream); the call returns after the stream
 * has finished the work.
 */
int pcpx_extract_bands(
    const float* xyz,
    size_t n,
    size_t stride_bytes,
    int axis,
    float below,
    float above,
    float* out_below,
    float* out_above,
    size_t capacity,
    uint64_t* counts,
    void* cuda_stream);

/* ---- instrumentation -------------------------------------------------------------------- */

/* Device time (CUDA events on the launching stream) of the last call of each kind made
 * through this index on the calling thread's most recent call; < 0 when never run. */
typedef struct pcpx_timings
{
    float build_ms;     /* whole index build */
    float sort_ms;      /*   of which radix sort */
    float query_sort_ms;/* sorting external queries by cell */
    float kernel_ms;    /* the query kernel proper (kNN / normals / radius / filter) */
    float total_ms;     /* whole call on the device incl. H2D / D2H staging */
    uint32_t kernel_launches; /* kernels launched by the last call */
    uint32_t retry_queries;   /* queries the block search answered through its exact tie path */
    uint32_t deferred_queries; /* kNN-shaped calls: queries the first pass (tile kernel / block search)
                                  handed on to the warp-per-query kernel (device shards: the primary's) */
    uint32_t expanded_queries; /* ... of those, queries whose first block attempt there was not final */
} pcpx_timings;

int pcpx_last_timings(const pcpx_index* index, pcpx_timings* out);

/* Process-wide tunables (performance only, never results).  Known names:
 *   "success_margin"  a kNN-shaped call first tries the cheapest (level, rings) block whose ball
 *                     is expected to hold success_margin * (k + 1) points (default 1.15).
 *   "pool_cap_mb"     cap of the per-device cache of freed device blocks, in MiB (default: one
 *                     eighth of the device's memory, at least 1024; 0 restores the default).
 *   "tile"            1 (default): calls whose queries are the indexed points themselves take the
 *                     tile-cooperative kernel (shared-memory staged candidates); 0: never.
 *   "tile_sub"        staged layout of the tile kernel: 1 = whole cells (staged in one pass),
 *                     2 = 2 x 2 sub-bins per cell, 0 (default) = chosen per call.
 *   "warp_retry"      1 (default): queries the first pass hands on are answered one warp per query
 *                     (octree descent, exact 64-bit keys); 0: per-thread retry kernels.
 *   "warp_all"        1: every kNN-shaped query takes the warp-per-query search (tests).
 *   "tile_cap"        largest scan radius of the tile kernel in cell sides (default 1).
 *   "tile_margin"     like success_margin, for the tile kernel's level (default 1.15). */
int pcpx_set_tuning(const char* name, double value);

/* Page-locked host memory for buffers handed to the calls above.  Pageable host memory is staged
 * by the driver through a bounce buffer (a 120 MB cloud: ~12 ms instead of 2.2 ms, and not
 * asynchronous); include/pcpx/pcp.hpp stages its flattened clouds and results in these. */
int pcpx_host_alloc(size_t bytes, void** out_ptr);
void pcpx_host_free(void* ptr);

/* Device memory the library keeps for reuse.  Temporaries and destroyed indices go back to a
 * per-device cache (cudaMalloc / cudaFree synchronise the device and cost up to milliseconds);
 * the cache is capped — one eighth of the device's memory by default (at least 1 GiB),
 * PCPX_POOL_CAP_MB in the environment or
 * pcpx_set_tuning("pool_cap_mb", x) — and blocks beyond the cap are returned to the driver at
 * once.  pcpx_trim(device) waits for the device to go idle and frees the whole cache, for
 * applications that share the GPU with other allocators. */
int pcpx_trim(int device);

/* Search work of a self-kNN over the whole cloud, summed over queries:
 * out4 = { candidate distance evaluations, cell-table lookups, levels tried,
 *          queries that needed more than one level }. */
int pcpx_debug_knn_stats(const pcpx_index* index, uint32_t k, double eps, uint64_t* out4);

#ifdef __cplusplus
}
#endif

#endif /* PCPX_H */
