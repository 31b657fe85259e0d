// Device-side launchers of the query kernels (query.cu).  All pointers are DEVICE pointers.
#pragma once
#include "index.hpp"

namespace pcpx {

// A batch of query points.  q == nullptr: the index's own points, thread t <-> sorted point t,
// result row = original index.  Otherwise thread t handles query order[t] (Morton order of the
// queries' cells) and writes result row order[t].
struct QueryBatch
{
    const float* q;
    uint32_t stride_f;
    const uint32_t* order;
    uint32_t nq;
    // device shards (pcpx_index_params.devices): the kNN-shaped launchers answer share `part` of
    // `parts` — a range of the tile list, or of the sorted queries [t_begin, nq) — and leave the
    // other rows of the output untouched
    uint32_t t_begin = 0;
    uint32_t part = 0, parts = 1;
    // by_position != 0: output rows are indexed by the query's SORTED position t instead of its
    // original row (a replica fills a local buffer the primary then reads in order — scattered
    // 12-byte rows written across NVLink cost several times what the kernel itself does)
    uint32_t by_position = 0;
    struct ShardInfo* shard_info = nullptr; // (host) filled by the launcher: which rows were answered
};

// What a sharded kNN-shaped launch answered: tiles [lo, hi) of the tile list of `tile_level`
// (use_tiles != 0), or the sorted positions [lo, hi).
struct ShardInfo
{
    int use_tiles   = 0;
    int tile_level  = 0;
    uint32_t lo = 0, hi = 0;
};

struct Tuning
{
    float success_margin = 1.15f; // a block is tried when its ball should hold margin * (k + 1) points
    int block_threads  = 128;
    // the tile path (tile_core.cuh) for calls whose queries are the indexed points
    int tile           = 1;    // 0: never
    int tile_first_cap = 0;    // batched form: candidates listed before the ball first shrinks (0: 2 (k + 1))
    int tile_min_queries = 24; // tiles with fewer points go to the per-thread path unstaged
    int tile_sub       = 0;    // staged layout: 1 = whole cells (staged in one pass), 2 = 2 x 2 sub-bins per cell, 0 = by call
    float tile_cap     = 1.0f; // largest scan radius in units of the main-level cell
    int warp_retry     = 1;    // what the first pass hands on: 1 = one warp per query (warp_core.cuh), 0 = per-thread retry kernels
    int warp_all       = 0;    // (tests) every kNN-shaped query by the warp-per-query search
    float tile_margin  = 1.15f; // main level: finest whose ball of one cell side holds margin * (k + 1) points
};
Tuning& tuning();

constexpr uint32_t kMaxK = 32; // register-resident list; 32 < k <= 256 takes the heap kernel (big_k.cuh)

void launch_knn(const pcpx_index& ix, const QueryBatch& qb, uint32_t k, float eps, uint32_t* idx,
                float* d2, uint32_t* count, uint32_t* exact_counter);
void launch_normals(const pcpx_index& ix, const QueryBatch& qb, uint32_t k, float eps,
                    float* centroids, float* normals, uint32_t* exact_counter);
void launch_mean_distance(const pcpx_index& ix, const QueryBatch& qb, uint32_t k, float eps,
                          float* means);
void launch_radius_count(const pcpx_index& ix, const QueryBatch& qb, const float* radii, float r,
                         uint32_t* count);
// PCA normal of every query's ball (normals: nq x 3; centroids: nq x 3 or nullptr; count: nq or
// nullptr), rows as launch_radius_count
void launch_radius_normals(const pcpx_index& ix, const QueryBatch& qb, const float* radii, float r,
                           float* normals, float* centroids, uint32_t* count);
void launch_radius_fill(const pcpx_index& ix, const QueryBatch& qb, const float* radii, float r,
                        const uint64_t* offsets, uint32_t* idx);
// dst[row(t) * width + j] = src[t * width + j] for the sorted positions t a shard answered (see
// QueryBatch::by_position); src may be peer memory, read in order
void launch_gather_rows(const pcpx_index& ix, const QueryBatch& qb, const ShardInfo& shard,
                        const uint32_t* src, uint32_t* dst, uint32_t width);
// every list of a CSR (offsets: nq + 1 device values) ascending by value, in place
void launch_sort_lists(const pcpx_index& ix, const uint64_t* offsets, uint32_t nq, uint32_t* idx);
// Axis-aligned boxes (query_box.cu, box_core.cuh): nb records of 6 floats {min xyz, max xyz},
// stride_f floats apart, in device memory; bb = a box every indexed point lies in.
struct BoxBatch
{
    const float* boxes;
    uint32_t stride_f;
    uint32_t nb;
    float bb[6];
};
// count[b] = size of box b's list; max_count (nullptr or one zeroed word) = the largest
void launch_box_count(const pcpx_index& ix, const BoxBatch& bx, uint32_t* count,
                      uint32_t* max_count);
// every box's list at idx + offsets[b] (total = offsets[nb]); returns the kernels launched
uint32_t launch_box_fill(const pcpx_index& ix, const BoxBatch& bx, const uint64_t* offsets,
                         uint64_t total, uint32_t* idx);
// every list ascending (PCPX_RADIUS_SORTED); max_count = the longest; returns the kernels launched
uint32_t launch_box_sort(const pcpx_index& ix, const uint64_t* offsets, uint32_t nb,
                         uint64_t total, uint32_t max_count, uint32_t* idx);
void launch_density_keep(const pcpx_index& ix, float r, uint32_t threshold, uint8_t* keep);
// DBSCAN labels (cluster.cu): labels = n_input device entries, at original positions; returns the
// number of clusters and sets *launches to the kernels launched.  Synchronises the stream.
uint64_t launch_cluster_by_density(const pcpx_index& ix, float r, uint32_t min_points,
                                   uint32_t* labels, uint32_t* launches);
// exclusive scan of `in` (n values) into `out` (n + 1 values, out[n] = total); 64-bit sums
void launch_exclusive_scan_u32(const pcpx_index& ix, const uint32_t* in, uint32_t n, uint64_t* out);
void launch_exclusive_scan_u8(const pcpx_index& ix, const uint8_t* in, uint32_t n, uint64_t* out);
void launch_compact_points(const pcpx_index& ix, const uint8_t* keep, const uint64_t* scan,
                           float* out_xyz);
void launch_mean_reduce(const pcpx_index& ix, const float* v, uint32_t n, double* out_sum,
                        uint32_t* out_valid);
void launch_normals_from_neighbourhoods(cudaStream_t stream, const float* nbr_xyz,
                                        const uint64_t* offsets, uint32_t n, float* normals);
// builds (once per level, kept for the life of the index) the tile list the tile path iterates over
pcpx_index::TileList const& ensure_tile_list(const pcpx_index& ix, int tile_level);
void launch_knn_stats(const pcpx_index& ix, uint32_t k, float eps, unsigned long long* stats4);

} // namespace pcpx
