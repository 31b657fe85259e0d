// Density-based clustering (pcpx_cluster_by_density): DBSCAN labels over the index's exact fp32
// ball, the bodies in cluster_core.cuh.  One thread per sorted position throughout, so the lanes
// of a warp walk the same few cells.
//   1. core flags (the density filter's early-exit walk), parent[t] = t
//   2. union: every core point joins its core neighbours at smaller sorted positions
//   3. flatten: parent[t] = root (no path halving here); the smallest original index of every set goes to its root
//   4. flag, at its original position, the core point holding its set's smallest index; an
//      exclusive scan of the flags numbers the clusters in ascending order of that index
//   5. labels: a core point's cluster, a border point's by the border rule, noise otherwise
#include <algorithm>

#include "cluster_core.cuh"
#include "query.hpp"

namespace pcpx {

namespace {

constexpr int kClusterBlock = 128;

uint32_t blocks_for(uint32_t n) { return std::max(1u, (n + kClusterBlock - 1) / kClusterBlock); }

__global__ void __launch_bounds__(kClusterBlock) cluster_core_kernel(
    GridView g, float r, uint32_t min_points, uint8_t* __restrict__ core, uint32_t* __restrict__ parent)
{
    uint32_t const t = blockIdx.x * kClusterBlock + threadIdx.x;
    if (t >= g.n)
        return;
    core[t]   = cluster_is_core(g, __ldg(g.pts + t), r, min_points);
    parent[t] = t;
}

// (`parent` is written by other threads during the pass: no __restrict__, no __ldg)
__global__ void __launch_bounds__(kClusterBlock) cluster_union_kernel(
    GridView g, float r, const uint8_t* __restrict__ core, uint32_t* parent)
{
    uint32_t const t = blockIdx.x * kClusterBlock + threadIdx.x;
    if (t >= g.n || !core[t])
        return;
    cluster_union_point(g, core, parent, t, r);
}

__global__ void __launch_bounds__(kClusterBlock) cluster_flatten_kernel(
    GridView g, const uint8_t* __restrict__ core, uint32_t* parent, uint32_t* __restrict__ min_orig)
{
    uint32_t const t = blockIdx.x * kClusterBlock + threadIdx.x;
    if (t >= g.n || !core[t])
        return;
    uint32_t const root = uf_root(parent, t);
    parent[t]           = root;
    atomicMin(min_orig + root, __float_as_uint(__ldg(&g.pts[t].w)));
}

__global__ void __launch_bounds__(kClusterBlock) cluster_first_kernel(
    GridView g, const uint8_t* __restrict__ core, const uint32_t* __restrict__ parent,
    const uint32_t* __restrict__ min_orig, uint8_t* __restrict__ first)
{
    uint32_t const t = blockIdx.x * kClusterBlock + threadIdx.x;
    if (t >= g.n || !core[t])
        return;
    uint32_t const orig = __float_as_uint(__ldg(&g.pts[t].w));
    if (min_orig[parent[t]] == orig)
        first[orig] = 1;
}

__global__ void __launch_bounds__(kClusterBlock) cluster_label_kernel(
    GridView g, float r, const uint8_t* __restrict__ core, const uint32_t* __restrict__ parent,
    const uint32_t* __restrict__ min_orig, const uint64_t* __restrict__ number,
    uint32_t* __restrict__ labels)
{
    uint32_t const t = blockIdx.x * kClusterBlock + threadIdx.x;
    if (t >= g.n)
        return;
    float4 const p     = __ldg(g.pts + t);
    uint32_t const src = core[t] ? t : cluster_border_source(g, core, p, r);
    labels[__float_as_uint(p.w)] =
        src == kClusterNone ? kClusterNone : (uint32_t)number[min_orig[parent[src]]];
}

} // namespace

uint64_t launch_cluster_by_density(const pcpx_index& ix, float r, uint32_t min_points,
                                   uint32_t* labels, uint32_t* launches)
{
    uint32_t const n = (uint32_t)ix.n_input, ni = ix.grid.n;
    cudaStream_t const s = ix.qstream();
    PCPX_CUDA(cudaMemsetAsync(labels, 0xFF, (size_t)n * 4, s)); // noise, and every un-indexed point
    DevBuf<uint8_t> core(std::max(ni, 1u)), first(n);
    DevBuf<uint32_t> parent(std::max(ni, 1u)), min_orig(std::max(ni, 1u));
    DevBuf<uint64_t> number(n + 1);
    PCPX_CUDA(cudaMemsetAsync(min_orig.get(), 0xFF, (size_t)ni * 4, s));
    PCPX_CUDA(cudaMemsetAsync(first.get(), 0, n, s));
    uint32_t const blocks = blocks_for(ni);
    cluster_core_kernel<<<blocks, kClusterBlock, 0, s>>>(ix.grid, r, min_points, core.get(),
                                                         parent.get());
    PCPX_CHECK_LAUNCH();
    cluster_union_kernel<<<blocks, kClusterBlock, 0, s>>>(ix.grid, r, core.get(), parent.get());
    PCPX_CHECK_LAUNCH();
    cluster_flatten_kernel<<<blocks, kClusterBlock, 0, s>>>(ix.grid, core.get(), parent.get(),
                                                            min_orig.get());
    PCPX_CHECK_LAUNCH();
    cluster_first_kernel<<<blocks, kClusterBlock, 0, s>>>(ix.grid, core.get(), parent.get(),
                                                          min_orig.get(), first.get());
    PCPX_CHECK_LAUNCH();
    launch_exclusive_scan_u8(ix, first.get(), n, number.get()); // (three kernels)
    cluster_label_kernel<<<blocks, kClusterBlock, 0, s>>>(ix.grid, r, core.get(), parent.get(),
                                                          min_orig.get(), number.get(), labels);
    PCPX_CHECK_LAUNCH();
    uint64_t n_clusters = 0;
    PCPX_CUDA(cudaMemcpyAsync(&n_clusters, number.get() + n, 8, cudaMemcpyDeviceToHost, s));
    PCPX_CUDA(cudaStreamSynchronize(s)); // the temporaries go back to the pool on return
    *launches = 8;
    return n_clusters;
}

} // namespace pcpx
