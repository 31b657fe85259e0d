// Index build, entirely on the device:
//   bbox reduce -> quantise + Morton encode -> hand-written radix sort -> float4 SoA reorder
//   -> per-level cell boundaries -> one hash table of (level, cell) -> [start, count).
// Replaces the sequential pointer-octree insertion of the reference
// (octree/linked_octree_node.hpp:143-331) and the recursive nth_element kd-tree build
// (kdtree/linked_kdtree.hpp:343-424); only the root voxel semantics survive (points outside a
// user-supplied voxel grid are not indexed, octree/linked_octree_node.hpp:174).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <vector>

#include "index.hpp"
#include "radix_sort.cuh"

namespace pcpx {
namespace {

constexpr int kBlock = 256;

inline uint32_t blocks_for(uint64_t n, int per_block) {
    return (uint32_t)std::max<uint64_t>(1, (n + per_block - 1) / per_block);
}

// ---- bbox ----------------------------------------------------------------------------------
// pcp::bounding_box (common/axis_aligned_bounding_box.hpp:214-251): per-axis min / max, which
// is exact in any evaluation order.  Also max |coordinate| (for the float safety margin) and,
// with a user voxel grid, the number of points inside it (inclusive on both ends, :111-124).
struct BBoxPartial
{
    float mn[3], mx[3], maxabs;
    uint32_t inside;
};

__global__ void __launch_bounds__(kBlock) bbox_kernel(
    const float* __restrict__ xyz, uint32_t n, int use_box, float bx0, float by0, float bz0,
    float bx1, float by1, float bz1, BBoxPartial* __restrict__ partials)
{
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    float maxabs    = 0.f;
    uint32_t inside = 0;
    for (uint32_t i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock)
    {
        float const x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
        mn[0] = fminf(mn[0], x), mn[1] = fminf(mn[1], y), mn[2] = fminf(mn[2], z);
        mx[0] = fmaxf(mx[0], x), mx[1] = fmaxf(mx[1], y), mx[2] = fmaxf(mx[2], z);
        maxabs = fmaxf(maxabs, fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z))));
        if (use_box)
            inside += x >= bx0 && y >= by0 && z >= bz0 && x <= bx1 && y <= by1 && z <= bz1;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
#pragma unroll
        for (int a = 0; a < 3; ++a)
        {
            mn[a] = fminf(mn[a], __shfl_xor_sync(0xFFFFFFFFu, mn[a], o));
            mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xFFFFFFFFu, mx[a], o));
        }
        maxabs = fmaxf(maxabs, __shfl_xor_sync(0xFFFFFFFFu, maxabs, o));
        inside += __shfl_xor_sync(0xFFFFFFFFu, inside, o);
    }
    __shared__ BBoxPartial sh[kBlock / 32];
    int const lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0)
    {
        for (int a = 0; a < 3; ++a)
            sh[warp].mn[a] = mn[a], sh[warp].mx[a] = mx[a];
        sh[warp].maxabs = maxabs, sh[warp].inside = inside;
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        BBoxPartial r = sh[0];
        for (int w = 1; w < kBlock / 32; ++w)
        {
            for (int a = 0; a < 3; ++a)
                r.mn[a] = fminf(r.mn[a], sh[w].mn[a]), r.mx[a] = fmaxf(r.mx[a], sh[w].mx[a]);
            r.maxabs = fmaxf(r.maxabs, sh[w].maxabs);
            r.inside += sh[w].inside;
        }
        partials[blockIdx.x] = r;
    }
}

// ---- quantise + Morton ---------------------------------------------------------------------
template <typename KeyT>
__global__ void __launch_bounds__(kBlock) encode_kernel(
    const float* __restrict__ xyz, uint32_t stride_f, uint32_t n, GridView g, int use_box,
    float bx0, float by0, float bz0, float bx1, float by1, float bz1, KeyT* __restrict__ keys,
    uint32_t* __restrict__ vals)
{
    uint32_t const i = blockIdx.x * kBlock + threadIdx.x;
    if (i >= n)
        return;
    float const x = xyz[(size_t)i * stride_f], y = xyz[(size_t)i * stride_f + 1],
                z = xyz[(size_t)i * stride_f + 2];
    bool inside = true;
    if (use_box)
        inside = x >= bx0 && y >= by0 && z >= bz0 && x <= bx1 && y <= by1 && z <= bz1;
    QueryCell const c = query_cell(g, x, y, z);
    uint64_t const m  = morton3(c.ux, c.uy, c.uz);
    // un-indexed points get the first code past the grid: they sort to the tail
    keys[i] = inside ? (KeyT)m : (KeyT)((KeyT)1 << (3 * g.lcap));
    vals[i]           = i;
}

// ---- SoA reorder + cell boundaries ---------------------------------------------------------
// One pass behind the sort: sorted point i is gathered into the float4 array, and — from the
// sorted CODES, so that no thread waits for a neighbour's gather — b(i), the coarsest level at
// which point i opens a new cell, is written and counted per level.  b(i) = 0 for i == 0,
// lcap + 1 when i shares even the finest cell with its predecessor; two Morton codes differ
// first at bit h <=> their coordinates differ first at bit h / 3.  Point i starts a cell at
// every level >= b(i).
template <typename KeyT>
__global__ void __launch_bounds__(kBlock) reorder_levels_kernel(
    const float* __restrict__ xyz, const uint32_t* __restrict__ order,
    const KeyT* __restrict__ codes, uint32_t n, uint32_t n_indexed, int lcap,
    float4* __restrict__ pts, uint8_t* __restrict__ bnd, uint32_t* __restrict__ hist)
{
    __shared__ uint32_t sh[kMaxLevel + 2];
    if (threadIdx.x < kMaxLevel + 2)
        sh[threadIdx.x] = 0;
    __syncthreads();
    // (grid-stride: a few global atomics per block on the ~20 counters, not per 256 points)
    for (uint32_t i = blockIdx.x * kBlock + threadIdx.x; i < n; i += gridDim.x * kBlock)
    {
        uint32_t const o = order[i];
        pts[i] = make_float4(xyz[3 * (size_t)o], xyz[3 * (size_t)o + 1], xyz[3 * (size_t)o + 2],
                             __uint_as_float(o));
        if (i < n_indexed)
        {
            int b = 0;
            if (i > 0)
            {
                uint64_t const diff = (uint64_t)(codes[i - 1] ^ codes[i]);
                b = diff == 0 ? lcap + 1 : lcap - (63 - __clzll((long long)diff)) / 3;
            }
            bnd[i] = (uint8_t)b;
            atomicAdd(&sh[b], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x < kMaxLevel + 2 && sh[threadIdx.x])
        atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// ---- hash table ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t claim_slot(HashSlot* table, uint32_t size, uint64_t key)
{
    uint32_t s = hash_slot(key, size);
    for (;;)
    {
        unsigned long long* kp = reinterpret_cast<unsigned long long*>(table + s);
        unsigned long long const prev = atomicCAS(kp, ~0ull, (unsigned long long)key);
        if (prev == ~0ull || prev == (unsigned long long)key)
            return s;
        s = s + 1 == size ? 0u : s + 1;
    }
}

// One pass over the cell boundaries: point i OPENS its cell at every level >= b(i) (start = i)
// and CLOSES the cell of point i - 1 at the same levels (it ends at i); i == n closes the last
// point's cells at every level.  Either side claims the slot if it comes first.  A slot's count
// starts at 0xFFFFFFFF (the table is cleared to 0xFF bytes): the opener subtracts start, the
// closer adds end + 1, in either order, which leaves count = end - start.
__global__ void __launch_bounds__(kBlock) table_build_kernel(GridView g, HashSlot* table,
                                                             const uint8_t* __restrict__ bnd)
{
    uint32_t const i = blockIdx.x * kBlock + threadIdx.x; // 0 .. n
    if (i > g.n)
        return;
    int const b = i == g.n ? 0 : bnd[i];
    if (b > g.lfine)
        return;
    if (i < g.n)
    {
        float4 const p    = g.pts[i];
        QueryCell const c = query_cell(g, p.x, p.y, p.z);
        for (int l = b; l <= g.lfine; ++l)
        {
            int const sh     = g.lcap - l;
            uint32_t const s = claim_slot(table, g.table_size,
                                          cell_key(l, c.ux >> sh, c.uy >> sh, c.uz >> sh));
            table[s].start   = i;
            atomicSub(&table[s].count, i);
        }
    }
    if (i > 0)
    {
        float4 const p    = g.pts[i - 1];
        QueryCell const c = query_cell(g, p.x, p.y, p.z);
        for (int l = b; l <= g.lfine; ++l)
        {
            int const sh     = g.lcap - l;
            uint32_t const s = claim_slot(table, g.table_size,
                                          cell_key(l, c.ux >> sh, c.uy >> sh, c.uz >> sh));
            atomicAdd(&table[s].count, i + 1u);
        }
    }
}


// ---- radix sort driver ---------------------------------------------------------------------
// Sorts (keys, vals) on bits [0, n_bits); returns true when the result is in the alt buffers.
// `hold` keeps the histogram / offset tables alive until the caller synchronises the stream.
template <typename KeyT, class Holder>
bool sort_pairs(KeyT* keys, uint32_t* vals, KeyT* keys_alt, uint32_t* vals_alt, uint32_t n,
                int n_bits, cudaStream_t stream, uint32_t* launches, Holder& hold)
{
    using namespace rsort;
    int const n_passes = (n_bits + kRadixBits - 1) / kRadixBits;
    if (n == 0 || n_passes == 0)
        return false;
    uint32_t const n_tiles = (n + kTile - 1) / kTile;
    hold.hist.alloc((size_t)n_passes * kRadix);
    if (n >= kLookbackMaxN)
        hold.counts.alloc((size_t)kRadix * n_tiles);
    DevBuf<uint32_t>& hist   = hold.hist;
    DevBuf<uint32_t>& counts = hold.counts;
    PCPX_CUDA(cudaMemsetAsync(hist.get(), 0, hist.bytes(), stream));
    uint32_t const hist_blocks = std::min<uint32_t>(n_tiles, 148u * 8u);
    digit_histograms<KeyT><<<hist_blocks, kThreads, 0, stream>>>(keys, n, 0, n_passes, hist.get());
    PCPX_CHECK_LAUNCH();
    ++*launches;

    size_t const smem = sizeof(ScatterSmem<KeyT>);
    PCPX_CUDA(cudaFuncSetAttribute(scatter<KeyT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)smem));
    PCPX_CUDA(cudaFuncSetAttribute(scatter_lookback<KeyT>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bool const lookback = n < kLookbackMaxN;
    if (lookback)
    {
        // per pass: [n_tiles][256] state words + one ticket, all zero
        size_t const per_pass = (size_t)n_tiles * kRadix + 1;
        hold.counts.alloc(per_pass * (size_t)n_passes);
        PCPX_CUDA(cudaMemsetAsync(hold.counts.get(), 0, hold.counts.bytes(), stream));
    }
    bool in_alt = false;
    for (int p = 0; p < n_passes; ++p)
    {
        KeyT* kin      = in_alt ? keys_alt : keys;
        uint32_t* vin  = in_alt ? vals_alt : vals;
        KeyT* kout     = in_alt ? keys : keys_alt;
        uint32_t* vout = in_alt ? vals : vals_alt;
        int const shift = p * kRadixBits;
        if (lookback)
        {
            uint32_t* state = hold.counts.get() + ((size_t)n_tiles * kRadix + 1) * (size_t)p;
            scatter_lookback<KeyT><<<n_tiles, kThreads, smem, stream>>>(
                kin, vin, kout, vout, n, shift, hist.get() + (size_t)p * kRadix, state,
                state + (size_t)n_tiles * kRadix);
            PCPX_CHECK_LAUNCH();
            *launches += 1;
            in_alt = !in_alt;
            continue;
        }
        tile_histogram<KeyT><<<n_tiles, kThreads, 0, stream>>>(kin, n, shift, n_tiles, counts.get());
        PCPX_CHECK_LAUNCH();
        tile_offsets<<<kRadix, kThreads, 0, stream>>>(counts.get(), n_tiles,
                                                       hist.get() + (size_t)p * kRadix);
        PCPX_CHECK_LAUNCH();
        scatter<KeyT><<<n_tiles, kThreads, smem, stream>>>(kin, vin, kout, vout, n, shift, n_tiles,
                                                            counts.get());
        PCPX_CHECK_LAUNCH();
        *launches += 3;
        in_alt = !in_alt;
    }
    return in_alt;
}

constexpr int kShortLevelCap = 10; // 3 x 10 bits + the "outside" flag fit a 32-bit sort key

int auto_level_cap(uint64_t n, float extent, float maxabs, uint32_t user_max)
{
    // enough levels that a 2-manifold of n points still reaches ~1 point per finest cell
    int lcap = (int)std::ceil(std::log2((double)std::max<uint64_t>(n, 2)) / 2.0) + 1;
    if (user_max)
        lcap = (int)user_max;
    // cells must stay well above the fp32 resolution of the coordinates (>= 64 ulps)
    double const ulp = std::max((double)maxabs, (double)extent) * std::ldexp(1.0, -23);
    int const by_res = (int)std::floor(std::log2((double)extent / (64.0 * ulp)));
    lcap             = std::min(lcap, by_res);
    return std::max(1, std::min(lcap, kMaxLevel));
}

} // namespace

// --------------------------------------------------------------------------------------------
// Temporaries of the sort; kept alive by the caller until the stream has been synchronised.
struct SortScratch
{
    DevBuf<unsigned char> keys, keys_alt;
    DevBuf<uint32_t> vals, vals_alt;
    DevBuf<uint32_t> hist, counts;
    bool in_alt = false;
    uint32_t* order() { return in_alt ? vals_alt.get() : vals.get(); }
};

template <typename KeyT>
static void encode_and_sort(pcpx_index& ix, const float* d_xyz, uint32_t n,
                            const pcpx_index_params& prm, SortScratch& sc, uint32_t* launches,
                            Event& e0, Event& e1)
{
    sc.keys.alloc((size_t)n * sizeof(KeyT));
    sc.keys_alt.alloc((size_t)n * sizeof(KeyT));
    sc.vals.alloc(n);
    sc.vals_alt.alloc(n);
    KeyT* keys     = reinterpret_cast<KeyT*>(sc.keys.get());
    KeyT* keys_alt = reinterpret_cast<KeyT*>(sc.keys_alt.get());
    encode_kernel<KeyT><<<blocks_for(n, kBlock), kBlock, 0, ix.stream>>>(
        d_xyz, 3u, n, ix.grid, prm.use_voxel_grid, prm.voxel_min[0], prm.voxel_min[1],
        prm.voxel_min[2], prm.voxel_max[0], prm.voxel_max[1], prm.voxel_max[2], keys,
        sc.vals.get());
    PCPX_CHECK_LAUNCH();
    ++*launches;
    e0.record(ix.stream);
    int const bits = 3 * ix.grid.lcap + (prm.use_voxel_grid ? 1 : 0);
    sc.in_alt = sort_pairs<KeyT>(keys, sc.vals.get(), keys_alt, sc.vals_alt.get(), n, bits,
                                 ix.stream, launches, sc);
    e1.record(ix.stream);
}

pcpx_index* build_index(const float* xyz, size_t n, size_t stride_bytes,
                        const pcpx_index_params* params)
{
    pcpx_index_params prm{};
    if (params)
        prm = *params;
    if (n >= 0xFFFFFFFFull)
        fail(PCPX_ERR_UNSUPPORTED, "clouds of 2^32 - 1 points or more need 64-bit indices");
    if (n && !xyz)
        fail(PCPX_ERR_INVALID_ARG, "xyz is NULL");
    if (stride_bytes == 0)
        stride_bytes = 12;
    if (stride_bytes < 12 || stride_bytes % 4)
        fail(PCPX_ERR_INVALID_ARG, "stride_bytes must be a multiple of 4 and >= 12");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        fail(PCPX_ERR_NO_DEVICE, "no CUDA device: libpcpx has no CPU path");
    int dev = prm.device;
    if (dev < 0)
        PCPX_CUDA(cudaGetDevice(&dev));
    if (dev >= ndev)
        fail(PCPX_ERR_INVALID_ARG, "device %d out of range (%d devices)", dev, ndev);
    ScopedDevice guard(dev);

    std::unique_ptr<pcpx_index> ixp(new pcpx_index());
    pcpx_index& ix = *ixp;
    ix.device      = dev;
    ix.n_input     = n;
    PCPX_CUDA(cudaStreamCreateWithFlags(&ix.stream, cudaStreamNonBlocking));
    uint32_t launches = 0;
    Event ev_begin, ev_end;
    ev_begin.record(ix.stream);

    uint32_t const n32 = (uint32_t)n;

    // 1. packed device copy of the cloud (12-byte stride)
    DevBuf<float> staged;
    const float* d_xyz = nullptr;
    bool const on_device = is_device_pointer(xyz);
    if (on_device && stride_bytes == 12)
        d_xyz = xyz;
    else if (n)
    {
        staged.alloc(3 * n);
        cudaMemcpyKind const kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        if (stride_bytes == 12) // packed rows: one DMA, not one per row
            PCPX_CUDA(cudaMemcpyAsync(staged.get(), xyz, 12 * n, kind, ix.stream));
        else
            PCPX_CUDA(cudaMemcpy2DAsync(staged.get(), 12, xyz, stride_bytes, 12, n, kind,
                                        ix.stream));
        d_xyz = staged.get();
    }

    // 2. bounding box
    BBoxPartial bb{};
    for (int a = 0; a < 3; ++a)
        bb.mn[a] = INFINITY, bb.mx[a] = -INFINITY;
    if (n)
    {
        uint32_t const nb = std::min<uint32_t>(blocks_for(n, kBlock * 8), 148u * 8u);
        DevBuf<BBoxPartial> partials(nb);
        bbox_kernel<<<nb, kBlock, 0, ix.stream>>>(
            d_xyz, n32, prm.use_voxel_grid, prm.voxel_min[0], prm.voxel_min[1], prm.voxel_min[2],
            prm.voxel_max[0], prm.voxel_max[1], prm.voxel_max[2], partials.get());
        PCPX_CHECK_LAUNCH();
        ++launches;
        std::vector<BBoxPartial> h(nb);
        read_back(ix.stream, h.data(), partials.get(), partials.bytes());
        for (auto const& p : h)
        {
            for (int a = 0; a < 3; ++a)
                bb.mn[a] = std::min(bb.mn[a], p.mn[a]), bb.mx[a] = std::max(bb.mx[a], p.mx[a]);
            bb.maxabs = std::max(bb.maxabs, p.maxabs);
            bb.inside += p.inside;
        }
    }
    if (prm.use_voxel_grid)
    {
        for (int a = 0; a < 3; ++a)
            ix.bbox_min[a] = prm.voxel_min[a], ix.bbox_max[a] = prm.voxel_max[a];
        ix.n_indexed = bb.inside;
    }
    else
    {
        for (int a = 0; a < 3; ++a)
            ix.bbox_min[a] = n ? bb.mn[a] : 0.f, ix.bbox_max[a] = n ? bb.mx[a] : 0.f;
        ix.n_indexed = n;
    }

    // 3. root cube and level cap
    float extent = 0.f, maxabs = 0.f;
    for (int a = 0; a < 3; ++a)
    {
        extent = std::max(extent, ix.bbox_max[a] - ix.bbox_min[a]);
        maxabs = std::max(maxabs, std::max(std::fabs(ix.bbox_min[a]), std::fabs(ix.bbox_max[a])));
    }
    if (!(extent > 0.f) || !std::isfinite(extent))
        extent = maxabs > 0.f && std::isfinite(maxabs) ? maxabs * 1e-3f : 1.f;
    extent *= 1.0001f; // the max corner falls strictly inside the last cell
    GridView& g = ix.grid;
    g.ox = ix.bbox_min[0], g.oy = ix.bbox_min[1], g.oz = ix.bbox_min[2];
    g.extent = extent;
    int const lcap_full =
        auto_level_cap(std::max<uint64_t>(ix.n_indexed, 1), extent, maxabs, prm.max_level);
    g.delta = 16.f * std::ldexp(std::max(extent, maxabs), -23);
    g.n     = (uint32_t)ix.n_indexed;
    // Ten levels fit a 32-bit sort key (4 radix passes over 8-byte pairs instead of 5 over
    // 12-byte pairs: 1.03 ms against 1.28 ms for 10 M points) and are as many as most clouds of
    // up to 2^24 points use.  So such a cloud is first indexed with 10 levels; if the cell counts
    // then say that an 11th level would still have held min_occ points per cell, the build is
    // repeated with the full code length.  Nothing downstream depends on the choice: the
    // levels above the cap are simply never stored.
    bool const try_short = prm.max_level == 0 && lcap_full > kShortLevelCap && ix.n_indexed > 0 &&
                           ix.n_indexed <= (1u << 24);
    double const min_occ = prm.min_cell_occupancy ? (double)prm.min_cell_occupancy : 4.0;
    float sort_ms        = 0.f;
    uint64_t total_cells = 0;
    for (int attempt = 0;; ++attempt)
    {
        g.lcap       = try_short && attempt == 0 ? kShortLevelCap : lcap_full;
        g.scale      = std::ldexp(1.f, g.lcap) / extent;
        g.lfine      = 0;
        ix.code_bits = 3u * (uint32_t)g.lcap;

        // 4. codes -> sort -> SoA
        // kPtsPad readable entries behind the last point: the kNN walk loads up to three entries
        // past the end of a span without a bounds test (knn_core.cuh: knn_scan_dist)
        ix.pts.alloc(n + kPtsPad);
        PCPX_CUDA(cudaMemsetAsync(ix.pts.get() + n, 0, kPtsPad * sizeof(float4), ix.stream));
        g.pts = ix.pts.get();
        SortScratch sc;
        Event ev_sort0, ev_sort1;
        if (n)
        {
            if (ix.code_bits + 1 <= 32)
                encode_and_sort<uint32_t>(ix, d_xyz, n32, prm, sc, &launches, ev_sort0, ev_sort1);
            else
                encode_and_sort<uint64_t>(ix, d_xyz, n32, prm, sc, &launches, ev_sort0, ev_sort1);
        }

        // 5. SoA + cells per level -> finest stored level
        std::vector<uint32_t> lh(kMaxLevel + 2, 0u);
        if (n)
        {
            DevBuf<uint32_t> d_lh(kMaxLevel + 2);
            PCPX_CUDA(cudaMemsetAsync(d_lh.get(), 0, d_lh.bytes(), ix.stream));
            ix.bnd.alloc(std::max<uint32_t>(g.n, 1u));
            uint32_t const reorder_blocks = std::min<uint32_t>(blocks_for(n, kBlock), 148u * 8u);
            const void* codes = sc.in_alt ? (const void*)sc.keys_alt.get() : (const void*)sc.keys.get();
            if (ix.code_bits + 1 <= 32)
                reorder_levels_kernel<uint32_t><<<reorder_blocks, kBlock, 0, ix.stream>>>(
                    d_xyz, sc.order(), static_cast<const uint32_t*>(codes), n32, g.n, g.lcap,
                    ix.pts.get(), ix.bnd.get(), d_lh.get());
            else
                reorder_levels_kernel<uint64_t><<<reorder_blocks, kBlock, 0, ix.stream>>>(
                    d_xyz, sc.order(), static_cast<const uint64_t*>(codes), n32, g.n, g.lcap,
                    ix.pts.get(), ix.bnd.get(), d_lh.get());
            PCPX_CHECK_LAUNCH();
            ++launches;
            read_back(ix.stream, lh.data(), d_lh.get(), d_lh.bytes());
        }
        else
            PCPX_CUDA(cudaStreamSynchronize(ix.stream));
        sort_ms += n ? elapsed_ms(ev_sort0, ev_sort1) : 0.f;
        // the stream is idle: the sort temporaries go when `sc` leaves scope
        uint64_t cells = 0;
        total_cells    = 0;
        for (int l = 0; l <= kMaxLevel; ++l)
            ix.cells_per_level[l] = 0;
        for (int l = 0; l <= g.lcap; ++l)
        {
            cells += lh[l]; // cells at level l = points that open a cell at a level <= l
            if (l > 0 && (double)g.n / (double)std::max<uint64_t>(cells, 1) < min_occ)
                break;
            g.lfine = l;
            ix.cells_per_level[l] = cells;
            total_cells += cells;
        }
        if (try_short && attempt == 0 && g.lfine == g.lcap)
        {
            // cells grow by the factor of the last step once more (x4 on a surface, x8 in a
            // volume): would level lcap + 1 have been stored?
            double const c1     = (double)ix.cells_per_level[g.lcap];
            double const c0     = (double)std::max<uint64_t>(ix.cells_per_level[g.lcap - 1], 1);
            double const growth = std::min(8.0, std::max(1.0, c1 / c0));
            if ((double)g.n / (c1 * growth) >= min_occ)
                continue; // yes: index again with the full code length
        }
        break;
    }
    staged.release();
    ix.n_cells = total_cells;

    // 6. hash table over all stored levels
    uint64_t const slots = std::max<uint64_t>(64, (uint64_t)((double)total_cells * 2.5) + 1);
    if (slots >= 0xFFFFFFFFull)
        fail(PCPX_ERR_UNSUPPORTED, "cell table too large");
    g.table_size = (uint32_t)slots;
    ix.table.alloc(slots);
    g.table = ix.table.get();
    PCPX_CUDA(cudaMemsetAsync(ix.table.get(), 0xFF, ix.table.bytes(), ix.stream));
    if (g.n)
    {
        table_build_kernel<<<blocks_for(g.n + 1u, kBlock), kBlock, 0, ix.stream>>>(g, ix.table.get(),
                                                                                   ix.bnd.get());
        PCPX_CHECK_LAUNCH();
        launches += 1;
    }
    ev_end.record(ix.stream);
    PCPX_CUDA(cudaStreamSynchronize(ix.stream));
    ix.timings.build_ms        = elapsed_ms(ev_begin, ev_end);
    ix.timings.sort_ms         = sort_ms;
    ix.timings.total_ms        = ix.timings.build_ms;
    ix.timings.kernel_launches = launches;
    return ixp.release();
}

void sort_queries_by_cell(const pcpx_index& ix, const float* d_queries, uint32_t stride_floats,
                          uint32_t nq, uint32_t* d_order, uint32_t* n_launched)
{
    // Morton order of the queries' own fine cells: neighbouring threads walk neighbouring cells.
    if (nq == 0)
        return;
    uint32_t launches = 0;
    SortScratch sc;
    sc.keys.alloc((size_t)nq * 8);
    sc.keys_alt.alloc((size_t)nq * 8);
    sc.vals_alt.alloc(nq);
    uint64_t* keys     = reinterpret_cast<uint64_t*>(sc.keys.get());
    uint64_t* keys_alt = reinterpret_cast<uint64_t*>(sc.keys_alt.get());
    encode_kernel<uint64_t><<<blocks_for(nq, kBlock), kBlock, 0, ix.qstream()>>>(
        d_queries, stride_floats, nq, ix.grid, 0, 0, 0, 0, 0, 0, 0, keys, d_order);
    PCPX_CHECK_LAUNCH();
    bool const alt = sort_pairs<uint64_t>(keys, d_order, keys_alt, sc.vals_alt.get(), nq,
                                          3 * ix.grid.lcap, ix.qstream(), &launches, sc);
    if (alt)
        PCPX_CUDA(cudaMemcpyAsync(d_order, sc.vals_alt.get(), (size_t)nq * 4,
                                  cudaMemcpyDeviceToDevice, ix.qstream()));
    PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
    if (n_launched)
        *n_launched += 1 + launches; // the encode kernel + the sort's
}

void sort_pairs_u64(const pcpx_index& ix, uint64_t* keys, uint32_t* vals, uint32_t n, int n_bits,
                    uint32_t* launches)
{
    if (n == 0)
        return;
    SortScratch sc;
    sc.keys_alt.alloc((size_t)n * 8);
    sc.vals_alt.alloc(n);
    uint64_t* keys_alt = reinterpret_cast<uint64_t*>(sc.keys_alt.get());
    bool const alt = sort_pairs<uint64_t>(keys, vals, keys_alt, sc.vals_alt.get(), n, n_bits,
                                          ix.qstream(), launches, sc);
    if (alt)
    {
        PCPX_CUDA(cudaMemcpyAsync(keys, keys_alt, (size_t)n * 8, cudaMemcpyDeviceToDevice,
                                  ix.qstream()));
        PCPX_CUDA(cudaMemcpyAsync(vals, sc.vals_alt.get(), (size_t)n * 4, cudaMemcpyDeviceToDevice,
                                  ix.qstream()));
    }
    PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // the scratch is freed on return
}

} // namespace pcpx
