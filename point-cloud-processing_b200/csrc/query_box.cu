// Axis-aligned box range search (pcpx_box_count, pcpx_box_search): one box per warp over the
// traversal of box_core.cuh.  A round looks up to 32 cells at once (one per lane); INSIDE cells
// add their span without a point being read; the points of PARTIAL leaves are spread over the
// lanes, 32 per step, and compacted in order with a ballot.  The fill copies short INSIDE spans
// itself and hands long ones to a grid-wide copy as fixed-size records, so that a box of millions
// of points is not one warp's work.
#include <algorithm>

#include "box_core.cuh"
#include "query.hpp"

namespace pcpx {

namespace {

constexpr int kBoxWarps        = 4; // boxes per CTA
constexpr uint32_t kBoxFull    = 0xFFFFFFFFu;
constexpr uint32_t kShortLists = 64; // longest list left to sort_lists_kernel (insertion sort)

struct BoxRecord
{
    uint32_t src, len; // sorted positions [src, src + len)
    uint64_t dst;      // ... are written to idx[dst ..]
};

struct BoxOut
{
    uint32_t* idx;     // the call's lists
    uint64_t base;     // this box's offset
    BoxRecord* rec;    // records of the grid-wide copy
    uint32_t* n_rec;   // ... and their count
};

uint32_t blocks_of(uint64_t n, uint32_t per_block)
{
    return (uint32_t)std::max<uint64_t>(1, (n + per_block - 1) / per_block);
}

// The traversal of box_visit (box_core.cuh) by one warp; returns the box's result count.  FILL:
// the results are written at o.idx[o.base ..] in the order of box_visit.
template <bool FILL>
__device__ __forceinline__ uint32_t box_warp_walk(const GridView& g, const BoxQ& b, uint64_t* st,
                                                  int lane, BoxOut const& o)
{
    uint32_t n_out = 0;
    if (b.empty)
        return 0;
    uint32_t c0[3];
    int const l0 = box_start(g, b, c0);
    uint64_t key = 0;
    bool valid   = box_start_cell(g, b, l0, c0, lane, key);
    int sp       = 0;
    for (;;)
    {
        bool const room = sp + 32 <= kBoxStackCap;
        uint32_t start = 0, count = 0;
        BoxKind const kind = valid ? box_cell(g, b, key, room, start, count) : kBoxNone;

        // ---- INSIDE spans, lane order ----
        if (!FILL)
            n_out += __reduce_add_sync(kBoxFull, kind == kBoxInside ? count : 0u);
        else
            for (uint32_t mm = __ballot_sync(kBoxFull, kind == kBoxInside); mm != 0u; mm &= mm - 1u)
            {
                int const j        = __ffs((int)mm) - 1;
                uint32_t const s   = __shfl_sync(kBoxFull, start, j);
                uint32_t const c   = __shfl_sync(kBoxFull, count, j);
                uint64_t const dst = o.base + n_out;
                if (c >= kBoxBigSpan)
                {
                    uint32_t const nr = (c + kBoxChunk - 1u) / kBoxChunk;
                    uint32_t r0       = 0;
                    if (lane == 0)
                        r0 = atomicAdd(o.n_rec, nr);
                    r0 = __shfl_sync(kBoxFull, r0, 0);
                    for (uint32_t r = (uint32_t)lane; r < nr; r += 32u)
                    {
                        uint32_t const off = r * kBoxChunk;
                        o.rec[r0 + r]      = BoxRecord{s + off, min(kBoxChunk, c - off), dst + off};
                    }
                }
                else
                    for (uint32_t i = (uint32_t)lane; i < c; i += 32u)
                        o.idx[dst + i] = __float_as_uint(__ldg(&g.pts[s + i].w));
                n_out += c;
            }

        // ---- PARTIAL leaves: their points spread over the lanes, 32 per step ----
        uint32_t const cnt = kind == kBoxLeaf ? count : 0u;
        uint32_t incl      = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1)
        {
            uint32_t const up = __shfl_up_sync(kBoxFull, incl, d);
            if (lane >= d)
                incl += up;
        }
        uint32_t const excl = incl - cnt, total = __shfl_sync(kBoxFull, incl, 31);
        for (uint32_t base = 0; base < total; base += 32u)
        {
            uint32_t const f = base + (uint32_t)lane;
            int src          = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1)
            {
                uint32_t const v = __shfl_sync(kBoxFull, excl, src + step);
                src += v <= f ? step : 0;
            }
            uint32_t const s = __shfl_sync(kBoxFull, start, src);
            uint32_t const e = __shfl_sync(kBoxFull, excl, src);
            bool hit         = false;
            float4 c         = make_float4(0.f, 0.f, 0.f, 0.f);
            if (f < total)
            {
                c   = load_pt(g.pts + s + (f - e));
                hit = box_contains(b, c);
            }
            uint32_t const m = __ballot_sync(kBoxFull, hit);
            if (FILL && hit)
                o.idx[o.base + n_out + (uint32_t)__popc(m & ((1u << lane) - 1u))] = __float_as_uint(c.w);
            n_out += (uint32_t)__popc(m);
        }

        // ---- the other PARTIAL cells on the stack, the lowest lane on top ----
        uint32_t const im = __ballot_sync(kBoxFull, kind == kBoxInner);
        if (kind == kBoxInner)
            st[sp + __popc(lane == 31 ? 0u : im >> (lane + 1))] = key;
        sp += __popc(im);
        __syncwarp();
        if (sp == 0)
            break;
        int const P = sp < kBoxParents ? sp : kBoxParents;
        valid       = (lane >> 3) < P;
        if (valid)
            key = box_child_key(st[sp - 1 - (lane >> 3)], lane & 7);
        sp -= P;
        __syncwarp();
    }
    return n_out;
}

__device__ __forceinline__ BoxQ fetch_box(const GridView& g, const BoxBatch& bx, uint32_t box)
{
    return box_prepare(g, bx.boxes + (size_t)box * bx.stride_f, bx.bb);
}

__global__ void __launch_bounds__(kBoxWarps * 32) box_count_kernel(
    GridView g, BoxBatch bx, uint32_t* __restrict__ count, uint32_t* __restrict__ max_count)
{
    __shared__ uint64_t stack[kBoxWarps][kBoxStackCap];
    int const lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t const box = blockIdx.x * kBoxWarps + (uint32_t)w;
    if (box >= bx.nb)
        return;
    BoxQ const b     = fetch_box(g, bx, box);
    uint32_t const c = box_warp_walk<false>(g, b, stack[w], lane, BoxOut{});
    if (lane == 0)
    {
        count[box] = c;
        if (max_count)
            atomicMax(max_count, c);
    }
}

__global__ void __launch_bounds__(kBoxWarps * 32) box_fill_kernel(
    GridView g, BoxBatch bx, const uint64_t* __restrict__ offsets, uint32_t* __restrict__ idx,
    BoxRecord* __restrict__ rec, uint32_t* __restrict__ n_rec)
{
    __shared__ uint64_t stack[kBoxWarps][kBoxStackCap];
    int const lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t const box = blockIdx.x * kBoxWarps + (uint32_t)w;
    if (box >= bx.nb)
        return;
    BoxQ const b = fetch_box(g, bx, box);
    box_warp_walk<true>(g, b, stack[w], lane, BoxOut{idx, offsets[box], rec, n_rec});
}

// the long INSIDE spans: one record (<= kBoxChunk points) per CTA at a time
__global__ void __launch_bounds__(256) box_copy_kernel(const float4* __restrict__ pts,
                                                       const BoxRecord* __restrict__ rec,
                                                       const uint32_t* __restrict__ n_rec,
                                                       uint32_t* __restrict__ idx)
{
    uint32_t const nr = *n_rec;
    for (uint32_t r = blockIdx.x; r < nr; r += gridDim.x)
    {
        BoxRecord const e = rec[r];
        for (uint32_t i = threadIdx.x; i < e.len; i += 256u)
            idx[e.dst + i] = __float_as_uint(__ldg(&pts[e.src + i].w));
    }
}

// sort keys of the lists: (list << 32) | value, one warp per list
__global__ void __launch_bounds__(128) box_sort_keys_kernel(const uint64_t* __restrict__ offsets,
                                                            uint32_t nb,
                                                            const uint32_t* __restrict__ idx,
                                                            uint64_t* __restrict__ keys)
{
    uint32_t const box = blockIdx.x * 4u + (threadIdx.x >> 5);
    if (box >= nb)
        return;
    uint64_t const a = offsets[box], e = offsets[box + 1];
    for (uint64_t i = a + (threadIdx.x & 31); i < e; i += 32u)
        keys[i] = ((uint64_t)box << 32) | idx[i];
}

} // namespace

void launch_box_count(const pcpx_index& ix, const BoxBatch& bx, uint32_t* count,
                      uint32_t* max_count)
{
    if (bx.nb == 0)
        return;
    box_count_kernel<<<blocks_of(bx.nb, kBoxWarps), kBoxWarps * 32, 0, ix.qstream()>>>(
        ix.grid, bx, count, max_count);
    PCPX_CHECK_LAUNCH();
}

uint32_t launch_box_fill(const pcpx_index& ix, const BoxBatch& bx, const uint64_t* offsets,
                         uint64_t total, uint32_t* idx)
{
    if (bx.nb == 0 || total == 0)
        return 0;
    // A span of L >= kBoxBigSpan points makes ceil(L / kBoxChunk) <= L / kBoxChunk + L /
    // kBoxBigSpan records, and the spans of the call are at most `total` points in all.
    uint64_t const cap = total / kBoxChunk + total / kBoxBigSpan + 2;
    DevBuf<BoxRecord> rec(cap);
    DevBuf<uint32_t> n_rec(1);
    PCPX_CUDA(cudaMemsetAsync(n_rec.get(), 0, 4, ix.qstream()));
    box_fill_kernel<<<blocks_of(bx.nb, kBoxWarps), kBoxWarps * 32, 0, ix.qstream()>>>(
        ix.grid, bx, offsets, idx, rec.get(), n_rec.get());
    PCPX_CHECK_LAUNCH();
    uint32_t const copy_blocks = (uint32_t)std::min<uint64_t>(cap, 148u * 16u);
    box_copy_kernel<<<copy_blocks, 256, 0, ix.qstream()>>>(ix.grid.pts, rec.get(), n_rec.get(), idx);
    PCPX_CHECK_LAUNCH();
    PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // the records are freed on return
    return 2;
}

uint32_t launch_box_sort(const pcpx_index& ix, const uint64_t* offsets, uint32_t nb,
                         uint64_t total, uint32_t max_count, uint32_t* idx)
{
    if (nb == 0 || max_count < 2)
        return 0;
    if (max_count <= kShortLists)
    {
        launch_sort_lists(ix, offsets, nb, idx);
        return 1;
    }
    // Long lists: one radix sort of (list, value) keys over the whole output.  Lists are
    // contiguous and in list order already, so sorting by the pair sorts every list in place.
    if (total >= 0xFFFFFFFFull)
        fail(PCPX_ERR_UNSUPPORTED, "sorting more than 2^32 - 2 box results in one call");
    DevBuf<uint64_t> keys(total);
    box_sort_keys_kernel<<<blocks_of(nb, 4), 128, 0, ix.qstream()>>>(offsets, nb, idx, keys.get());
    PCPX_CHECK_LAUNCH();
    uint32_t launches = 1;
    int const list_bits = nb > 1 ? 32 - __builtin_clz(nb - 1u) : 0;
    sort_pairs_u64(ix, keys.get(), idx, (uint32_t)total, 32 + list_bits, &launches);
    return launches;
}

} // namespace pcpx
