// Axis-aligned box range search over the multi-level grid.  Predicate:
// pcp::axis_aligned_bounding_box_t::contains (common/axis_aligned_bounding_box.hpp:99-149),
// min <= p <= max on every axis in fp32, inclusive on both ends.
//
// Cells are classified in QUANTISED coordinates, not against float faces.  A point's fine
// coordinate u = quantise(x) (grid_core.cuh) is monotone in x, so with lo = quantise(min) and
// hi = quantise(max):
//   u < lo  =>  x < min        u > lo  =>  x > min   (x <= min would give u <= lo)
//   u > hi  =>  x > max        u < hi  =>  x < max
// A cell whose fine range lies strictly between lo and hi on every axis therefore holds only
// points inside the box (INSIDE: its span is emitted without reading a point), a cell whose range
// misses [lo, hi] on some axis holds none (OUTSIDE), and only the cells that share a fine cell
// with a face of the box (PARTIAL) need the per-point test.  Nothing is evaluated on nominal
// faces, so no float slack is involved and the decisions are exact.  A bound that every indexed
// point satisfies (min <= bbox min, max >= bbox max) is unbounded on that side, so that a box
// covering the cloud is the root cell, INSIDE, one span.
//
// The traversal is shared by the device kernels (query_box.cu: one box per warp) and the host
// emulation of the tests (box_visit below), which run the same rounds in the same order:
//   * round 0 looks up the start batch: the <= 2 x 2 x 2 cells of the finest stored level at which
//     the box's fine range spans at most two cells per axis;
//   * every later round pops up to kBoxParents cells off a stack and looks up their 8 children,
//     lane 8 q + j <-> child j (x lowest) of the q-th cell from the top;
//   * in a round, INSIDE spans are emitted in lane order, then the hits of the PARTIAL leaves
//     (finest level, <= kBoxLeafSize points, or no room left on the stack) in lane order, points
//     of a leaf in sorted order; the other PARTIAL cells are pushed, the lowest lane on top.
#pragma once
#include "grid_core.cuh"

namespace pcpx {

constexpr int kBoxParents        = 4;   // cells opened per round (8 children each)
constexpr int kBoxStackCap       = 256; // cells waiting to be opened, per box
constexpr uint32_t kBoxLeafSize  = 32;  // a PARTIAL cell this small is tested point by point
constexpr uint32_t kBoxBigSpan   = 256; // INSIDE spans this long go to the grid-wide copy ...
constexpr uint32_t kBoxChunk     = 4096; // ... as records of at most this many points

enum BoxKind : int
{
    kBoxNone   = 0, // outside the box, or not in the table
    kBoxInside = 1, // whole span in the box
    kBoxLeaf   = 2, // PARTIAL, points tested one by one
    kBoxInner  = 3  // PARTIAL, opened in a later round
};

struct BoxQ
{
    float mn[3], mx[3]; // the box
    int32_t lo[3], hi[3]; // quantised bounds; -1 / 2^lcap: every indexed point satisfies that side
    bool empty;           // NaN bound or min > max on some axis: no traversal at all
};

// `bb`: a box that every indexed point lies in (the index's bounding box or voxel grid)
PCPX_HD BoxQ box_prepare(const GridView& g, const float* box, const float* bb)
{
    BoxQ b;
    float const o[3] = {g.ox, g.oy, g.oz};
    b.empty          = false;
    for (int a = 0; a < 3; ++a)
    {
        b.mn[a] = box[a], b.mx[a] = box[3 + a];
        b.empty = b.empty || !(b.mn[a] <= b.mx[a]); // also every NaN bound
        b.lo[a] = b.mn[a] <= bb[a] ? -1 : (int32_t)quantise(b.mn[a], o[a], g.scale, g.lcap);
        b.hi[a] = b.mx[a] >= bb[3 + a] ? (int32_t)(1u << g.lcap)
                                        : (int32_t)quantise(b.mx[a], o[a], g.scale, g.lcap);
    }
    b.empty = b.empty || g.n == 0;
    return b;
}

PCPX_HD bool box_contains(const BoxQ& b, float4 const& p)
{
    return p.x >= b.mn[0] && p.y >= b.mn[1] && p.z >= b.mn[2] && p.x <= b.mx[0] &&
           p.y <= b.mx[1] && p.z <= b.mx[2];
}

// finest stored level at which the box's fine range [max(lo, 0), min(hi, 2^lcap - 1)] spans at
// most two cells per axis; `c0`: the range's first cell there
PCPX_HD int box_start(const GridView& g, const BoxQ& b, uint32_t c0[3])
{
    int32_t const top = (int32_t)(1u << g.lcap) - 1;
    int l             = g.lfine;
    for (;; --l)
    {
        int const s = g.lcap - l;
        bool ok     = true;
        for (int a = 0; a < 3; ++a)
        {
            uint32_t const lo = (uint32_t)(b.lo[a] < 0 ? 0 : b.lo[a]);
            uint32_t const hi = (uint32_t)(b.hi[a] > top ? top : b.hi[a]);
            ok = ok && (hi >> s) - (lo >> s) <= 1u;
            c0[a] = lo >> s;
        }
        if (ok || l == 0)
            return l;
    }
}

// lane j < 8 of round 0: the start cell c0 + (j & 1, j >> 1 & 1, j >> 2); false when that cell
// lies past the box's range (or the grid)
PCPX_HD bool box_start_cell(const GridView& g, const BoxQ& b, int l, const uint32_t c0[3], int j,
                            uint64_t& key)
{
    if (j >= 8)
        return false;
    int const s      = g.lcap - l;
    int32_t const top = (int32_t)(1u << g.lcap) - 1;
    uint32_t c[3];
    for (int a = 0; a < 3; ++a)
    {
        c[a]              = c0[a] + (uint32_t)((j >> a) & 1);
        uint32_t const hi = (uint32_t)(b.hi[a] > top ? top : b.hi[a]);
        if (c[a] > (hi >> s))
            return false;
    }
    key = cell_key(l, c[0], c[1], c[2]);
    return true;
}

// child j (x lowest) of the cell `parent`
PCPX_HD uint64_t box_child_key(uint64_t parent, int j)
{
    int const l       = (int)(parent >> 57) + 1;
    uint32_t const cx = 2u * (uint32_t)(parent & 0x7FFFFu) + (uint32_t)(j & 1),
                   cy = 2u * (uint32_t)((parent >> 19) & 0x7FFFFu) + (uint32_t)((j >> 1) & 1),
                   cz = 2u * (uint32_t)((parent >> 38) & 0x7FFFFu) + (uint32_t)((j >> 2) & 1);
    return cell_key(l, cx, cy, cz);
}

// class of the cell `key` against the box: OUTSIDE cells are not looked up
PCPX_HD BoxKind box_cell(const GridView& g, const BoxQ& b, uint64_t key, bool room,
                         uint32_t& start, uint32_t& count)
{
    int const l = (int)(key >> 57), s = g.lcap - l;
    bool inside = true;
    for (int a = 0; a < 3; ++a)
    {
        int32_t const c  = (int32_t)((key >> (19 * a)) & 0x7FFFFu);
        int32_t const f0 = c << s, f1 = f0 + (1 << s) - 1; // the cell's fine range on axis a
        if (f1 < b.lo[a] || f0 > b.hi[a])
            return kBoxNone;
        inside = inside && f0 > b.lo[a] && f1 < b.hi[a];
    }
    start = 0, count = 0;
    if (!find_cell(g, key, start, count))
        return kBoxNone;
    if (inside)
        return kBoxInside;
    return (l >= g.lfine || count <= kBoxLeafSize || !room) ? kBoxLeaf : kBoxInner;
}

// The traversal one box at a time, in the order of the device kernels (see the top of the file):
// span(start, count) for every INSIDE span, point(p) for every hit of a PARTIAL leaf (p = sorted
// position).  `stack`: kBoxStackCap entries.
template <class Span, class Point>
PCPX_HD void box_visit(const GridView& g, const BoxQ& b, uint64_t* stack, Span&& span,
                       Point&& point)
{
    if (b.empty)
        return;
    uint64_t key[32];
    bool valid[32];
    uint32_t c0[3];
    int const l0 = box_start(g, b, c0);
    for (int j = 0; j < 32; ++j)
        valid[j] = box_start_cell(g, b, l0, c0, j, key[j]);
    int sp = 0;
    for (;;)
    {
        bool const room = sp + 32 <= kBoxStackCap;
        BoxKind kind[32];
        uint32_t start[32], count[32];
        for (int j = 0; j < 32; ++j)
            kind[j] = valid[j] ? box_cell(g, b, key[j], room, start[j], count[j]) : kBoxNone;
        for (int j = 0; j < 32; ++j)
            if (kind[j] == kBoxInside)
                span(start[j], count[j]);
        for (int j = 0; j < 32; ++j)
            if (kind[j] == kBoxLeaf)
                for (uint32_t p = start[j]; p < start[j] + count[j]; ++p)
                    if (box_contains(b, load_pt(g.pts + p)))
                        point(p);
        for (int j = 31; j >= 0; --j)
            if (kind[j] == kBoxInner)
                stack[sp++] = key[j];
        if (sp == 0)
            return;
        int const P = sp < kBoxParents ? sp : kBoxParents;
        for (int j = 0; j < 32; ++j)
        {
            valid[j] = (j >> 3) < P;
            if (valid[j])
                key[j] = box_child_key(stack[sp - 1 - (j >> 3)], j & 7);
        }
        sp -= P;
    }
}

} // namespace pcpx
