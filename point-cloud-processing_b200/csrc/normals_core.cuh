// Per-query epilogues on top of the top-K list: PCA normal / tangent plane and mean neighbour
// distance; the PCA over a radius ball.  __host__ __device__ (see grid_core.cuh).
#pragma once
#include "eig3.cuh"
#include "knn_core.cuh"
#include "radius_core.cuh"

namespace pcpx {

// Rare path of the normals kernel: the k-th and (k+1)-th distances are bit-equal, so WHICH of
// the tied points belongs to the neighbourhood is decided by the original index (the parity
// contract), which the position-keyed list does not carry.  `ids` is the exact (d2, original
// index) list; the block at `level` is walked once more and the members are accumulated in
// two passes exactly like normal_from_positions.
template <int K, class F>
PCPX_HD void for_each_in_block(const GridView& g, const QueryCell& qc, int level, F&& f)
{
    int const sh = g.lcap - level;
    uint32_t const cx = qc.ux >> sh, cy = qc.uy >> sh, cz = qc.uz >> sh;
    uint32_t const last = (1u << level) - 1u;
    uint64_t const key0 = cell_key(level, cx, cy, cz);
    for (int i = 0; i < 27; ++i)
    {
        Offset3 const o = block27_offset(i);
        int const dx = o.dx, dy = o.dy, dz = o.dz;
        if ((dx < 0 && cx == 0u) || (dx > 0 && cx == last) || (dy < 0 && cy == 0u) ||
            (dy > 0 && cy == last) || (dz < 0 && cz == 0u) || (dz > 0 && cz == last))
            continue;
        uint32_t start, count;
        if (!find_cell(g, key0 + key_delta(dx, dy, dz), start, count))
            continue;
        for (uint32_t p = start; p < start + count; ++p)
            f(load_pt(g.pts + p));
    }
}

template <int K>
PCPX_HD bool is_member(const TopK<K>& ids, uint32_t k, uint32_t id)
{
    bool m = false;
#pragma unroll
    for (int j = 0; j < K; ++j)
        m = m || ((uint32_t)j < k && ids.a[j] != kEmptyEntry && (uint32_t)ids.a[j] == id);
    return m;
}

template <int K>
PCPX_HD uint32_t normal_from_ids(const GridView& g, const QueryCell& qc, int level,
                                 const TopK<K>& ids, uint32_t k, float* n3, float* centroid3,
                                 float* gap)
{
    float sx = 0.f, sy = 0.f, sz = 0.f;
    uint32_t n = 0;
    for_each_in_block<K>(g, qc, level, [&](float4 const& c) {
        if (is_member(ids, k, f2u(c.w)))
        {
            sx += c.x, sy += c.y, sz += c.z;
            ++n;
        }
    });
    float const inv = 1.f / (float)n;
    float const mx = sx * inv, my = sy * inv, mz = sz * inv;
    Sym3 m{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for_each_in_block<K>(g, qc, level, [&](float4 const& c) {
        if (is_member(ids, k, f2u(c.w)))
        {
            float const x = c.x - mx, y = c.y - my, z = c.z - mz;
            m.xx += x * x, m.xy += x * y, m.xz += x * z;
            m.yy += y * y, m.yz += y * z, m.zz += z * z;
        }
    });
    smallest_eigenvector(m, n3[0], n3[1], n3[2], gap);
    if (centroid3)
        centroid3[0] = mx, centroid3[1] = my, centroid3[2] = mz;
    return n;
}

// ---- two-pass fast paths (see knn_core.cuh) ---------------------------------------------------

// Second pass of the fused normal: moments of the neighbours about the QUERY point (the
// neighbourhood surrounds it, so the shift removes the cancellation a raw one-pass covariance
// would have), then scatter = S2 - S1 S1^T / n, which equals the reference's centred V' V'^T
// (common/normals/normal_estimation.hpp:50-52) up to fp32 rounding — far inside the 1e-4
// |cos| tolerance.  Returns false when more than k points lie within the k-th distance (a
// bit-equal tie across the boundary): the caller then decides membership by original index.
template <int K, class Region, class SL>
PCPX_HD bool normal_two_pass(const GridView& g, const Region& region, const SL& sl,
                             float qx, float qy, float qz,
                             const TopD<K>& top, uint32_t k, float eps, float* n3,
                             float* centroid3, float* gap)
{
    float const tau = top.kth(k);
    uint32_t n      = 0;
    float s1x = 0.f, s1y = 0.f, s1z = 0.f;
    Sym3 s2{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for_each_within(g, region, sl, qx, qy, qz, tau, eps,
                    [&](float4 const&, uint32_t, float, float dx, float dy, float dz) {
                        ++n;
                        s1x += dx, s1y += dy, s1z += dz;
                        s2.xx += dx * dx, s2.xy += dx * dy, s2.xz += dx * dz;
                        s2.yy += dy * dy, s2.yz += dy * dz, s2.zz += dz * dz;
                    });
    if (n > k)
        return false;
    float const inv = 1.f / (float)n; // n == 0: NaN centroid, zero scatter -> (0,0,1)
    float const mx = s1x * inv, my = s1y * inv, mz = s1z * inv;
    Sym3 m;
    m.xx = s2.xx - s1x * mx, m.xy = s2.xy - s1x * my, m.xz = s2.xz - s1x * mz;
    m.yy = s2.yy - s1y * my, m.yz = s2.yz - s1y * mz, m.zz = s2.zz - s1z * mz;
    if (n == 0)
        m = Sym3{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    smallest_eigenvector(m, n3[0], n3[1], n3[2], gap);
    if (centroid3)
        centroid3[0] = qx + mx, centroid3[1] = qy + my, centroid3[2] = qz + mz;
    return true;
}

// The same PCA over a ball: exactly the points pcpx_radius_search returns for (q, r), the query
// itself included when it is an indexed point (radius_visit).  One walk accumulates the moments
// about the query point as above (the ball surrounds the query), so no per-neighbour data is
// kept anywhere.  n == 0: NaN centroid and (0,0,1); n == 1: the reference's centred scatter of a
// single point is exactly zero -> (0,0,1) (the shifted form would leave rounding residue).
// Returns n.
PCPX_HD uint32_t radius_normal(const GridView& g, float qx, float qy, float qz, float r, float* n3,
                               float* centroid3)
{
    uint32_t n = 0;
    float s1x = 0.f, s1y = 0.f, s1z = 0.f;
    Sym3 s2{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    radius_visit(g, qx, qy, qz, r, [&](float4 const& c, uint32_t) {
        float const dx = c.x - qx, dy = c.y - qy, dz = c.z - qz;
        ++n;
        s1x += dx, s1y += dy, s1z += dz;
        s2.xx += dx * dx, s2.xy += dx * dy, s2.xz += dx * dz;
        s2.yy += dy * dy, s2.yz += dy * dz, s2.zz += dz * dz;
        return false;
    });
    float const inv = 1.f / (float)n; // n == 0: NaN centroid
    float const mx = s1x * inv, my = s1y * inv, mz = s1z * inv;
    Sym3 m{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (n > 1)
    {
        m.xx = s2.xx - s1x * mx, m.xy = s2.xy - s1x * my, m.xz = s2.xz - s1x * mz;
        m.yy = s2.yy - s1y * my, m.yz = s2.yz - s1y * mz, m.zz = s2.zz - s1z * mz;
    }
    smallest_eigenvector_fast(m, n3[0], n3[1], n3[2]);
    if (centroid3)
        centroid3[0] = qx + mx, centroid3[1] = qy + my, centroid3[2] = qz + mz;
    return n;
}

// Second pass of the kNN kernel: every neighbour goes straight to its rank in the output row.
// Returns false when ranks are ambiguous (bit-equal distances); nothing written then is final.
template <int K, class Region, class SL>
PCPX_HD bool knn_two_pass_emit(const GridView& g, const Region& region, const SL& sl,
                               float qx, float qy, float qz,
                               const TopD<K>& top, uint32_t k, float eps, uint32_t* idx_row,
                               float* d2_row, uint32_t* out_count)
{
    if (top.has_internal_tie(k))
        return false;
    float const tau = top.kth(k);
    uint32_t n      = 0;
    for_each_within(g, region, sl, qx, qy, qz, tau, eps,
                    [&](float4 const& c, uint32_t, float d2, float, float, float) {
                        uint32_t const r = top.rank_of(d2);
                        if (r < k)
                        {
                            idx_row[r] = f2u(c.w);
                            if (d2_row)
                                d2_row[r] = d2;
                        }
                        ++n;
                    });
    if (n > k)
        return false;
    for (uint32_t j = n; j < k; ++j)
    {
        idx_row[j] = 0xFFFFFFFFu; // PCPX_NO_NEIGHBOUR
        if (d2_row)
            d2_row[j] = INFINITY;
    }
    if (out_count)
        *out_count = n;
    return true;
}

// algorithm/average_distance_to_neighbors.hpp:56-70 from the distance list alone.
template <int K>
PCPX_HD float mean_distance_d(const TopD<K>& top, uint32_t k)
{
    float sum  = 0.f;
    uint32_t n = 0;
#pragma unroll
    for (int j = 0; j < K; ++j)
        if ((uint32_t)j < k && top.a[j] < INFINITY)
        {
#ifdef __CUDA_ARCH__
            sum = __fadd_rn(sum, __fsqrt_rn(top.a[j]));
#else
            sum = sum + sqrtf(top.a[j]);
#endif
            ++n;
        }
#ifdef __CUDA_ARCH__
    return __fdiv_rn(sum, (float)n);
#else
    return sum / (float)n;
#endif
}

} // namespace pcpx
