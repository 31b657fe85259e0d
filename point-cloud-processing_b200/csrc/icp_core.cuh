// Rigid registration (pcpx_nearest_within, pcpx_icp): the per-query bodies of the kernels of
// icp.cu, __host__ __device__ so that the CPU emulation (tests/emu/emu_icp.cu) runs the same code.
#pragma once
#include "radius_core.cuh"

namespace pcpx {

constexpr uint32_t kIcpNone = 0xFFFFFFFFu;
constexpr uint64_t kIcpNoKey = ~0ull;

// fp64 arithmetic never contracted into FMA (see fmul_x)
PCPX_HD double dmul_x(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
PCPX_HD double dadd_x(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// A rigid transform handed to the kernels by value: rows 0-2 of the row-major 4 x 4
struct Rigid34
{
    double m[12];
};

// y_a = ((R[a][0] x + R[a][1] y) + R[a][2] z) + t[a] in fp64 without FMA, rounded once to fp32
PCPX_HD void rigid_apply(const Rigid34& T, float x, float y, float z, float out[3])
{
#pragma unroll
    for (int a = 0; a < 3; ++a)
    {
        double const* r = T.m + 4 * a;
        double const s  = dadd_x(dadd_x(dadd_x(dmul_x(r[0], x), dmul_x(r[1], y)), dmul_x(r[2], z)), r[3]);
        out[a]          = (float)s;
    }
}

PCPX_HD bool finite3(float x, float y, float z)
{
    return fabsf(x) <= 3.402823466e38f && fabsf(y) <= 3.402823466e38f && fabsf(z) <= 3.402823466e38f;
}

// The indexed point q with the smallest (fl(d2), original index) among those with
// fl(d2(query, q)) <= fl(r * r): returns its key (d2 bits << 32 | original index), kIcpNoKey when
// there is none (always for a non-finite query or an empty index), and the point's sorted position
// in best_pos.
// Walk: from `start_level` (the kNN planner's level for k = 1: a block of a few points) towards
// the root, each level's 3 x 3 x 3 block walked flat like radius_visit, cells whose lower bound
// exceeds min(r * r, best d2) skipped; a level ends the search once everything outside its block
// is provably farther than the best so far (strictly: an equal d2 outside could hold a smaller
// index) or than r.  The walk never goes coarser than radius_level's level, whose block holds the
// whole ball.
PCPX_HD uint64_t nearest_within(const GridView& g, int start_level, float qx, float qy, float qz,
                                float r, uint32_t& best_pos)
{
    uint64_t best = kIcpNoKey;
    best_pos      = 0;
    if (g.n == 0 || !finite3(qx, qy, qz))
        return best;
    float const rr     = fmul_x(r, r);
    QueryCell const qc = query_cell(g, qx, qy, qz);
    BlockGeom b;
    int const lr = radius_level(g, qc, qx, qy, qz, r, rr, b);
    float bound  = rr; // min(r * r, best d2)
    for (int l = start_level > lr ? start_level : lr;; --l)
    {
        b = block_geom(g, qc, l, qx, qy, qz);
        CellList cl;
        collect_block27(g, b, l, cl, nullptr, bound);
        int e = 0;
        uint32_t p = 0, pend = 0;
        float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
        for (;;)
        {
            if (p >= pend)
            {
                uint32_t s, en;
                do // spans the best so far has excluded are skipped (the sentinel never is)
                {
                    s = cl.start[e], en = cl.end[e];
                } while (cl.lb2[e++] > bound);
                if (s == kSpanEnd)
                    break;
                p = s, pend = en;
                c = load_pt(g.pts + p);
            }
            float4 const a = c;
            c = load_pt(g.pts + p + 1); // unconditional: the array is padded (kPtsPad)
            float const d2 = sqdist_x(fsub_x(a.x, qx), fsub_x(a.y, qy), fsub_x(a.z, qz));
            if (d2 <= bound)
            {
                uint64_t const key = ((uint64_t)f2u(d2) << 32) | f2u(a.w);
                if (key < best)
                    best = key, best_pos = p, bound = d2;
            }
            ++p;
        }
        if (l <= lr || rr < b.block_lb2 || bound < b.block_lb2)
            return best;
    }
}

// ---- the contribution of one pair (y, q) to the reduced sums (layout: icp_solve.hpp) ----------
// Term k of the pair, the centre c subtracted in fp64.  `nrm`: the target normal (point-to-plane).
struct IcpPair
{
    double py[3]; // y - c
    double pq[3]; // q - c  (point-to-point)
    double J[6];  // [(y - c) x n, n]  (point-to-plane)
    double r;     // (y - q) . n
    double d2;
};

PCPX_HD IcpPair icp_pair(uint32_t metric, const float y[3], float4 q, const float* nrm,
                         const double c[3], float d2)
{
    IcpPair P;
    double const yd[3] = {(double)y[0], (double)y[1], (double)y[2]};
    double const qd[3] = {(double)q.x, (double)q.y, (double)q.z};
    for (int a = 0; a < 3; ++a)
        P.py[a] = yd[a] - c[a], P.pq[a] = qd[a] - c[a];
    P.d2 = (double)d2;
    if (metric == 0)
    {
        double const n[3] = {(double)nrm[0], (double)nrm[1], (double)nrm[2]};
        P.J[0] = dadd_x(dmul_x(P.py[1], n[2]), -dmul_x(P.py[2], n[1]));
        P.J[1] = dadd_x(dmul_x(P.py[2], n[0]), -dmul_x(P.py[0], n[2]));
        P.J[2] = dadd_x(dmul_x(P.py[0], n[1]), -dmul_x(P.py[1], n[0]));
        P.J[3] = n[0], P.J[4] = n[1], P.J[5] = n[2];
        P.r    = dadd_x(dadd_x(dmul_x(yd[0] - qd[0], n[0]), dmul_x(yd[1] - qd[1], n[1])),
                        dmul_x(yd[2] - qd[2], n[2]));
    }
    else
    {
        for (int a = 0; a < 6; ++a)
            P.J[a] = 0.0;
        P.r = 0.0;
    }
    return P;
}

// term k (0 <= k < icp_terms(metric)) of the pair; k is a compile-time constant in the kernels
PCPX_HD double icp_term(uint32_t metric, const IcpPair& P, int k)
{
    if (metric == 0)
    {
        if (k < 21)
        {
            int i = 0, j = k; // k -> (i, j), i <= j, upper triangle row by row
            while (j >= 6 - i)
                j -= 6 - i, ++i;
            return dmul_x(P.J[i], P.J[i + j]);
        }
        if (k < 27)
            return dmul_x(P.J[k - 21], P.r);
        return k == 27 ? P.d2 : 1.0;
    }
    if (k < 3)
        return P.py[k];
    if (k < 6)
        return P.pq[k - 3];
    if (k < 15)
        return dmul_x(P.py[(k - 6) / 3], P.pq[(k - 6) % 3]);
    return k == 15 ? P.d2 : 1.0;
}

// Whether the pair counts: every pair for point-to-point; for point-to-plane only a pair whose
// target normal is finite.
PCPX_HD bool icp_pair_valid(uint32_t metric, const float* nrm)
{
    return metric != 0 || finite3(nrm[0], nrm[1], nrm[2]);
}

} // namespace pcpx
