// Density-based clustering (pcpx_cluster_by_density): the per-point bodies of the kernels of
// cluster.cu, __host__ __device__ so that the CPU emulation (tests/emu/emu_cluster.cu) runs the
// same code.  N(p) is the ball of radius_visit: the indexed q with fl(d2(p, q)) <= fl(r * r), p
// itself included.  d2 is symmetric bit for bit (negating a difference does not change its
// square), so q in N(p) <=> p in N(q) and the union pass needs every edge from one side only.
#pragma once
#include "radius_core.cuh"

namespace pcpx {

constexpr uint32_t kClusterNone = 0xFFFFFFFFu;

// p is core iff |N(p)| >= min_points: the walk of density_keep_kernel, stopped at the threshold
PCPX_HD bool cluster_is_core(const GridView& g, float4 p, float r, uint32_t min_points)
{
    uint32_t cnt = 0;
    if (min_points > 0)
        radius_visit_lazy(g, p.x, p.y, p.z, r, [&](float4 const&, uint32_t) {
            return ++cnt >= min_points;
        });
    return cnt >= min_points;
}

// ---- lock-free union-find over sorted positions (the ECL-CC scheme) --------------------------
// Invariant: parent[x] <= x.  A hook only ever replaces a root's self-link by a smaller position
// of the other set, so the root of a set is its smallest position whatever the interleaving of
// the threads.  Other threads write `parent` while a find walks it: every load is volatile
// (never __ldg, which may serve a stale line), and the path-halving stores are plain: any value
// they write is an ancestor, so a lost or late one only costs a longer walk.
PCPX_HD uint32_t uf_load(const uint32_t* p)
{
    return *static_cast<const volatile uint32_t*>(p);
}

PCPX_HD uint32_t uf_cas(uint32_t* p, uint32_t expected, uint32_t desired)
{
#ifdef __CUDA_ARCH__
    return atomicCAS(p, expected, desired);
#else
    uint32_t const old = *p; // (the emulation is sequential)
    if (old == expected)
        *p = desired;
    return old;
#endif
}

// root of x, halving the path on the way
PCPX_HD uint32_t uf_find(uint32_t* parent, uint32_t x)
{
    uint32_t cur = uf_load(parent + x);
    if (cur != x)
    {
        uint32_t prev = x, next;
        while (cur > (next = uf_load(parent + cur)))
        {
            *static_cast<volatile uint32_t*>(parent + prev) = next;
            prev = cur;
            cur  = next;
        }
    }
    return cur;
}

// root of x without writing: the find of the flatten pass.  A halving store there could land
// after another thread's parent[t] = root and leave t pointing at an ancestor short of its root.
PCPX_HD uint32_t uf_root(const uint32_t* parent, uint32_t x)
{
    uint32_t next;
    while (x > (next = uf_load(parent + x)))
        x = next;
    return x;
}

// Joins the sets whose representatives are a and b (both found just before): the larger root is
// hooked under the smaller with a CAS; a failed CAS returns the new parent of the would-be root,
// and the hook is retried from there.  On return `a` is a position of the joined set.
PCPX_HD void uf_join(uint32_t* parent, uint32_t& a, uint32_t b)
{
    while (a != b)
    {
        if (a < b)
        {
            uint32_t const ret = uf_cas(parent + b, b, a);
            if (ret == b)
                return;
            b = ret;
        }
        else
        {
            uint32_t const ret = uf_cas(parent + a, a, b);
            if (ret == a)
            {
                a = b;
                return;
            }
            a = ret;
        }
    }
}

// Union pass of one core point t: join t with every core neighbour at a smaller sorted position.
// The finds come first, so two points already in one set cost no CAS.
PCPX_HD void cluster_union_point(const GridView& g, const uint8_t* core, uint32_t* parent,
                                 uint32_t t, float r)
{
    float4 const p = load_pt(g.pts + t);
    uint32_t rt    = t;
    radius_visit(g, p.x, p.y, p.z, r, [&](float4 const&, uint32_t q) {
        if (q < t && core[q])
        {
            uint32_t const rq = uf_find(parent, q);
            rt                = uf_find(parent, rt);
            if (rt != rq)
                uf_join(parent, rt, rq);
        }
        return false;
    });
}

// Border rule of a non-core point p: the sorted position of the core q in N(p) with the smallest
// (fl(d2), original index), or kClusterNone when N(p) holds no core point (p is noise).
PCPX_HD uint32_t cluster_border_source(const GridView& g, const uint8_t* core, float4 p, float r)
{
    uint64_t best = ~0ull;
    uint32_t src  = kClusterNone;
    radius_visit(g, p.x, p.y, p.z, r, [&](float4 const& c, uint32_t q) {
        if (core[q])
        {
            // the d2 of the ball test itself; non-negative, so its bits order like its value
            float const d2     = sqdist_x(fsub_x(c.x, p.x), fsub_x(c.y, p.y), fsub_x(c.z, p.z));
            uint64_t const key = ((uint64_t)f2u(d2) << 32) | f2u(c.w);
            if (key < best)
                best = key, src = q;
        }
        return false;
    });
    return src;
}

} // namespace pcpx
