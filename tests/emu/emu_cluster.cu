// TEST HARNESS ONLY — not part of libpcpx.so and never a product path.
//
// The emulated index of emu.cu plus the steps of pcpx_cluster_by_density (cluster.cu) run one
// point after another on the CPU: the same core, union, ball and border bodies (cluster_core.cuh),
// the union-find sequential, so that `-m "not gpu"` tests can compare the labels with a brute
// force.  Built as its own library (tests/emu_cluster_lib.py).
#include "emu.cu"

#include "cluster_core.cuh"

// labels (n_input entries, original positions) and core flags (n_input bytes, original
// positions; 0 for un-indexed points); returns the number of clusters
extern "C" uint64_t emu_cluster(void* h, float r, uint32_t min_points, uint32_t* labels,
                                uint8_t* core_out)
{
    EmuIndex* ix       = static_cast<EmuIndex*>(h);
    GridView const& g  = ix->g;
    uint32_t const n   = (uint32_t)ix->n_input, ni = g.n;
    std::vector<uint8_t> core(ni), first(n, 0);
    std::vector<uint32_t> parent(ni), min_orig(ni, kClusterNone);
    std::vector<uint64_t> number(n + 1, 0);
    for (uint32_t i = 0; i < n; ++i)
        labels[i] = kClusterNone, core_out[i] = 0;
    for (uint32_t t = 0; t < ni; ++t)
    {
        core[t]   = cluster_is_core(g, g.pts[t], r, min_points);
        parent[t] = t;
        core_out[f2u(g.pts[t].w)] = core[t];
    }
    for (uint32_t t = 0; t < ni; ++t)
        if (core[t])
            cluster_union_point(g, core.data(), parent.data(), t, r);
    for (uint32_t t = 0; t < ni; ++t)
        if (core[t])
        {
            uint32_t const root = uf_root(parent.data(), t);
            parent[t]           = root;
            min_orig[root]      = std::min(min_orig[root], f2u(g.pts[t].w));
        }
    for (uint32_t t = 0; t < ni; ++t)
        if (core[t] && min_orig[parent[t]] == f2u(g.pts[t].w))
            first[f2u(g.pts[t].w)] = 1;
    for (uint32_t i = 0; i < n; ++i)
        number[i + 1] = number[i] + first[i];
    for (uint32_t t = 0; t < ni; ++t)
    {
        uint32_t const src = core[t] ? t : cluster_border_source(g, core.data(), g.pts[t], r);
        labels[f2u(g.pts[t].w)] =
            src == kClusterNone ? kClusterNone : (uint32_t)number[min_orig[parent[src]]];
    }
    return number[n];
}
