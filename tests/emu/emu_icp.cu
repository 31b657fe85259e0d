// TEST HARNESS ONLY — not part of libpcpx.so and never a product path.
//
// The emulated index of emu.cu plus the correspondence pass of pcpx_nearest_within / pcpx_icp
// (icp.cu) run one query after another on the CPU: the same transform, nearest-within walk and
// pair terms (icp_core.cuh), the same host solve and loop (icp_solve.hpp), the sums added in
// query order, so that `-m "not gpu"` tests can compare them with a brute force and with numpy.
// Built as its own library (tests/emu_icp_lib.py).
#include "emu.cu"

#include "icp_core.cuh"
#include "icp_solve.hpp"

static int emu_nearest_level(const EmuIndex* ix)
{
    return choose_plan(ix->g.n, ix->cells_per_level, ix->g.lfine, 1u, 1.15).level;
}

// one correspondence pass under T (nullptr: the queries as they are); sums (may be NULL) in the
// layout of icp_solve.hpp, in query order; idx / d2 / corr (may be NULL) per query
static void emu_pass(const EmuIndex* ix, const float* q, size_t nq, const double* T, float r,
                     uint32_t metric, const float* normals, const double* c, double* sums,
                     uint32_t* idx, float* d2, uint32_t* corr)
{
    GridView const& g = ix->g;
    int const level   = emu_nearest_level(ix);
    int const nt      = icp_terms(metric);
    if (sums)
        for (int k = 0; k < nt; ++k)
            sums[k] = 0.0;
    Rigid34 R{};
    if (T)
        for (int i = 0; i < 12; ++i)
            R.m[i] = T[i];
    for (size_t i = 0; i < nq; ++i)
    {
        float y[3] = {q[3 * i], q[3 * i + 1], q[3 * i + 2]};
        if (T)
            rigid_apply(R, q[3 * i], q[3 * i + 1], q[3 * i + 2], y);
        uint32_t pos;
        uint64_t const key = nearest_within(g, level, y[0], y[1], y[2], r, pos);
        if (idx)
            idx[i] = key == kIcpNoKey ? kIcpNone : (uint32_t)key;
        if (d2)
            d2[i] = key == kIcpNoKey ? INFINITY : u2f((uint32_t)(key >> 32));
        uint32_t cr = kIcpNone;
        if (key != kIcpNoKey && sums)
        {
            uint32_t const orig = (uint32_t)key;
            float nrm[3]        = {0.f, 0.f, 0.f};
            if (metric == 0)
                nrm[0] = normals[3 * (size_t)orig], nrm[1] = normals[3 * (size_t)orig + 1],
                nrm[2] = normals[3 * (size_t)orig + 2];
            if (icp_pair_valid(metric, nrm))
            {
                IcpPair const P = icp_pair(metric, y, g.pts[pos], nrm, c, u2f((uint32_t)(key >> 32)));
                for (int k = 0; k < nt; ++k)
                    sums[k] += icp_term(metric, P, k);
                cr = orig;
            }
        }
        if (corr)
            corr[i] = cr;
    }
}

extern "C" {

void emu_nearest_within(void* h, const float* q, size_t nq, const double* T, float r,
                        uint32_t* idx, float* d2)
{
    emu_pass(static_cast<EmuIndex*>(h), q, nq, T, r, 0u, nullptr, nullptr, nullptr, idx, d2,
             nullptr);
}

// the reduced sums of one pass (kIcpMaxTerms doubles) and the pairs (ns entries)
void emu_icp_sums(void* h, const float* src, size_t ns, const double* T, float r, uint32_t metric,
                  const float* normals, const double* c, double* sums, uint32_t* corr)
{
    emu_pass(static_cast<EmuIndex*>(h), src, ns, T, r, metric, normals, c, sums, nullptr, nullptr,
             corr);
}

// the step x = (omega, v) the solver takes from the sums
void emu_icp_solve(uint32_t metric, const double* sums, double* x)
{
    if (metric == 0)
        icp_solve_plane(sums, x);
    else
        icp_solve_point(sums, x);
}

void emu_icp_update(double* T, const double* x, const double* c) { icp_update(T, x, c); }

// the whole loop of pcpx_icp over the emulated index; T: init in, result out; out3 = {iterations,
// stop_reason, pairs of the final pass}
void emu_icp(void* h, const float* src, size_t ns, const float* normals, uint32_t metric,
             uint32_t max_it, float r, double rot_tol, double trans_tol, const double* c,
             double* T, uint64_t* out3, uint32_t* corr)
{
    EmuIndex* ix = static_cast<EmuIndex*>(h);
    IcpLoopResult const lr = icp_loop(metric, max_it, rot_tol, trans_tol, c, T,
                                      [&](const double* Tc, double* s) {
                                          emu_pass(ix, src, ns, Tc, r, metric, normals, c, s,
                                                   nullptr, nullptr, nullptr);
                                      });
    double s[kIcpMaxTerms];
    emu_pass(ix, src, ns, T, r, metric, normals, c, s, nullptr, nullptr, corr);
    out3[0] = lr.iterations, out3[1] = lr.stop_reason, out3[2] = (uint64_t)icp_pairs(metric, s);
}

} // extern "C"
