// TEST HARNESS ONLY — not part of libpcpx.so and never a product path.
//
// The emulated index of emu.cu plus the ball PCA of radius_normals_kernel (query_body.inc):
// radius_normal (normals_core.cuh) per query, run on the CPU so that `-m "not gpu"` tests can
// compare the device body with the oracle.  Built as its own library (tests/emu_ball_lib.py).
#include "emu.cu"

extern "C" int emu_radius_normals(void* h, const float* q, size_t nq, const float* radii, float r,
                                  float* nrm, float* ctr, uint32_t* cnt)
{
    EmuIndex* ix = static_cast<EmuIndex*>(h);
    for (size_t i = 0; i < nq; ++i)
    {
        float x, y, z;
        size_t row;
        fetch(ix, q, i, x, y, z, row);
        uint32_t const c = radius_normal(ix->g, x, y, z, radii ? radii[row] : r, nrm + 3 * row,
                                         ctr ? ctr + 3 * row : nullptr);
        if (cnt)
            cnt[row] = c;
    }
    return 0;
}
