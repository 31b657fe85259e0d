// TEST HARNESS ONLY — not part of libpcpx.so and never a product path.
//
// The emulated index of emu.cu plus the box traversal of box_count_kernel / box_fill_kernel
// (query_box.cu): box_visit (box_core.cuh) per box, run on the CPU so that `-m "not gpu"` tests
// can compare the classification of cells with a brute force.  Built as its own library
// (tests/emu_box_lib.py).
#include "emu.cu"

#include "box_core.cuh"

// the box every indexed point lies in, as the device call takes it (pcpx_index bbox_min/max):
// the voxel grid when there is one, else the bounding box of the whole input
static void emu_box_bounds(EmuIndex* ix, const float* voxel6, float bb[6])
{
    for (int a = 0; a < 3; ++a)
        bb[a] = INFINITY, bb[3 + a] = -INFINITY;
    for (uint64_t i = 0; i < ix->n_input; ++i)
    {
        float const v[3] = {ix->pts[i].x, ix->pts[i].y, ix->pts[i].z};
        for (int a = 0; a < 3; ++a)
            bb[a] = std::min(bb[a], v[a]), bb[3 + a] = std::max(bb[3 + a], v[a]);
    }
    for (int a = 0; a < 6; ++a)
        bb[a] = voxel6 ? voxel6[a] : (ix->n_input ? bb[a] : 0.f);
}

// counts[b] = the size of box b's result; idx (when not NULL) = the lists at offsets[b], in the
// order of the device fill; spans (when not NULL) = the number of INSIDE spans of every box
extern "C" int emu_box_search(void* h, const float* boxes, size_t nb, size_t stride_f,
                              const float* voxel6, uint32_t* counts, const uint64_t* offsets,
                              uint32_t* idx, uint64_t* spans)
{
    EmuIndex* ix = static_cast<EmuIndex*>(h);
    float bb[6];
    emu_box_bounds(ix, voxel6, bb);
    std::vector<uint64_t> stack(kBoxStackCap);
    for (size_t i = 0; i < nb; ++i)
    {
        BoxQ const b  = box_prepare(ix->g, boxes + i * stride_f, bb);
        uint64_t n    = 0, n_spans = 0;
        uint32_t* out = idx ? idx + offsets[i] : nullptr;
        box_visit(
            ix->g, b, stack.data(),
            [&](uint32_t s, uint32_t c) {
                if (out)
                    for (uint32_t p = s; p < s + c; ++p)
                        out[n + (p - s)] = f2u(ix->g.pts[p].w);
                n += c, ++n_spans;
            },
            [&](uint32_t p) {
                if (out)
                    out[n] = f2u(ix->g.pts[p].w);
                ++n;
            });
        counts[i] = (uint32_t)n;
        if (spans)
            spans[i] = n_spans;
    }
    return 0;
}
