// Drop-in check of the box range search: the single-box and batched range_search overloads of
// the octree (axis_aligned_bounding_box_t) and of the kd-tree (kd_axis_aligned_bounding_box_t,
// float and double coordinates) against `contains` over every element, including a small box on a
// lattice far from the origin.  Exit code 0 = every check holds; 2 = no GPU (libpcpx has no CPU
// path).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <random>

#include <pcpx/pcp.hpp>

#define REQUIRE(cond)                                                                          \
    do                                                                                         \
    {                                                                                          \
        if (!(cond))                                                                           \
        {                                                                                      \
            std::fprintf(stderr, "REQUIRE failed at %s:%d: %s\n", __FILE__, __LINE__, #cond);  \
            std::exit(1);                                                                      \
        }                                                                                      \
    } while (0)

static auto const point_map = [](pcp::point_t const& p) { return p; };
using aabb_t                = pcp::axis_aligned_bounding_box_t<pcp::point_t>;

// indices of the elements `in` holds, ascending
template <class Pred>
static std::vector<std::uint32_t> expected(std::vector<pcp::point_t> const& pts, Pred&& in)
{
    std::vector<std::uint32_t> out;
    for (std::size_t i = 0; i < pts.size(); ++i)
        if (in(pts[i]))
            out.push_back(static_cast<std::uint32_t>(i));
    return out;
}

// the elements a single-box call returned, as indices (points are distinct)
static std::vector<std::uint32_t> as_indices(std::vector<pcp::point_t> const& pts,
                                             std::vector<pcp::point_t> const& got)
{
    std::vector<std::uint32_t> out;
    for (auto const& g : got)
        for (std::size_t i = 0; i < pts.size(); ++i)
            if (pts[i].x() == g.x() && pts[i].y() == g.y() && pts[i].z() == g.z())
                out.push_back(static_cast<std::uint32_t>(i));
    std::sort(out.begin(), out.end());
    return out;
}

static std::vector<aabb_t> random_boxes(std::vector<pcp::point_t> const& pts, int n, float side,
                                        unsigned seed)
{
    std::mt19937 gen(seed);
    std::uniform_int_distribution<std::size_t> pick(0, pts.size() - 1);
    std::uniform_real_distribution<float> h(0.f, side);
    std::vector<aabb_t> boxes;
    for (int i = 0; i < n; ++i)
    {
        pcp::point_t const c = pts[pick(gen)];
        float const hx = h(gen), hy = h(gen), hz = h(gen);
        aabb_t b;
        b.min = {c.x() - hx, c.y() - hy, c.z() - hz};
        b.max = {c.x() + hx, c.y() + hy, c.z() + hz};
        boxes.push_back(b);
    }
    return boxes;
}

static void check_cloud(std::vector<pcp::point_t> const& pts, std::vector<aabb_t> const& boxes)
{
    pcp::linked_octree_t octree(pts.cbegin(), pts.cend(), point_map);
    auto const coordinate_map = [](pcp::point_t const& p) {
        return std::array<float, 3u>{p.x(), p.y(), p.z()};
    };
    auto const coordinate_map_d = [](pcp::point_t const& p) {
        return std::array<double, 3u>{p.x(), p.y(), p.z()};
    };
    pcp::basic_linked_kdtree_t<pcp::point_t, 3u, decltype(coordinate_map)> kdtree{
        pts.begin(), pts.end(), coordinate_map};
    pcp::basic_linked_kdtree_t<pcp::point_t, 3u, decltype(coordinate_map_d)> kdtree_d{
        pts.begin(), pts.end(), coordinate_map_d};

    std::vector<pcp::kd_axis_aligned_bounding_box_t<float, 3>> kd_boxes;
    std::vector<pcp::kd_axis_aligned_bounding_box_t<double, 3>> kd_boxes_d;
    for (auto const& b : boxes)
    {
        pcp::kd_axis_aligned_bounding_box_t<float, 3> k;
        k.min = {b.min.x(), b.min.y(), b.min.z()}, k.max = {b.max.x(), b.max.y(), b.max.z()};
        kd_boxes.push_back(k);
        pcp::kd_axis_aligned_bounding_box_t<double, 3> kd;
        // double boxes a fraction of an fp32 ulp inside the float ones: the outward rounding and
        // the exact host filter must drop the points on the float faces
        for (int a = 0; a < 3; ++a)
            kd.min[a] = static_cast<double>(k.min[a]) + 1e-12, kd.max[a] = static_cast<double>(k.max[a]) - 1e-12;
        kd_boxes_d.push_back(kd);
    }

    std::vector<std::uint64_t> off, off_kd, off_kd_d;
    std::vector<std::uint32_t> idx, idx_kd, idx_kd_d;
    octree.range_search(boxes.begin(), boxes.end(), off, idx);
    kdtree.range_search(kd_boxes.begin(), kd_boxes.end(), off_kd, idx_kd);
    kdtree_d.range_search(kd_boxes_d.begin(), kd_boxes_d.end(), off_kd_d, idx_kd_d);
    REQUIRE(off.size() == boxes.size() + 1 && off == off_kd && idx == idx_kd);
    REQUIRE(off_kd_d.size() == boxes.size() + 1);
    for (std::size_t b = 0; b < boxes.size(); ++b)
    {
        auto const want = expected(pts, [&](pcp::point_t const& p) { return boxes[b].contains(p); });
        std::vector<std::uint32_t> const got(idx.begin() + static_cast<std::ptrdiff_t>(off[b]),
                                             idx.begin() + static_cast<std::ptrdiff_t>(off[b + 1]));
        REQUIRE(got == want); // batched lists are ascending
        auto const want_d = expected(pts, [&](pcp::point_t const& p) {
            return kd_boxes_d[b].contains(coordinate_map_d(p));
        });
        std::vector<std::uint32_t> const got_d(
            idx_kd_d.begin() + static_cast<std::ptrdiff_t>(off_kd_d[b]),
            idx_kd_d.begin() + static_cast<std::ptrdiff_t>(off_kd_d[b + 1]));
        REQUIRE(got_d == want_d);
        if (b < 40) // the single-box overloads (host gather of elements)
        {
            REQUIRE(as_indices(pts, octree.range_search(boxes[b], point_map)) == want);
            REQUIRE(as_indices(pts, kdtree.range_search(kd_boxes[b])) == want);
            REQUIRE(as_indices(pts, kdtree_d.range_search(kd_boxes_d[b])) == want_d);
        }
    }
    // a sphere batch still takes the same template
    std::vector<pcp::sphere_t<pcp::point_t>> spheres{{pts[0], 0.1f}};
    octree.range_search(spheres.begin(), spheres.end(), off, idx);
    REQUIRE(off.size() == 2 && off[1] >= 1);
}

int main()
{
    if (pcpx_device_count() < 1)
    {
        std::fprintf(stderr, "no CUDA device: libpcpx has no CPU path\n");
        return 2;
    }
    std::mt19937 gen(11);
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::vector<pcp::point_t> cube;
    for (int i = 0; i < 20000; ++i)
        cube.push_back({u(gen), u(gen), u(gen)});
    auto boxes = random_boxes(cube, 200, 0.3f, 1);
    aabb_t all;
    all.min = {-2.f, -2.f, -2.f}, all.max = {2.f, 2.f, 2.f};
    boxes.push_back(all);
    check_cloud(cube, boxes);

    // 9 x 9 x 9 lattice, spacing 1e-4, near x = y = z = 100 (dropin_test.cpp): boxes with their
    // faces on lattice points
    std::vector<pcp::point_t> far;
    for (int i = 0; i < 9; ++i)
        for (int j = 0; j < 9; ++j)
            for (int l = 0; l < 9; ++l)
                far.push_back({100.f + 1e-4f * i, 100.f + 1e-4f * j, 100.f + 1e-4f * l});
    std::vector<aabb_t> far_boxes;
    std::uniform_int_distribution<std::size_t> pick(0, far.size() - 1);
    for (int i = 0; i < 100; ++i)
    {
        pcp::point_t const a = far[pick(gen)], b = far[pick(gen)];
        aabb_t box;
        box.min = {std::min(a.x(), b.x()), std::min(a.y(), b.y()), std::min(a.z(), b.z())};
        box.max = {std::max(a.x(), b.x()), std::max(a.y(), b.y()), std::max(a.z(), b.z())};
        far_boxes.push_back(box);
    }
    aabb_t sub;
    sub.min = far[(2 * 9 + 2) * 9 + 2], sub.max = far[(6 * 9 + 6) * 9 + 6];
    far_boxes.push_back(sub);
    check_cloud(far, far_boxes);

    std::printf("box_search_test: all checks hold\n");
    return 0;
}
