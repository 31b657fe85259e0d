// Drop-in check of pcp::gpu_radius_map: estimate_normals over a ball map written the way the
// reference's users write it — a lambda over octree.range_search(sphere_t{p, r}) or over the
// kd-tree's range_search(sphere_a{p, r}) — gives the same normals (up to sign) as the one fused
// call that make_gpu_radius_map selects.  Exit code 0 = every check holds; 2 = no GPU (libpcpx
// has no CPU path).
#include <cmath>
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

// rows whose normals differ by more than 1 - |cos| = 1e-4, among balls of >= 5 points
static std::size_t mismatches(std::vector<pcp::normal_t> const& a, std::vector<pcp::normal_t> const& b,
                              std::vector<std::size_t> const& ball_size)
{
    std::size_t bad = 0;
    for (std::size_t i = 0; i < a.size(); ++i)
    {
        double const dot = static_cast<double>(a[i].x()) * b[i].x() +
                           static_cast<double>(a[i].y()) * b[i].y() +
                           static_cast<double>(a[i].z()) * b[i].z();
        if (ball_size[i] >= 5 && 1.0 - std::fabs(dot) > 1e-4)
            ++bad;
    }
    return bad;
}

int main()
{
    if (pcpx_device_count() < 1)
    {
        std::fprintf(stderr, "no CUDA device: libpcpx has no CPU path\n");
        return 2;
    }
    // a gently curved, noisy sheet of 20 k points: every ball of ~40 points is well conditioned
    std::mt19937 gen(7);
    std::uniform_real_distribution<float> u(0.f, 1.f);
    std::normal_distribution<float> g(0.f, 1.f);
    std::vector<pcp::point_t> points;
    for (int i = 0; i < 20000; ++i)
    {
        float const x = u(gen), y = u(gen);
        points.push_back({x, y, 0.05f * std::sin(3.f * x) * std::cos(2.f * y) + 5e-4f * g(gen)});
    }
    float const r = 0.025f;
    using normals_t = std::vector<pcp::normal_t>;
    auto const identity = pcp::algorithm::default_normal_transform<pcp::point_t, pcp::normal_t>;

    pcp::linked_octree_t octree(points.cbegin(), points.cend(), point_map);
    REQUIRE(octree.size() == points.size());

    // the recognised map: one fused ball -> PCA call for the whole range (both overloads)
    auto const ball = pcp::make_gpu_radius_map(octree, r, point_map);
    normals_t fused(points.size()), fused_par(points.size());
    pcp::algorithm::estimate_normals(points.cbegin(), points.cend(), fused.begin(), point_map, ball,
                                     identity);
    pcp::algorithm::estimate_normals(std::execution::par, points.cbegin(), points.cend(),
                                     fused_par.begin(), point_map, ball, identity);
    for (std::size_t i = 0; i < points.size(); ++i)
        REQUIRE(fused[i].x() == fused_par[i].x() && fused[i].y() == fused_par[i].y() &&
                fused[i].z() == fused_par[i].z());

    // called on one element it answers like the octree's own range search
    std::vector<pcp::sphere_t<pcp::point_t>> spheres;
    for (auto const& p : points)
        spheres.push_back(pcp::sphere_t<pcp::point_t>{p, r});
    std::vector<std::uint64_t> offsets;
    std::vector<std::uint32_t> members;
    octree.range_search(spheres.begin(), spheres.end(), offsets, members);
    std::vector<std::size_t> ball_size(points.size());
    for (std::size_t i = 0; i < points.size(); ++i)
        ball_size[i] = static_cast<std::size_t>(offsets[i + 1] - offsets[i]);
    REQUIRE(ball(points[123]).size() == ball_size[123]);
    double mean = 0;
    for (auto s : ball_size)
        mean += static_cast<double>(s) / static_cast<double>(ball_size.size());
    REQUIRE(mean > 30 && mean < 60);

    // the lambdas of the reference's examples: the map is called once per element
    auto const octree_ball = [&](pcp::point_t const& p) {
        return octree.range_search(pcp::sphere_t<pcp::point_t>{p, r}, point_map);
    };
    normals_t via_octree;
    pcp::algorithm::estimate_normals(points.cbegin(), points.cend(), std::back_inserter(via_octree),
                                     point_map, octree_ball, identity);
    REQUIRE(via_octree.size() == points.size());
    REQUIRE(mismatches(fused, via_octree, ball_size) == 0);

    auto const coordinate_map = [](pcp::point_t const& p) {
        return std::array<float, 3u>{p.x(), p.y(), p.z()};
    };
    pcp::basic_linked_kdtree_t<pcp::point_t, 3u, decltype(coordinate_map)> kdtree{
        points.begin(), points.end(), coordinate_map};
    auto const kd_ball = [&](pcp::point_t const& p) {
        return kdtree.range_search(pcp::sphere_a<float>{{p.x(), p.y(), p.z()}, r});
    };
    normals_t via_kdtree(points.size());
    pcp::algorithm::estimate_normals(points.cbegin(), points.cend(), via_kdtree.begin(), point_map,
                                     kd_ball, identity);
    REQUIRE(mismatches(fused, via_kdtree, ball_size) == 0);

    // foreign queries (not the indexed cloud): the map over the kd-tree's own elements
    std::vector<pcp::point_t> shifted(points.begin(), points.begin() + 2000);
    for (auto& p : shifted)
        p = pcp::point_t{p.x() + 1e-3f, p.y() - 1e-3f, p.z()};
    normals_t fused_ext(shifted.size()), lambda_ext(shifted.size());
    auto const kd_map = pcp::make_gpu_radius_map(kdtree, r, point_map);
    pcp::algorithm::estimate_normals(shifted.cbegin(), shifted.cend(), fused_ext.begin(), point_map,
                                     kd_map, identity);
    pcp::algorithm::estimate_normals(shifted.cbegin(), shifted.cend(), lambda_ext.begin(), point_map,
                                     kd_ball, identity);
    std::vector<std::size_t> ext_size(shifted.size());
    for (std::size_t i = 0; i < shifted.size(); ++i)
        ext_size[i] = kd_ball(shifted[i]).size();
    REQUIRE(mismatches(fused_ext, lambda_ext, ext_size) == 0);

    std::printf("radius_normals_test: all checks hold (mean ball %.1f points)\n", mean);
    return 0;
}
