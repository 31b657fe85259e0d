// Check of pcp::algorithm::cluster_by_density on an octree and a kd-tree against an O(n^2)
// brute-force DBSCAN of the same contract: core iff the ball (fp32 d2 <= fp32 r * r, itself
// included) holds >= min_points elements; clusters = connected components of the core points,
// numbered by their smallest element index; a border element takes the label of its core
// neighbour with the smallest (d2, index); noise otherwise.  Exit code 0 = every check holds;
// 2 = no GPU (libpcpx has no CPU path).
#include <cstdio>
#include <cstdlib>
#include <numeric>
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

static float d2_of(pcp::point_t const& a, pcp::point_t const& b)
{
    float const dx = a.x() - b.x(), dy = a.y() - b.y(), dz = a.z() - b.z();
    float const xx = dx * dx, yy = dy * dy, zz = dz * dz;
    float const s = xx + yy;
    return s + zz;
}

static std::uint32_t find(std::vector<std::uint32_t>& parent, std::uint32_t x)
{
    while (parent[x] != x)
        x = parent[x] = parent[parent[x]];
    return x;
}

static std::vector<std::uint32_t> brute_force(std::vector<pcp::point_t> const& pts, float r,
                                              std::size_t min_points, std::size_t& n_clusters)
{
    std::size_t const n = pts.size();
    float const rr      = r * r;
    std::vector<char> core(n);
    for (std::size_t i = 0; i < n; ++i)
    {
        std::size_t c = 0;
        for (std::size_t j = 0; j < n; ++j)
            c += d2_of(pts[i], pts[j]) <= rr;
        core[i] = c >= min_points;
    }
    std::vector<std::uint32_t> parent(n);
    std::iota(parent.begin(), parent.end(), 0u);
    for (std::size_t i = 0; i < n; ++i)
        for (std::size_t j = 0; j < i; ++j)
            if (core[i] && core[j] && d2_of(pts[i], pts[j]) <= rr)
            {
                std::uint32_t const a = find(parent, (std::uint32_t)i), b = find(parent, (std::uint32_t)j);
                parent[std::max(a, b)] = std::min(a, b); // roots stay the smallest index
            }
    std::vector<std::uint32_t> number(n, PCPX_NOISE), labels(n, PCPX_NOISE);
    n_clusters = 0;
    for (std::size_t i = 0; i < n; ++i)
        if (core[i])
        {
            std::uint32_t const root = find(parent, (std::uint32_t)i);
            if (number[root] == PCPX_NOISE)
                number[root] = (std::uint32_t)n_clusters++;
            labels[i] = number[root];
        }
    for (std::size_t i = 0; i < n; ++i)
        if (!core[i])
        {
            float best = 0.f;
            std::size_t src = n;
            for (std::size_t j = 0; j < n; ++j) // ascending j: the first of equal d2 wins
            {
                float const d2 = d2_of(pts[i], pts[j]);
                if (core[j] && d2 <= rr && (src == n || d2 < best))
                    best = d2, src = j;
            }
            if (src != n)
                labels[i] = labels[src];
        }
    return labels;
}

int main()
{
    if (pcpx_device_count() < 1)
    {
        std::fprintf(stderr, "no CUDA device: libpcpx has no CPU path\n");
        return 2;
    }
    // 40 Gaussian blobs with 5 % uniform noise, and a few exact duplicates
    std::mt19937 gen(11);
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::normal_distribution<float> g(0.f, 0.02f);
    std::vector<pcp::point_t> centres, points;
    for (int c = 0; c < 40; ++c)
        centres.push_back({u(gen), u(gen), u(gen)});
    for (int i = 0; i < 3800; ++i)
    {
        auto const& c = centres[static_cast<std::size_t>(i) % centres.size()];
        points.push_back({c.x() + g(gen), c.y() + g(gen), c.z() + g(gen)});
    }
    for (int i = 0; i < 200; ++i)
        points.push_back({u(gen), u(gen), u(gen)});
    for (int i = 0; i < 20; ++i)
        points.push_back(points[static_cast<std::size_t>(i) * 7]);

    pcp::linked_octree_t octree(points.cbegin(), points.cend(), point_map);
    REQUIRE(octree.size() == points.size());
    auto const coordinate_map = [](pcp::point_t const& p) {
        return std::array<float, 3u>{p.x(), p.y(), p.z()};
    };
    pcp::basic_linked_kdtree_t<pcp::point_t, 3u, decltype(coordinate_map)> kdtree{
        points.begin(), points.end(), coordinate_map};

    std::size_t checked_clusters = 0;
    for (float const r : {0.01f, 0.03f, 0.2f})
        for (std::size_t const min_points : {std::size_t{0}, std::size_t{1}, std::size_t{4},
                                             std::size_t{12}, std::size_t{1} << 40})
        {
            std::size_t want_n = 0, oct_n = 0, kd_n = 0;
            auto const want = brute_force(points, r, min_points, want_n);
            auto const oct  = pcp::algorithm::cluster_by_density(octree, r, min_points, &oct_n);
            auto const kd   = pcp::algorithm::cluster_by_density(kdtree, r, min_points, &kd_n);
            REQUIRE(oct == want && oct_n == want_n);
            REQUIRE(kd == want && kd_n == want_n);
            if (min_points <= 1)
                for (auto l : oct)
                    REQUIRE(l != PCPX_NOISE);
            checked_clusters += want_n;
        }
    REQUIRE(checked_clusters > 40);
    std::printf("cluster_test: all checks hold (%zu clusters over the settings)\n", checked_clusters);
    return 0;
}
