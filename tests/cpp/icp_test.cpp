// Check of pcp::algorithm::icp on an octree and a kd-tree target, with float and double source
// points: a wavy surface moved by a known rigid motion must be registered back to within 1e-5
// in rotation and translation, by both metrics, and both trees must give the same bytes.
// Exit code 0 = every check holds; 2 = no GPU (libpcpx has no CPU path).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
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

// rotation by `deg` about (1, 2, 2) / 3 and then translation t
static std::array<double, 16> motion(double deg, double tx, double ty, double tz)
{
    double const a = deg * 3.14159265358979323846 / 180.0, c = std::cos(a), s = std::sin(a);
    double const k[3] = {1.0 / 3.0, 2.0 / 3.0, 2.0 / 3.0};
    double const K[9] = {0.0, -k[2], k[1], k[2], 0.0, -k[0], -k[1], k[0], 0.0};
    std::array<double, 16> M{};
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            M[i * 4 + j] = (i == j ? c : 0.0) + s * K[i * 3 + j] + (1.0 - c) * k[i] * k[j];
    M[3] = tx, M[7] = ty, M[11] = tz, M[15] = 1.0;
    return M;
}

// |T M - I| in rotation (max entry) and translation
static void residual(std::array<double, 16> const& T, std::array<double, 16> const& M, double& rot,
                     double& trans)
{
    rot = trans = 0.0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 4; ++j)
        {
            double v = 0.0;
            for (int k = 0; k < 4; ++k)
                v += T[i * 4 + k] * M[k * 4 + j];
            if (j < 3)
                rot = std::fmax(rot, std::fabs(v - (i == j ? 1.0 : 0.0)));
            else
                trans = std::fmax(trans, std::fabs(v));
        }
}

int main()
{
    if (pcpx_device_count() < 1)
    {
        std::fprintf(stderr, "no CUDA device: libpcpx has no CPU path\n");
        return 2;
    }
    std::mt19937 gen(5);
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::vector<pcp::point_t> target;
    std::vector<pcp::normal_t> normals;
    for (int i = 0; i < 20000; ++i)
    {
        float const x = u(gen), y = u(gen);
        float const z = 0.2f * std::sin(3.f * x) * std::cos(2.f * y);
        float const gx = 0.6f * std::cos(3.f * x) * std::cos(2.f * y);
        float const gy = -0.4f * std::sin(3.f * x) * std::sin(2.f * y);
        float const l = std::sqrt(gx * gx + gy * gy + 1.f);
        target.push_back({x, y, z});
        normals.push_back({-gx / l, -gy / l, 1.f / l});
    }
    auto const M = motion(5.0, 0.03, -0.02, 0.01);
    std::vector<pcp::point_t> source;
    std::vector<pcp::basic_point_t<double>> source_d;
    for (auto const& p : target)
    {
        double q[3];
        for (int a = 0; a < 3; ++a)
            q[a] = M[a * 4] * p.x() + M[a * 4 + 1] * p.y() + M[a * 4 + 2] * p.z() + M[a * 4 + 3];
        source.push_back({(float)q[0], (float)q[1], (float)q[2]});
        source_d.push_back({q[0], q[1], q[2]});
    }
    pcp::linked_octree_t octree(target.cbegin(), target.cend(), point_map);
    auto const coordinate_map = [](pcp::point_t const& p) {
        return std::array<float, 3u>{p.x(), p.y(), p.z()};
    };
    pcp::basic_linked_kdtree_t<pcp::point_t, 3u, decltype(coordinate_map)> kdtree{
        target.begin(), target.end(), coordinate_map};
    auto const map_d = [](pcp::basic_point_t<double> const& p) { return p; };

    for (std::uint32_t const metric : {PCPX_ICP_POINT_TO_PLANE, PCPX_ICP_POINT_TO_POINT})
    {
        pcp::icp::params_t prm;
        prm.metric         = metric;
        prm.max_distance   = 0.2f;
        prm.max_iterations = 100;
        auto const a = pcp::algorithm::icp(octree, normals, source.begin(), source.end(), point_map, prm);
        auto const b = pcp::algorithm::icp(kdtree, normals, source.begin(), source.end(), point_map, prm);
        auto const d = pcp::algorithm::icp(octree, normals, source_d.begin(), source_d.end(), map_d, prm);
        REQUIRE(a.stop_reason == PCPX_ICP_CONVERGED);
        REQUIRE(a.n_correspondences == target.size() && a.fitness == 1.0);
        REQUIRE(std::memcmp(a.transform.data(), b.transform.data(), sizeof a.transform) == 0);
        REQUIRE(a.iterations == b.iterations && a.rmse == b.rmse);
        double rot, trans;
        residual(a.transform, M, rot, trans);
        REQUIRE(rot < 1e-5 && trans < 1e-5);
        residual(d.transform, M, rot, trans);
        REQUIRE(d.stop_reason == PCPX_ICP_CONVERGED && rot < 1e-5 && trans < 1e-5);
        std::printf("metric %u: %u iterations, rmse %.3g\n", metric, a.iterations, a.rmse);
    }
    std::printf("icp_test: all checks hold\n");
    return 0;
}
