// pcpx/pcp.hpp — C++17 drop-in front end over the C ABI (include/pcpx.h, libpcpx.so).
//
// Keeps the call signatures of pcp's neighbourhood hot path (namespace `pcp`, same class and
// function names, same concepts: Element + PointViewMap / CoordinateMap / KnnMap / TransformOp)
// so that code written against the reference's headers compiles against these and runs the
// queries on a B200 instead of walking a pointer octree on the CPU.  Written from the
// reference's interface, not from its implementation; each entity cites what it stands in for
// (paths relative to the reference's include/pcp/).
//
// What is different, by design:
//   * the containers are immutable after construction (the index is built on the device in
//     one shot; there is no insert / erase / iterator over tree nodes),
//   * every query has a BATCHED overload next to the per-query one; the per-query overloads
//     cost one kernel launch each and exist for source compatibility,
//   * `estimate_normals` recognises `pcp::gpu_knn_map` (an index + k) and then runs the fused
//     kNN -> PCA kernel once for the whole range, and `pcp::gpu_radius_map` (an index + a
//     radius) the fused ball -> PCA kernel; with any other KnnMap it calls the map per
//     element like the reference does and batches only the PCA (still on the GPU),
//   * failures throw std::runtime_error (the reference has no error path at all); there is no
//     CPU fallback anywhere.
#ifndef PCPX_PCP_HPP
#define PCPX_PCP_HPP

#include <algorithm>
#include <array>
#include <atomic>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <exception>
#include <execution>
#include <iterator>
#include <limits>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "../pcpx.h"

namespace pcp {

// ---- geometric value types (common/points/point.hpp:21-93, point_view.hpp:24-80,
//      common/normals/normal.hpp:20-94) -----------------------------------------------------
template <class T>
class basic_point_t
{
  public:
    using component_type  = T;
    using coordinate_type = T;

    basic_point_t() noexcept = default;
    basic_point_t(T x, T y, T z) noexcept : c_{x, y, z} {}
    template <class PointView, class = decltype(std::declval<PointView const&>().x())>
    basic_point_t(PointView const& o) noexcept : c_{T(o.x()), T(o.y()), T(o.z())}
    {
    }

    T const& x() const { return c_[0]; }
    T const& y() const { return c_[1]; }
    T const& z() const { return c_[2]; }
    void x(T v) { c_[0] = v; }
    void y(T v) { c_[1] = v; }
    void z(T v) { c_[2] = v; }

    basic_point_t operator-() const noexcept { return {-c_[0], -c_[1], -c_[2]}; }
    template <class V>
    basic_point_t operator+(V const& v) const noexcept
    {
        return {c_[0] + v.x(), c_[1] + v.y(), c_[2] + v.z()};
    }
    friend basic_point_t operator*(T k, basic_point_t const& p) noexcept
    {
        return {k * p.c_[0], k * p.c_[1], k * p.c_[2]};
    }
    friend basic_point_t operator/(basic_point_t const& p, T k) noexcept
    {
        return {p.c_[0] / k, p.c_[1] / k, p.c_[2] / k};
    }

  private:
    T c_[3] = {T(0), T(0), T(0)}; // 12 bytes for float, no padding: a contiguous range of
                                  // point_t goes to the C ABI as `const float*`, stride 12
};
using point_t = basic_point_t<float>;

template <class Point>
class basic_point_view_t
{
  public:
    using component_type  = typename Point::component_type;
    using coordinate_type = typename Point::coordinate_type;

    basic_point_view_t() noexcept = default;
    explicit basic_point_view_t(Point* p) noexcept : p_(p) {}
    coordinate_type const& x() const { return p_->x(); }
    coordinate_type const& y() const { return p_->y(); }
    coordinate_type const& z() const { return p_->z(); }
    void x(coordinate_type v) { p_->x(v); }
    void y(coordinate_type v) { p_->y(v); }
    void z(coordinate_type v) { p_->z(v); }
    Point const* point() const noexcept { return p_; }
    Point* point() noexcept { return p_; }
    void point(Point* p) noexcept { p_ = p; }

  private:
    Point* p_ = nullptr;
};
using point_view_t = basic_point_view_t<point_t>;

// common/points/vertex.hpp:30-117: a point view that also carries a 64-bit identifier (the
// GraphVertex concept of the reference: id() / id(value)); equality is equality of identifiers.
template <class PointView>
class basic_point_view_vertex_t : public basic_point_view_t<PointView>
{
  public:
    using id_type     = std::uint64_t;
    using self_type   = basic_point_view_vertex_t<PointView>;
    using point_type  = basic_point_view_t<PointView>;
    using parent_type = point_type;

    id_type id() const { return id_; }
    void id(id_type value) { id_ = value; }

    basic_point_view_vertex_t()                 = default;
    basic_point_view_vertex_t(self_type const&) = default;
    basic_point_view_vertex_t(self_type&&)      = default;
    self_type& operator=(self_type const&) = default;
    self_type& operator=(self_type&&) = default;
    explicit basic_point_view_vertex_t(PointView* point) : parent_type(point), id_(0u) {}
    explicit basic_point_view_vertex_t(id_type id) : parent_type(), id_(id) {}
    explicit basic_point_view_vertex_t(PointView* point, id_type id) : parent_type(point), id_(id) {}

    bool operator==(self_type const& other) const { return id_ == other.id_; }
    bool operator!=(self_type const& other) const { return id_ != other.id_; }

  private:
    id_type id_ = 0u;
};
using vertex_t = basic_point_view_vertex_t<point_t>;

template <class T>
struct basic_normal_t
{
    using component_type = T;
    basic_normal_t() = default;
    basic_normal_t(T x, T y, T z) : c_{x, y, z} {}
    T const& x() const { return c_[0]; }
    T const& y() const { return c_[1]; }
    T const& z() const { return c_[2]; }
    T const& nx() const { return c_[0]; }
    T const& ny() const { return c_[1]; }
    T const& nz() const { return c_[2]; }
    void x(T v) { c_[0] = v; }
    void y(T v) { c_[1] = v; }
    void z(T v) { c_[2] = v; }
    basic_normal_t operator-() const { return {-c_[0], -c_[1], -c_[2]}; }

  private:
    T c_[3] = {T(0), T(0), T(0)};
};
using normal_t = basic_normal_t<float>;

namespace common {
// common/vector3d_queries.hpp:31-35,48-64
template <class T>
bool floating_point_equals(T a, T b, T eps = static_cast<T>(1e-5))
{
    return std::abs(a - b) < eps;
}
template <class A, class B>
bool are_vectors_equal(A const& a, B const& b,
                       typename A::component_type eps = static_cast<typename A::component_type>(1e-5))
{
    return floating_point_equals(a.x(), b.x(), eps) && floating_point_equals(a.y(), b.y(), eps) &&
           floating_point_equals(a.z(), b.z(), eps);
}
// common/norm.hpp:60-82,102-112
template <class V>
typename V::component_type norm(V const& v)
{
    return std::sqrt(v.x() * v.x() + v.y() * v.y() + v.z() * v.z());
}
template <class P1, class P2>
typename P1::coordinate_type squared_distance(P1 const& p1, P2 const& p2)
{
    auto const dx = p2.x() - p1.x(), dy = p2.y() - p1.y(), dz = p2.z() - p1.z();
    return dx * dx + dy * dy + dz * dz;
}
} // namespace common

// ---- ranges (common/sphere.hpp:20-57, common/axis_aligned_bounding_box.hpp:99-149) ----------
template <class Point>
struct sphere_t
{
    Point position{0.f, 0.f, 0.f};
    typename Point::coordinate_type radius = 0;
    Point center() const { return position; }
    bool contains(Point const& p) const
    {
        return common::squared_distance(position, p) <= radius * radius;
    }
};

template <class T>
struct sphere_a
{
    using point_type = std::array<T, 3>;
    point_type position{};
    T radius{};
    point_type center() const { return position; }
    bool contains(point_type const& p) const
    {
        T const dx = p[0] - position[0], dy = p[1] - position[1], dz = p[2] - position[2];
        return dx * dx + dy * dy + dz * dz <= radius * radius;
    }
};

template <class Point>
struct axis_aligned_bounding_box_t
{
    using point_type = Point;
    Point min{0.f, 0.f, 0.f}, max{0.f, 0.f, 0.f};
    template <class P>
    bool contains(P const& p) const
    {
        return p.x() >= min.x() && p.y() >= min.y() && p.z() >= min.z() && p.x() <= max.x() &&
               p.y() <= max.y() && p.z() <= max.z();
    }
    Point center() const { return (min + max) / 2.f; }
    // common/axis_aligned_bounding_box.hpp:119-129
    template <class P>
    Point nearest_point_from(P const& p) const
    {
        return Point{std::clamp(p.x(), min.x(), max.x()), std::clamp(p.y(), min.y(), max.y()),
                     std::clamp(p.z(), min.z(), max.z())};
    }
};

// common/axis_aligned_bounding_box.hpp:12-77: the kd-tree's box over std::array coordinates
template <class CoordinateType, std::size_t K>
struct kd_axis_aligned_bounding_box_t
{
    using scalar_type = CoordinateType;
    using point_type  = std::array<CoordinateType, K>;
    point_type min{}, max{};
    bool contains(point_type const& p) const
    {
        for (std::size_t i = 0; i < K; ++i)
            if (!(p[i] >= min[i] && p[i] <= max[i]))
                return false;
        return true;
    }
    point_type center() const
    {
        point_type c{};
        for (std::size_t i = 0; i < K; ++i)
            c[i] = (min[i] + max[i]) / CoordinateType(2);
        return c;
    }
    point_type nearest_point_from(point_type const& p) const
    {
        point_type q = p;
        for (std::size_t i = 0; i < K; ++i)
            q[i] = std::clamp(q[i], min[i], max[i]);
        return q;
    }
};

// common/axis_aligned_bounding_box.hpp:214-251 (point views) and :164-201 (coordinate maps).
// Per-axis minima / maxima are exact in any order, so these host loops, the reference's
// accumulate / par for_each and the device bbox_kernel all agree bit for bit.
template <class ForwardIter, class Point, class AABB = axis_aligned_bounding_box_t<Point>>
inline AABB bounding_box(ForwardIter begin, ForwardIter end)
{
    using T = typename Point::coordinate_type;
    T lo[3] = {std::numeric_limits<T>::max(), std::numeric_limits<T>::max(),
               std::numeric_limits<T>::max()};
    T hi[3] = {std::numeric_limits<T>::lowest(), std::numeric_limits<T>::lowest(),
               std::numeric_limits<T>::lowest()};
    for (auto it = begin; it != end; ++it)
    {
        T const c[3] = {static_cast<T>(it->x()), static_cast<T>(it->y()), static_cast<T>(it->z())};
        for (int a = 0; a < 3; ++a)
            lo[a] = c[a] < lo[a] ? c[a] : lo[a], hi[a] = c[a] > hi[a] ? c[a] : hi[a];
    }
    AABB box;
    box.min = Point{lo[0], lo[1], lo[2]};
    box.max = Point{hi[0], hi[1], hi[2]};
    return box;
}
template <class CoordinateType, std::size_t K, class CoordinateMap, class ForwardIter>
inline kd_axis_aligned_bounding_box_t<CoordinateType, K>
kd_bounding_box(ForwardIter begin, ForwardIter end, CoordinateMap const& coordinate_map)
{
    kd_axis_aligned_bounding_box_t<CoordinateType, K> box;
    for (std::size_t i = 0; i < K; ++i)
        box.min[i] = std::numeric_limits<CoordinateType>::max(),
        box.max[i] = std::numeric_limits<CoordinateType>::lowest();
    for (auto it = begin; it != end; ++it)
    {
        auto const p = coordinate_map(*it);
        for (std::size_t i = 0; i < K; ++i)
            box.min[i] = p[i] < box.min[i] ? p[i] : box.min[i],
            box.max[i] = p[i] > box.max[i] ? p[i] : box.max[i];
    }
    return box;
}

// common/intersections.hpp:87-130.  The reference compares the SQUARED box distance with the
// un-squared radius (:101, :129) — the slip behind its missed points for radii above 1; these
// use radius * radius, the predicate the range searches of this library are built on.
template <class Point>
inline bool intersects(axis_aligned_bounding_box_t<Point> const& b, sphere_t<Point> const& s)
{
    Point const c = s.center();
    if (b.contains(c))
        return true;
    return common::squared_distance(b.nearest_point_from(c), c) <= s.radius * s.radius;
}
template <class CoordinateType>
inline bool intersects(kd_axis_aligned_bounding_box_t<CoordinateType, 3> const& b,
                       sphere_a<CoordinateType> const& s)
{
    auto const c = s.center();
    if (b.contains(c))
        return true;
    auto const q = b.nearest_point_from(c);
    CoordinateType const dx = q[0] - c[0], dy = q[1] - c[1], dz = q[2] - c[2];
    return dx * dx + dy * dy + dz * dz <= s.radius * s.radius;
}

// ---- index parameters (octree/linked_octree_node.hpp:31-40, kdtree/linked_kdtree.hpp:26-33):
// accepted for source compatibility; tree shape does not change exact results, only the voxel
// grid does (points outside it are not indexed).
template <class Point>
struct octree_parameters_t
{
    using point_type = Point;
    using aabb_type  = axis_aligned_bounding_box_t<Point>;
    std::uint32_t node_capacity = 32u;
    std::uint8_t max_depth      = 21u;
    aabb_type voxel_grid{};
};
namespace kdtree {
enum class construction_t { nth_element, presort };
struct construction_params_t
{
    std::size_t max_depth                           = 12u;
    construction_t construction                     = construction_t::nth_element;
    std::size_t min_element_count_for_parallel_exec = 32'768;
    bool compute_max_depth                          = false;
    std::size_t max_elements_per_leaf               = 64u;
};
} // namespace kdtree

namespace execution {
struct gpu_policy
{
};
inline constexpr gpu_policy gpu{}; // accepted wherever the reference takes a std::execution policy
} // namespace execution

// ---- the device index ----------------------------------------------------------------------
namespace detail {
inline void check(int rc, char const* what)
{
    if (rc != PCPX_OK)
        throw std::runtime_error(std::string(what) + ": " + pcpx_last_error());
}
struct index_deleter
{
    void operator()(pcpx_index* p) const { pcpx_index_destroy(p); }
};
using index_ptr = std::unique_ptr<pcpx_index, index_deleter>;

inline std::vector<int>& device_list()
{
    static std::vector<int> devices; // empty: the current device
    return devices;
}
// Page-locked host buffer (pcpx_host_alloc): what the flattened clouds and the results of the
// batched calls are staged in — pageable memory costs ~5x on both PCIe transfers.
// (page-locking is expensive — ~0.5 ms per MB —, so released blocks are kept, a few of them, and
// handed out again: a loop that builds a tree and estimates normals per cloud pins its staging
// memory once)
class pinned_pool
{
  public:
    static pinned_pool& instance()
    {
        static pinned_pool* p = new pinned_pool(); // (never destroyed: outlives every buffer)
        return *p;
    }
    void* acquire(std::size_t bytes, std::size_t& got)
    {
        {
            std::lock_guard<std::mutex> lock(m_);
            std::size_t best = blocks_.size();
            for (std::size_t i = 0; i < blocks_.size(); ++i)
                if (blocks_[i].second >= bytes && blocks_[i].second <= 2 * bytes + 4096 &&
                    (best == blocks_.size() || blocks_[i].second < blocks_[best].second))
                    best = i;
            if (best != blocks_.size())
            {
                void* p = blocks_[best].first;
                got     = blocks_[best].second;
                blocks_.erase(blocks_.begin() + static_cast<std::ptrdiff_t>(best));
                return p;
            }
        }
        void* raw = nullptr;
        check(pcpx_host_alloc(bytes, &raw), "pcpx_host_alloc");
        got = bytes;
        return raw;
    }
    void release(void* p, std::size_t bytes)
    {
        if (!p)
            return;
        {
            std::lock_guard<std::mutex> lock(m_);
            if (blocks_.size() < 6)
            {
                blocks_.emplace_back(p, bytes);
                return;
            }
        }
        pcpx_host_free(p);
    }

  private:
    std::mutex m_;
    std::vector<std::pair<void*, std::size_t>> blocks_;
};

template <class T>
class pinned_buffer
{
  public:
    pinned_buffer() = default;
    explicit pinned_buffer(std::size_t n) { reset(n); }
    ~pinned_buffer() { pinned_pool::instance().release(p_, bytes_); }
    pinned_buffer(pinned_buffer const&)            = delete;
    pinned_buffer& operator=(pinned_buffer const&) = delete;
    void reset(std::size_t n)
    {
        pinned_pool::instance().release(p_, bytes_);
        p_ = nullptr, n_ = 0, bytes_ = 0;
        if (n == 0)
            return;
        p_ = static_cast<T*>(pinned_pool::instance().acquire(n * sizeof(T), bytes_));
        n_ = n;
    }
    T* data() { return p_; }
    T const* data() const { return p_; }
    std::size_t size() const { return n_; }
    T& operator[](std::size_t i) { return p_[i]; }
    T const& operator[](std::size_t i) const { return p_[i]; }

  private:
    T* p_              = nullptr;
    std::size_t n_     = 0;
    std::size_t bytes_ = 0;
};

// f(first, last) over [0, n) cut into contiguous chunks, one host thread per chunk (the
// element-wise loops either side of a device call — flattening 10 M points, handing 10 M normals
// to the transform — cost more than the call itself when they run on one core)
template <class F>
void parallel_chunks(std::size_t n, F&& f)
{
    unsigned const hw      = std::thread::hardware_concurrency();
    std::size_t const want = n / 65536u;
    std::size_t const t    = std::min<std::size_t>({want, hw ? hw : 1u, 16u});
    if (t <= 1)
    {
        f(std::size_t{0}, n);
        return;
    }
    std::vector<std::thread> threads;
    threads.reserve(t - 1);
    std::size_t const step = (n + t - 1) / t;
    for (std::size_t c = 1; c < t; ++c)
        threads.emplace_back([&f, c, step, n] { f(std::min(n, c * step), std::min(n, (c + 1) * step)); });
    f(std::size_t{0}, std::min(n, step));
    for (auto& th : threads)
        th.join();
}
template <class Iter>
inline constexpr bool is_random_access_v =
    std::is_base_of_v<std::random_access_iterator_tag,
                      typename std::iterator_traits<Iter>::iterator_category>;

inline index_ptr make_index(float const* xyz, std::size_t n, pcpx_index_params const& prm0);
inline index_ptr make_index(std::vector<float> const& xyz, pcpx_index_params const& prm0)
{
    return make_index(xyz.data(), xyz.size() / 3, prm0);
}
inline index_ptr make_index(float const* xyz, std::size_t n, pcpx_index_params const& prm0)
{
    pcpx_index_params prm = prm0;
    std::vector<int> const& devs = device_list();
    if (prm.n_devices == 0 && !devs.empty())
    {
        prm.n_devices = static_cast<std::uint32_t>(devs.size() < 8 ? devs.size() : 8);
        for (std::uint32_t i = 0; i < prm.n_devices; ++i)
            prm.devices[i] = devs[i];
    }
    pcpx_index* raw = nullptr;
    check(pcpx_index_create(xyz, n, 12, &prm, &raw), "pcpx_index_create");
    return index_ptr(raw);
}
// fp32 bounds that contain [v, v] when v is wider than float
template <class T>
float round_down_f32(T v)
{
    float const f = static_cast<float>(v);
    if constexpr (std::is_same_v<T, float>)
        return f;
    else
        return static_cast<T>(f) > v ? std::nextafter(f, -std::numeric_limits<float>::infinity()) : f;
}
template <class T>
float round_up_f32(T v)
{
    float const f = static_cast<float>(v);
    if constexpr (std::is_same_v<T, float>)
        return f;
    else
        return static_cast<T>(f) < v ? std::nextafter(f, std::numeric_limits<float>::infinity()) : f;
}
template <class R, class = void>
struct is_aabb : std::false_type
{
};
template <class R>
struct is_aabb<R, std::void_t<decltype(std::declval<R const&>().min),
                              decltype(std::declval<R const&>().max)>> : std::true_type
{
};
template <class R>
inline constexpr bool is_aabb_v = is_aabb<R>::value;
template <class PV>
void push_xyz(std::vector<float>& out, PV const& p)
{
    out.push_back(static_cast<float>(p.x()));
    out.push_back(static_cast<float>(p.y()));
    out.push_back(static_cast<float>(p.z()));
}
} // namespace detail

// GPUs used by every tree built from now on (the reference's constructors have nowhere to say
// it): the index is replicated on all of them and the batched kNN-shaped calls
// (nearest_neighbours batches, estimate_normals / estimate_tangent_planes with a gpu_knn_map,
// average_distance_to_neighbors) are sharded over them; devices[0] holds the results.  An empty
// list (the default) means the current device.  See pcpx_index_params.devices (pcpx.h).
inline void use_devices(std::vector<int> devices) { detail::device_list() = std::move(devices); }
inline int device_count() { return pcpx_device_count(); }

// Flat result of a batched kNN: row i holds counts[i] valid original indices, nearest first.
struct knn_result_t
{
    std::size_t k = 0;
    std::vector<std::uint32_t> indices; // n_queries x k, padded with PCPX_NO_NEIGHBOUR
    std::vector<float> squared_distances;
    std::vector<std::uint32_t> counts;
    std::size_t size() const { return counts.size(); }
};

// Shared machinery of the two container facades: element storage + the GPU index.
template <class Element>
class device_spatial_index
{
  public:
    using element_type = Element;

    std::size_t size() const { return n_indexed_; }
    bool empty() const { return size() == 0u; }
    pcpx_index const* handle() const { return index_.get(); }
    // Are these n flattened query points the indexed cloud itself, in its original order?  Then a
    // batched call passes queries == NULL and takes the tile kernel instead of sorting and
    // searching them as foreign points (same rows: exclusion is by coordinates, not identity).
    bool is_own_cloud(float const* xyz, std::size_t n) const
    {
        if (n == 0 || n != elements_.size() || xyz_.size() != 3 * n)
            return false;
        std::atomic<bool> same{true};
        detail::parallel_chunks(n, [&](std::size_t first, std::size_t last) {
            if (std::memcmp(xyz + 3 * first, xyz_.data() + 3 * first, 12 * (last - first)) != 0)
                same.store(false, std::memory_order_relaxed);
        });
        return same.load();
    }
    std::vector<Element> const& elements() const { return elements_; }

    knn_result_t knn_batch(std::vector<float> const& queries, std::size_t k, double eps) const
    {
        knn_result_t r;
        r.k               = k;
        std::size_t const n = queries.size() / 3;
        r.counts.assign(n, 0u);
        if (k == 0 || n == 0)
            return r;
        r.indices.assign(n * k, PCPX_NO_NEIGHBOUR);
        r.squared_distances.assign(n * k, std::numeric_limits<float>::infinity());
        detail::check(pcpx_knn(index_.get(), queries.data(), n, 12, static_cast<std::uint32_t>(k),
                               eps, r.indices.data(), r.squared_distances.data(), r.counts.data()),
                      "pcpx_knn");
        return r;
    }

    std::vector<Element> gather(std::uint32_t const* idx, std::size_t n) const
    {
        std::vector<Element> out;
        out.reserve(n);
        for (std::size_t j = 0; j < n; ++j)
            out.push_back(elements_[idx[j]]);
        return out;
    }

    // sphere range search, CSR over original indices
    void radius_batch(std::vector<float> const& centres, std::vector<float> const& radii,
                      std::vector<std::uint64_t>& offsets, std::vector<std::uint32_t>& idx) const
    {
        std::size_t const n = centres.size() / 3;
        offsets.assign(n + 1, 0u);
        std::uint32_t* lists = nullptr;
        // (lists ascending by original index: a defined order costs one small kernel)
        detail::check(pcpx_radius_search(index_.get(), centres.data(), n, 12, radii.data(), 0.f,
                                         offsets.data(), &lists, PCPX_RADIUS_SORTED),
                      "pcpx_radius_search");
        idx.assign(lists, lists + offsets[n]);
        pcpx_free(lists, 0);
    }

    // box range search, CSR over original indices, every list ascending
    void box_batch(std::vector<float> const& boxes, std::vector<std::uint64_t>& offsets,
                   std::vector<std::uint32_t>& idx) const
    {
        std::size_t const n = boxes.size() / 6;
        offsets.assign(n + 1, 0u);
        std::uint32_t* lists = nullptr;
        detail::check(pcpx_box_search(index_.get(), boxes.data(), n, 24, offsets.data(), &lists,
                                      PCPX_RADIUS_SORTED),
                      "pcpx_box_search");
        idx.assign(lists, lists + offsets[n]);
        pcpx_free(lists, 0);
    }
    // one box as 6 fp32 values, rounded outward when the coordinates are wider than float (a
    // NaN bound stays NaN: the box is empty either way)
    template <class T>
    static void push_box(std::vector<float>& out, T const (&mn)[3], T const (&mx)[3])
    {
        for (int a = 0; a < 3; ++a)
            out.push_back(detail::round_down_f32(mn[a]));
        for (int a = 0; a < 3; ++a)
            out.push_back(detail::round_up_f32(mx[a]));
    }

  protected:
    template <class ForwardIter, class ToXyz>
    void build(ForwardIter begin, ForwardIter end, ToXyz&& to_xyz, pcpx_index_params const& prm)
    {
        if constexpr (detail::is_random_access_v<ForwardIter>)
        {
            // The tree's own copy of the elements (the reference's nodes hold copies too) is the
            // longest single piece of the constructor — 30 ms for 10 M points on one core —, and
            // nothing below needs it: it runs on a helper thread while the coordinates are
            // flattened straight from the caller's range, uploaded and indexed.
            std::size_t const n = static_cast<std::size_t>(std::distance(begin, end));
            std::exception_ptr copy_error;
            struct joiner
            {
                std::thread t;
                ~joiner()
                {
                    if (t.joinable())
                        t.join();
                }
            } copier{std::thread([&] {
                try
                {
                    elements_.assign(begin, end);
                }
                catch (...)
                {
                    copy_error = std::current_exception();
                }
            })};
            xyz_.reset(3 * n); // pinned: one DMA at PCIe speed; kept (is_own_cloud)
            detail::parallel_chunks(n, [&](std::size_t first, std::size_t last) {
                for (std::size_t i = first; i < last; ++i)
                    to_xyz(xyz_.data() + 3 * i, begin[static_cast<std::ptrdiff_t>(i)]);
            });
            index_ = detail::make_index(xyz_.data(), n, prm);
            copier.t.join();
            if (copy_error)
                std::rethrow_exception(copy_error);
        }
        else
        {
            elements_.assign(begin, end);
            std::size_t const n = elements_.size();
            xyz_.reset(3 * n);
            for (std::size_t i = 0; i < n; ++i)
                to_xyz(xyz_.data() + 3 * i, elements_[i]);
            index_ = detail::make_index(xyz_.data(), n, prm);
        }
        pcpx_index_info info{};
        detail::check(pcpx_index_info_get(index_.get(), &info), "pcpx_index_info_get");
        n_indexed_ = static_cast<std::size_t>(info.n_indexed);
        for (int a = 0; a < 3; ++a)
            bbox_[a] = info.bbox_min[a], bbox_[3 + a] = info.bbox_max[a];
    }

    std::vector<Element> elements_;
    detail::pinned_buffer<float> xyz_; // the elements' coordinates, original order
    detail::index_ptr index_;
    std::size_t n_indexed_ = 0;
    float bbox_[6]         = {0, 0, 0, 0, 0, 0};
};

// ---- octree facade (octree/linked_octree.hpp:40-283) ---------------------------------------
template <class Element, class ParamsType = octree_parameters_t<pcp::point_t>>
class basic_linked_octree_t : public device_spatial_index<Element>
{
    using base = device_spatial_index<Element>;

  public:
    using element_type    = Element;
    using params_type     = ParamsType;
    using aabb_type       = typename ParamsType::aabb_type;
    using aabb_point_type = typename aabb_type::point_type;
    using value_type      = Element;

    basic_linked_octree_t(basic_linked_octree_t&&) = default;

    // octree/linked_octree.hpp:71: an empty octree over a given voxel grid, filled by insert()
    explicit basic_linked_octree_t(params_type const& params) : params_(params), has_params_(true) {}

    // octree/linked_octree.hpp:179-206.  The device index is immutable, so an insertion rebuilds
    // it over everything inserted so far (a few ms per 10 M points): insert ranges, not single
    // elements in a loop.  Like the reference, elements outside the voxel grid are rejected
    // (octree/linked_octree_node.hpp:174) and not counted.
    template <class ForwardIter, class PointViewMap>
    std::size_t insert(ForwardIter begin, ForwardIter end, PointViewMap const& point_view)
    {
        std::vector<element_type> all = this->elements_;
        std::size_t inserted          = 0;
        for (auto it = begin; it != end; ++it)
            if (!has_params_ || params_.voxel_grid.contains(point_view(*it)))
            {
                all.push_back(*it);
                ++inserted;
            }
        if (inserted)
        {
            pcpx_index_params prm{};
            prm.device = -1;
            if (has_params_)
                set_voxel_grid(prm, params_);
            construct(all.begin(), all.end(), point_view, prm);
        }
        return inserted;
    }
    template <class PointViewMap>
    bool insert(element_type const& e, PointViewMap const& point_view)
    {
        return insert(&e, &e + 1, point_view) == 1u;
    }

    // octree/linked_octree.hpp:83-91: explicit voxel grid — elements outside it are not indexed
    template <class ForwardIter, class PointViewMap>
    explicit basic_linked_octree_t(ForwardIter begin, ForwardIter end,
                                   PointViewMap const& point_view, params_type const& params)
    {
        pcpx_index_params prm{};
        prm.device = -1;
        set_voxel_grid(prm, params);
        params_ = params, has_params_ = true;
        construct(begin, end, point_view, prm);
    }

    // octree/linked_octree.hpp:103-121: bounding box computed from the elements
    template <class ForwardIter, class PointViewMap>
    explicit basic_linked_octree_t(ForwardIter begin, ForwardIter end,
                                   PointViewMap const& point_view)
    {
        pcpx_index_params prm{};
        prm.device = -1;
        construct(begin, end, point_view, prm);
    }

    aabb_type voxel_grid() const
    {
        aabb_type b;
        b.min = aabb_point_type{this->bbox_[0], this->bbox_[1], this->bbox_[2]};
        b.max = aabb_point_type{this->bbox_[3], this->bbox_[4], this->bbox_[5]};
        return b;
    }

    // octree/linked_octree.hpp:245-254 (one kernel launch per call: prefer the batched overload)
    template <class TPointView, class PointViewMap>
    std::vector<element_type> nearest_neighbours(TPointView const& target, std::size_t k,
                                                 PointViewMap const&, double eps = 1e-5) const
    {
        std::vector<float> q;
        detail::push_xyz(q, target);
        knn_result_t const r = this->knn_batch(q, k, eps);
        return this->gather(r.indices.data(), r.counts.empty() ? 0u : r.counts[0]);
    }

    // batched: one target per element of [begin, end)
    template <class ForwardIter, class PointViewMap>
    knn_result_t nearest_neighbours(ForwardIter begin, ForwardIter end, std::size_t k,
                                    PointViewMap const& point_view, double eps = 1e-5) const
    {
        std::vector<float> q;
        for (auto it = begin; it != end; ++it)
            detail::push_xyz(q, point_view(*it));
        return this->knn_batch(q, k, eps);
    }

    // octree/linked_octree.hpp:264-276 for the sphere range
    template <class Point, class PointViewMap>
    std::vector<element_type> range_search(sphere_t<Point> const& range, PointViewMap const&) const
    {
        std::vector<float> c, r{static_cast<float>(range.radius)};
        detail::push_xyz(c, range.position);
        std::vector<std::uint64_t> off;
        std::vector<std::uint32_t> idx;
        this->radius_batch(c, r, off, idx);
        return this->gather(idx.data(), idx.size());
    }

    // ... and for the box range (pcpx_box_search)
    template <class Point, class PointViewMap>
    std::vector<element_type> range_search(axis_aligned_bounding_box_t<Point> const& range,
                                           PointViewMap const& point_view) const
    {
        std::vector<float> b;
        this->push_box(b, {range.min.x(), range.min.y(), range.min.z()},
                       {range.max.x(), range.max.y(), range.max.z()});
        std::vector<std::uint64_t> off;
        std::vector<std::uint32_t> idx;
        this->box_batch(b, off, idx);
        if constexpr (std::is_same_v<std::decay_t<decltype(range.min.x())>, float>)
            return this->gather(idx.data(), idx.size());
        else
        {
            // the box was rounded outward to fp32: the exact predicate on what it returned
            std::vector<element_type> out;
            for (auto i : idx)
                if (range.contains(point_view(this->elements_[i])))
                    out.push_back(this->elements_[i]);
            return out;
        }
    }

    // batched sphere or box ranges -> CSR (offsets, original indices), every list ascending
    template <class RangeIter>
    void range_search(RangeIter begin, RangeIter end, std::vector<std::uint64_t>& offsets,
                      std::vector<std::uint32_t>& indices) const
    {
        using range_type = typename std::iterator_traits<RangeIter>::value_type;
        if constexpr (detail::is_aabb_v<range_type>)
        {
            std::vector<float> b;
            for (auto it = begin; it != end; ++it)
                this->push_box(b, {it->min.x(), it->min.y(), it->min.z()},
                               {it->max.x(), it->max.y(), it->max.z()});
            this->box_batch(b, offsets, indices);
        }
        else
        {
            std::vector<float> c, r;
            for (auto it = begin; it != end; ++it)
            {
                detail::push_xyz(c, it->position);
                r.push_back(static_cast<float>(it->radius));
            }
            this->radius_batch(c, r, offsets, indices);
        }
    }

  private:
    static void set_voxel_grid(pcpx_index_params& prm, params_type const& params)
    {
        prm.use_voxel_grid = 1;
        prm.voxel_min[0] = params.voxel_grid.min.x(), prm.voxel_min[1] = params.voxel_grid.min.y(),
        prm.voxel_min[2] = params.voxel_grid.min.z();
        prm.voxel_max[0] = params.voxel_grid.max.x(), prm.voxel_max[1] = params.voxel_grid.max.y(),
        prm.voxel_max[2] = params.voxel_grid.max.z();
    }

    params_type params_{};
    bool has_params_ = false;

    template <class ForwardIter, class PointViewMap>
    void construct(ForwardIter begin, ForwardIter end, PointViewMap const& point_view,
                   pcpx_index_params const& prm)
    {
        this->build(begin, end,
                    [&](float* xyz, element_type const& e) {
                        auto const p = point_view(e);
                        xyz[0] = static_cast<float>(p.x()), xyz[1] = static_cast<float>(p.y());
                        xyz[2] = static_cast<float>(p.z());
                    },
                    prm);
    }
};
using linked_octree_t = basic_linked_octree_t<pcp::point_t>;

// ---- kd-tree facade (kdtree/linked_kdtree.hpp:64-560); K = 3 only ---------------------------
template <class Element, std::size_t K, class CoordinateMap>
class basic_linked_kdtree_t : public device_spatial_index<Element>
{
    static_assert(K == 3, "the GPU index is three-dimensional");

  public:
    using element_type     = Element;
    using coordinates_type = std::invoke_result_t<CoordinateMap, Element>;
    using coordinate_type  = typename coordinates_type::value_type;

    template <class ForwardIter>
    basic_linked_kdtree_t(ForwardIter begin, ForwardIter end,
                          CoordinateMap coordinate_map         = CoordinateMap{},
                          kdtree::construction_params_t params = kdtree::construction_params_t{})
        : coordinate_map_(coordinate_map)
    {
        (void)params; // median-split depth has no counterpart in the grid index
        pcpx_index_params prm{};
        prm.device = -1;
        this->build(begin, end,
                    [&](float* xyz, element_type const& e) {
                        auto const c = coordinate_map_(e);
                        xyz[0] = static_cast<float>(c[0]), xyz[1] = static_cast<float>(c[1]);
                        xyz[2] = static_cast<float>(c[2]);
                    },
                    prm);
    }

    // kdtree/linked_kdtree.hpp:200-244
    std::vector<element_type> nearest_neighbours(coordinates_type const& target, std::size_t k,
                                                 coordinate_type eps = static_cast<coordinate_type>(1e-5)) const
    {
        std::vector<float> q{static_cast<float>(target[0]), static_cast<float>(target[1]),
                             static_cast<float>(target[2])};
        knn_result_t const r = this->knn_batch(q, k, static_cast<double>(eps));
        return this->gather(r.indices.data(), r.counts.empty() ? 0u : r.counts[0]);
    }
    // kdtree/linked_kdtree.hpp:256-263
    std::vector<element_type> nearest_neighbours(element_type const& e, std::size_t k,
                                                 coordinate_type eps = static_cast<coordinate_type>(1e-5)) const
    {
        return nearest_neighbours(coordinate_map_(e), k, eps);
    }
    // batched over elements
    template <class ForwardIter>
    knn_result_t nearest_neighbours(ForwardIter begin, ForwardIter end, std::size_t k,
                                    coordinate_type eps = static_cast<coordinate_type>(1e-5)) const
    {
        std::vector<float> q;
        for (auto it = begin; it != end; ++it)
        {
            auto const c = coordinate_map_(*it);
            q.insert(q.end(), {static_cast<float>(c[0]), static_cast<float>(c[1]),
                               static_cast<float>(c[2])});
        }
        return this->knn_batch(q, k, static_cast<double>(eps));
    }
    // kdtree/linked_kdtree.hpp:270-316 for the kd box range (pcpx_box_search).  Coordinates other
    // than float: the box is rounded outward to fp32 and the exact predicate filters the result.
    std::vector<element_type>
    range_search(kd_axis_aligned_bounding_box_t<coordinate_type, 3> const& range) const
    {
        std::vector<float> b;
        this->push_box(b, {range.min[0], range.min[1], range.min[2]},
                       {range.max[0], range.max[1], range.max[2]});
        std::vector<std::uint64_t> off;
        std::vector<std::uint32_t> idx;
        this->box_batch(b, off, idx);
        if constexpr (std::is_same_v<coordinate_type, float>)
            return this->gather(idx.data(), idx.size());
        else
        {
            std::vector<element_type> out;
            for (auto i : idx)
                if (range.contains(coordinate_map_(this->elements_[i])))
                    out.push_back(this->elements_[i]);
            return out;
        }
    }
    // batched kd boxes -> CSR (offsets, original indices), every list ascending; non-float
    // coordinates as above, with each list filtered by the exact predicate
    template <class BoxIter>
    void range_search(BoxIter begin, BoxIter end, std::vector<std::uint64_t>& offsets,
                      std::vector<std::uint32_t>& indices) const
    {
        std::vector<float> b;
        for (auto it = begin; it != end; ++it)
            this->push_box(b, {it->min[0], it->min[1], it->min[2]},
                           {it->max[0], it->max[1], it->max[2]});
        this->box_batch(b, offsets, indices);
        if constexpr (!std::is_same_v<coordinate_type, float>)
        {
            std::vector<std::uint64_t> off{0u};
            std::vector<std::uint32_t> kept;
            std::size_t q = 0;
            for (auto it = begin; it != end; ++it, ++q)
            {
                for (std::uint64_t j = offsets[q]; j < offsets[q + 1]; ++j)
                    if (it->contains(coordinate_map_(this->elements_[indices[j]])))
                        kept.push_back(indices[j]);
                off.push_back(kept.size());
            }
            offsets.swap(off), indices.swap(kept);
        }
    }
    // kdtree/linked_kdtree.hpp:270-277 for sphere_a
    std::vector<element_type> range_search(sphere_a<coordinate_type> const& range) const
    {
        std::vector<float> c{static_cast<float>(range.position[0]),
                             static_cast<float>(range.position[1]),
                             static_cast<float>(range.position[2])};
        std::vector<float> r{static_cast<float>(range.radius)};
        std::vector<std::uint64_t> off;
        std::vector<std::uint32_t> idx;
        this->radius_batch(c, r, off, idx);
        return this->gather(idx.data(), idx.size());
    }

  private:
    CoordinateMap coordinate_map_;
};

// ---- KnnMap that the algorithms recognise ---------------------------------------------------
// A KnnMap (traits/knn_map.hpp:22-45) bound to a device index and a k.  Calling it answers one
// query like any other KnnMap; handing it to estimate_normals / average_distance(s)_to_neighbors
// lets them run the whole range as one fused device call.
template <class Index, class PointViewMap>
struct gpu_knn_map
{
    Index const* index;
    std::size_t k;
    PointViewMap point_view;
    double eps = 1e-5;

    template <class Key>
    std::vector<typename Index::element_type> operator()(Key const& key) const
    {
        std::vector<float> q;
        detail::push_xyz(q, point_view(key));
        knn_result_t const r = index->knn_batch(q, k, eps);
        return index->gather(r.indices.data(), r.counts.empty() ? 0u : r.counts[0]);
    }
};
template <class Index, class PointViewMap>
gpu_knn_map<Index, PointViewMap> make_gpu_knn_map(Index const& index, std::size_t k,
                                                  PointViewMap point_view, double eps = 1e-5)
{
    return gpu_knn_map<Index, PointViewMap>{&index, k, point_view, eps};
}
namespace detail {
template <class T>
struct is_gpu_knn_map : std::false_type
{
};
template <class I, class P>
struct is_gpu_knn_map<gpu_knn_map<I, P>> : std::true_type
{
};
} // namespace detail

// The ball counterpart: a KnnMap bound to a device index and a radius.  Called on one element it
// answers like `[&](auto const& e) { return index.range_search(sphere_t{point_view(e), radius},
// point_view); }` (octree/linked_octree.hpp:264-276, common/sphere.hpp:27-35); handed to
// estimate_normals it makes the whole range one fused ball -> PCA device call.
template <class Index, class PointViewMap>
struct gpu_radius_map
{
    Index const* index;
    float radius;
    PointViewMap point_view;

    template <class Key>
    std::vector<typename Index::element_type> operator()(Key const& key) const
    {
        std::vector<float> c, r{radius};
        detail::push_xyz(c, point_view(key));
        std::vector<std::uint64_t> off;
        std::vector<std::uint32_t> idx;
        index->radius_batch(c, r, off, idx);
        return index->gather(idx.data(), idx.size());
    }
};
template <class Index, class PointViewMap>
gpu_radius_map<Index, PointViewMap> make_gpu_radius_map(Index const& index, float radius,
                                                        PointViewMap point_view)
{
    return gpu_radius_map<Index, PointViewMap>{&index, radius, point_view};
}
namespace detail {
template <class T>
struct is_gpu_radius_map : std::false_type
{
};
template <class I, class P>
struct is_gpu_radius_map<gpu_radius_map<I, P>> : std::true_type
{
};
} // namespace detail

// common/normals/normal_estimation.hpp:32-78 for ONE neighbourhood (a device call; batch instead)
template <class ForwardIter, class PointViewMap, class Normal = pcp::normal_t>
Normal estimate_normal(ForwardIter it, ForwardIter end, PointViewMap const& point_map)
{
    std::vector<float> nbr;
    for (; it != end; ++it)
        detail::push_xyz(nbr, point_map(*it));
    std::uint64_t const off[2] = {0u, nbr.size() / 3};
    float n[3]                 = {0.f, 0.f, 0.f};
    detail::check(pcpx_normals_from_neighbourhoods(nbr.data(), off, 1, -1, n),
                  "pcpx_normals_from_neighbourhoods");
    return Normal{n[0], n[1], n[2]};
}

namespace algorithm {

// algorithm/common.hpp:31-34
template <class Input, class Normal>
inline auto const default_normal_transform = [](Input const&, Normal const& n) {
    return n;
};

// algorithm/estimate_normals.hpp:116-164 (no execution policy)
template <class ForwardIter1, class ForwardIter2, class PointViewMap, class KnnMap,
          class TransformOp, class Normal = pcp::normal_t>
void estimate_normals(ForwardIter1 begin, ForwardIter1 end, ForwardIter2 out_begin,
                      PointViewMap const& point_map, KnnMap&& knn_map, TransformOp&& op)
{
    using knn_type      = std::decay_t<KnnMap>;
    std::size_t const n = static_cast<std::size_t>(std::distance(begin, end));
    detail::pinned_buffer<float> normals(3 * n);
    if constexpr (detail::is_gpu_knn_map<knn_type>::value || detail::is_gpu_radius_map<knn_type>::value)
    {
        // the whole range in ONE fused kNN (or ball) -> scatter matrix -> eigensolve call
        detail::pinned_buffer<float> q(3 * n);
        auto const put = [&](std::size_t i, auto const& element) {
            auto const p = point_map(element);
            q[3 * i] = static_cast<float>(p.x()), q[3 * i + 1] = static_cast<float>(p.y());
            q[3 * i + 2] = static_cast<float>(p.z());
        };
        if constexpr (detail::is_random_access_v<ForwardIter1>)
            detail::parallel_chunks(n, [&](std::size_t first, std::size_t last) {
                for (std::size_t i = first; i < last; ++i)
                    put(i, begin[static_cast<std::ptrdiff_t>(i)]);
            });
        else
        {
            std::size_t i = 0;
            for (auto it = begin; it != end; ++it, ++i)
                put(i, *it);
        }
        // the range is the indexed cloud itself (the usual call): no query upload, no query
        // sort, the tile kernel
        bool const own = knn_map.index->is_own_cloud(q.data(), n);
        if constexpr (detail::is_gpu_knn_map<knn_type>::value)
            detail::check(pcpx_estimate_normals(knn_map.index->handle(), own ? nullptr : q.data(), n,
                                                12, static_cast<std::uint32_t>(knn_map.k),
                                                knn_map.eps, normals.data()),
                          "pcpx_estimate_normals");
        else
            detail::check(pcpx_estimate_normals_radius(knn_map.index->handle(),
                                                       own ? nullptr : q.data(), n, 12, nullptr,
                                                       knn_map.radius, normals.data(), nullptr),
                          "pcpx_estimate_normals_radius");
    }
    else
    {
        // arbitrary KnnMap: the map is called per element as in the reference
        // (algorithm/estimate_normals.hpp:80-90); only the PCA is batched, on the device
        std::vector<float> nbr;
        std::vector<std::uint64_t> off(1, 0u);
        for (auto it = begin; it != end; ++it)
        {
            auto const neighbours = knn_map(*it);
            for (auto const& e : neighbours)
                detail::push_xyz(nbr, point_map(e));
            off.push_back(nbr.size() / 3);
        }
        detail::check(pcpx_normals_from_neighbourhoods(nbr.data(), off.data(), n, -1,
                                                       normals.data()),
                      "pcpx_normals_from_neighbourhoods");
    }
    if constexpr (detail::is_random_access_v<ForwardIter1> && detail::is_random_access_v<ForwardIter2>)
        detail::parallel_chunks(n, [&](std::size_t first, std::size_t last) {
            for (std::size_t i = first; i < last; ++i)
                out_begin[static_cast<std::ptrdiff_t>(i)] =
                    op(begin[static_cast<std::ptrdiff_t>(i)],
                       Normal{normals[3 * i], normals[3 * i + 1], normals[3 * i + 2]});
        });
    else
    {
        std::size_t i = 0;
        for (auto it = begin; it != end; ++it, ++i, ++out_begin)
            *out_begin = op(*it, Normal{normals[3 * i], normals[3 * i + 1], normals[3 * i + 2]});
    }
}

// algorithm/estimate_normals.hpp:50-93 (execution policy accepted and ignored: the device call
// is already data-parallel)
template <class ExecutionPolicy, class ForwardIter1, class ForwardIter2, class PointViewMap,
          class KnnMap, class TransformOp, class Normal = pcp::normal_t,
          class = std::enable_if_t<
              std::is_execution_policy_v<std::decay_t<ExecutionPolicy>> ||
              std::is_same_v<std::decay_t<ExecutionPolicy>, pcp::execution::gpu_policy>>>
void estimate_normals(ExecutionPolicy&&, ForwardIter1 begin, ForwardIter1 end,
                      ForwardIter2 out_begin, PointViewMap const& point_map, KnnMap&& knn_map,
                      TransformOp&& op)
{
    estimate_normals<ForwardIter1, ForwardIter2, PointViewMap, KnnMap, TransformOp, Normal>(
        begin, end, out_begin, point_map, std::forward<KnnMap>(knn_map),
        std::forward<TransformOp>(op));
}

// algorithm/estimate_normals.hpp:187-302.  Same signature and same result as the reference's
// sequential breadth-first propagation (built with libstdc++, see pcpx.h: edge_order); the kNN
// graph is gathered on the host from `knn_map` (one batched device call when it is a
// gpu_knn_map), the search itself runs on the GPU.  `op(element, normal)` is invoked for the
// root with (0, 0, 1) and for every element whose normal was negated — the same set of calls
// the reference makes, in input order instead of search order.  `edge_order` is a pcpx
// extension (default: what the reference does under libstdc++).
template <class ForwardIter1, class IndexMap, class KnnMap, class PointViewMap, class NormalMap,
          class TransformOp>
void propagate_normal_orientations(ForwardIter1 begin, ForwardIter1 end, IndexMap const& index_map,
                                   KnnMap&& knn_map, PointViewMap&& point_map,
                                   NormalMap& normal_map, TransformOp&& op,
                                   int edge_order = PCPX_EDGES_FURTHEST_FIRST)
{
    using knn_type    = std::decay_t<KnnMap>;
    using normal_type = std::decay_t<decltype(normal_map(*begin))>;
    using scalar_type = typename normal_type::component_type;
    std::size_t const n = static_cast<std::size_t>(std::distance(begin, end));
    if (n == 0)
        return;
    std::vector<float> xyz, nrm;
    xyz.reserve(3 * n), nrm.reserve(3 * n);
    for (auto it = begin; it != end; ++it)
    {
        detail::push_xyz(xyz, point_map(*it));
        auto const nn = normal_map(*it);
        nrm.push_back(static_cast<float>(nn.nx()));
        nrm.push_back(static_cast<float>(nn.ny()));
        nrm.push_back(static_cast<float>(nn.nz()));
    }
    std::vector<std::uint32_t> nbr;
    std::size_t k = 0;
    if constexpr (detail::is_gpu_knn_map<knn_type>::value)
    {
        knn_result_t const r = knn_map.index->knn_batch(xyz, knn_map.k, knn_map.eps);
        k                    = r.k;
        nbr.assign(n * k, PCPX_NO_NEIGHBOUR);
        auto const& elements = knn_map.index->elements();
        for (std::size_t i = 0; i < n; ++i)
            for (std::size_t j = 0; j < r.counts[i]; ++j)
                nbr[i * k + j] =
                    static_cast<std::uint32_t>(index_map(elements[r.indices[i * k + j]]));
    }
    else
    {
        std::vector<std::vector<std::uint32_t>> rows(n);
        std::size_t i = 0;
        for (auto it = begin; it != end; ++it, ++i)
        {
            auto const neighbours = knn_map(*it);
            for (auto const& e : neighbours)
                rows[i].push_back(static_cast<std::uint32_t>(index_map(e)));
            k = std::max(k, rows[i].size());
        }
        nbr.assign(n * k, PCPX_NO_NEIGHBOUR);
        for (i = 0; i < n; ++i)
            std::copy(rows[i].begin(), rows[i].end(), nbr.begin() + static_cast<std::ptrdiff_t>(i * k));
    }
    std::vector<float> const before = nrm;
    detail::check(pcpx_orient_normals_graph(xyz.data(), n, 12, nbr.data(),
                                            static_cast<std::uint32_t>(k), edge_order, -1,
                                            nrm.data(), nullptr, nullptr),
                  "pcpx_orient_normals_graph");
    std::size_t i = 0;
    for (auto it = begin; it != end; ++it, ++i)
        if (nrm[3 * i] != before[3 * i] || nrm[3 * i + 1] != before[3 * i + 1] ||
            nrm[3 * i + 2] != before[3 * i + 2])
            op(*it, normal_type{static_cast<scalar_type>(nrm[3 * i]),
                                static_cast<scalar_type>(nrm[3 * i + 1]),
                                static_cast<scalar_type>(nrm[3 * i + 2])});
}

// algorithm/average_distance_to_neighbors.hpp:39-73 for the index's own elements, in their
// original order (bit-exact fp32 per point), and :95-113 for their mean.
template <class Index, class ScalarType = float>
std::vector<ScalarType> average_distances_to_neighbors(Index const& index, std::size_t k,
                                                       double eps = 1e-5, double* mean = nullptr)
{
    std::vector<float> per(index.elements().size());
    double mu = 0.0;
    detail::check(pcpx_mean_knn_distance(index.handle(), static_cast<std::uint32_t>(k), eps,
                                         per.data(), &mu),
                  "pcpx_mean_knn_distance");
    if (mean)
        *mean = mu;
    return std::vector<ScalarType>(per.begin(), per.end());
}
template <class Index, class ScalarType = float>
ScalarType average_distance_to_neighbors(Index const& index, std::size_t k, double eps = 1e-5)
{
    double mu = 0.0;
    detail::check(pcpx_mean_knn_distance(index.handle(), static_cast<std::uint32_t>(k), eps,
                                         nullptr, &mu),
                  "pcpx_mean_knn_distance");
    return static_cast<ScalarType>(mu);
}

// The density outlier filter of examples/filter_point_cloud_noise_by_density.cpp:81-91 as a
// library call: keep element i iff the ball of `radius` around it holds >= threshold elements
// (itself included).  Returns the kept elements in their original relative order (what
// std::remove_if + erase leaves); `mask` optionally receives the per-element decision.
template <class Index>
std::vector<typename Index::element_type> filter_by_density(Index const& index, float radius,
                                                            std::size_t density_threshold,
                                                            std::vector<std::uint8_t>* mask = nullptr)
{
    std::size_t const n = index.elements().size();
    std::vector<std::uint8_t> keep(n);
    std::size_t kept = 0;
    detail::check(pcpx_density_filter(index.handle(), radius,
                                      static_cast<std::uint32_t>(density_threshold), keep.data(),
                                      nullptr, &kept),
                  "pcpx_density_filter");
    std::vector<typename Index::element_type> out;
    out.reserve(kept);
    for (std::size_t i = 0; i < n; ++i)
        if (keep[i])
            out.push_back(index.elements()[i]);
    if (mask)
        *mask = std::move(keep);
    return out;
}

// pcpx extension (the reference has no clustering): DBSCAN of the indexed elements over the
// exact ball of `radius` (pcpx_cluster_by_density).  Returns one label per element, in element
// order: the cluster, numbered 0 .. C-1 in ascending order of each cluster's smallest core
// element index, or PCPX_NOISE.  An element is core iff filter_by_density(radius, min_points)
// keeps it; with min_points <= 1 this is Euclidean clustering.  `n_clusters` receives C.
template <class Index>
std::vector<std::uint32_t> cluster_by_density(Index const& index, float radius,
                                              std::size_t min_points,
                                              std::size_t* n_clusters = nullptr)
{
    std::vector<std::uint32_t> labels(index.elements().size());
    std::uint64_t c = 0;
    // (a ball holds fewer than 2^32 elements: every larger threshold means no element is core)
    auto const threshold = static_cast<std::uint32_t>(
        std::min<std::size_t>(min_points, std::numeric_limits<std::uint32_t>::max()));
    detail::check(pcpx_cluster_by_density(index.handle(), radius, threshold, labels.data(), &c),
                  "pcpx_cluster_by_density");
    if (n_clusters)
        *n_clusters = static_cast<std::size_t>(c);
    return labels;
}

// pcpx extension (the reference has no registration): rigid ICP of a source range against the
// indexed target (pcpx_icp).  `target_normals`: one normal per target element, in element order
// (what estimate_normals over the index writes); point-to-plane needs them, point-to-point ignores
// them.  Coordinates of other scalar types are rounded to fp32.  The parameter and result types
// are pcp::icp::params_t and pcp::icp::result_t.
} // namespace algorithm
namespace icp {
struct params_t
{
    std::uint32_t metric         = PCPX_ICP_POINT_TO_PLANE; // or PCPX_ICP_POINT_TO_POINT
    std::uint32_t max_iterations = 30;
    float max_distance           = 0.f; // correspondence bound: required, finite, > 0
    double rotation_tolerance    = 0.0; // 0 = 1e-6 rad
    double translation_tolerance = 0.0; // 0 = 1e-6 x the diagonal of the target's root voxel
    std::array<double, 16> init{1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
};
struct result_t
{
    std::array<double, 16> transform; // row-major 4 x 4: source -> target
    std::uint32_t iterations;
    std::uint32_t stop_reason; // PCPX_ICP_CONVERGED / _MAX_ITERATIONS / _TOO_FEW
    std::uint64_t n_correspondences;
    double fitness;
    double rmse;
};
} // namespace icp
namespace algorithm {

template <class Index, class NormalRange, class ForwardIter, class PointMap>
icp::result_t icp(Index const& target_index, NormalRange const& target_normals,
                  ForwardIter source_begin, ForwardIter source_end, PointMap const& point_map,
                  icp::params_t const& params)
{
    std::vector<float> src;
    for (auto it = source_begin; it != source_end; ++it)
    {
        auto const& p = point_map(*it);
        src.push_back(static_cast<float>(p.x()));
        src.push_back(static_cast<float>(p.y()));
        src.push_back(static_cast<float>(p.z()));
    }
    std::vector<float> nrm;
    if (params.metric == PCPX_ICP_POINT_TO_PLANE)
        for (auto const& n : target_normals)
        {
            nrm.push_back(static_cast<float>(n.x()));
            nrm.push_back(static_cast<float>(n.y()));
            nrm.push_back(static_cast<float>(n.z()));
        }
    if (params.metric == PCPX_ICP_POINT_TO_PLANE && nrm.size() != 3 * target_index.elements().size())
        throw std::invalid_argument("icp: point-to-plane needs one normal per target element");
    pcpx_icp_params prm{};
    prm.metric                = params.metric;
    prm.max_iterations        = params.max_iterations;
    prm.max_distance          = params.max_distance;
    prm.rotation_tolerance    = params.rotation_tolerance;
    prm.translation_tolerance = params.translation_tolerance;
    icp::result_t out{};
    pcpx_icp_result res{};
    detail::check(pcpx_icp(target_index.handle(), nrm.empty() ? nullptr : nrm.data(), 12,
                           src.data(), src.size() / 3, 12, &prm, params.init.data(),
                           out.transform.data(), &res, nullptr),
                  "pcpx_icp");
    out.iterations        = res.iterations;
    out.stop_reason       = res.stop_reason;
    out.n_correspondences = res.n_correspondences;
    out.fitness           = res.fitness;
    out.rmse              = res.rmse;
    return out;
}

// ---- radius-search callers (SURVEY.md 8f rank 3) ---------------------------------------------
namespace bilateral {
// algorithm/bilateral_filter.hpp:28-33
struct params_t
{
    double sigmaf = 1.;  ///< standard deviation of the spatial weight f (support = 2 sigmaf)
    double sigmag = 0.1; ///< standard deviation of the influence weight g
    std::size_t K = 1u;  ///< iterations
};
namespace detail {
template <class Iter, class PointMap, class NormalMap>
void flatten(Iter begin, Iter end, PointMap const& point_map, NormalMap const& normal_map,
             std::vector<float>& xyz, std::vector<float>& nrm)
{
    for (auto it = begin; it != end; ++it)
    {
        pcp::detail::push_xyz(xyz, point_map(*it));
        auto const n = normal_map(*it);
        nrm.push_back(static_cast<float>(n.nx()));
        nrm.push_back(static_cast<float>(n.ny()));
        nrm.push_back(static_cast<float>(n.nz()));
    }
}
} // namespace detail
} // namespace bilateral

// Drop-in for algorithm/bilateral_filter.hpp:301-421: same signature, the K iterations
// (index rebuild + one kernel each) run on the GPU; *out_begin++ receives points constructible
// from (x, y, z).
template <class RandomAccessIter, class OutputIter, class PointMap, class NormalMap>
OutputIter bilateral_filter_points(RandomAccessIter begin, RandomAccessIter end,
                                   OutputIter out_begin, PointMap const& point_map,
                                   NormalMap const& normal_map, bilateral::params_t const& params)
{
    using point_type  = std::decay_t<decltype(point_map(*begin))>;
    using scalar_type = typename point_type::coordinate_type;
    std::vector<float> xyz, nrm;
    bilateral::detail::flatten(begin, end, point_map, normal_map, xyz, nrm);
    std::size_t const n = xyz.size() / 3;
    std::vector<float> out(xyz.size());
    detail::check(pcpx_bilateral_filter_points(xyz.data(), n, 12, nrm.data(), 12, params.sigmaf,
                                               params.sigmag,
                                               static_cast<std::uint32_t>(params.K), -1,
                                               out.data(), nullptr),
                  "pcpx_bilateral_filter_points");
    for (std::size_t i = 0; i < n; ++i)
        *out_begin++ = point_type{static_cast<scalar_type>(out[3 * i]),
                                  static_cast<scalar_type>(out[3 * i + 1]),
                                  static_cast<scalar_type>(out[3 * i + 2])};
    return out_begin;
}

// Drop-in for algorithm/bilateral_filter.hpp:452-575.
template <class RandomAccessIter, class OutputIter, class PointMap, class NormalMap>
OutputIter bilateral_filter_normals(RandomAccessIter begin, RandomAccessIter end,
                                    OutputIter out_begin, PointMap const& point_map,
                                    NormalMap const& normal_map, bilateral::params_t const& params)
{
    using normal_type = std::decay_t<decltype(normal_map(*begin))>;
    using scalar_type = typename normal_type::component_type;
    std::vector<float> xyz, nrm;
    bilateral::detail::flatten(begin, end, point_map, normal_map, xyz, nrm);
    std::size_t const n = xyz.size() / 3;
    std::vector<float> out(xyz.size());
    detail::check(pcpx_bilateral_filter_normals(xyz.data(), n, 12, nrm.data(), 12, params.sigmaf,
                                                params.sigmag,
                                                static_cast<std::uint32_t>(params.K), -1,
                                                out.data(), nullptr),
                  "pcpx_bilateral_filter_normals");
    for (std::size_t i = 0; i < n; ++i)
        *out_begin++ = normal_type{static_cast<scalar_type>(out[3 * i]),
                                   static_cast<scalar_type>(out[3 * i + 1]),
                                   static_cast<scalar_type>(out[3 * i + 2])};
    return out_begin;
}

namespace wlop {
// algorithm/wlop.hpp:233-241, plus the seed of the start set (the reference draws it from
// std::random_device, :346-358, which no caller can reproduce)
struct params_t
{
    std::size_t I = 0u;   ///< size of the resampled cloud
    double mu     = 0.45; ///< repulsion coefficient, in [0, 0.5]
    double h      = 0.;   ///< support radius
    std::size_t k = 10u;  ///< solver iterations
    bool uniform  = true; ///< WLOP density weights; false = plain LOP
    std::uint32_t seed = 5489u; ///< std::mt19937 seed of the start set (pcpx extension)
};

// Drop-in for algorithm/wlop.hpp:278-438.  `Point` = the type written to out_begin.
template <class Point = pcp::point_t, class RandomAccessIter, class OutputIter, class PointMap>
OutputIter wlop(RandomAccessIter begin, RandomAccessIter end, OutputIter out_begin,
                PointMap point_map, params_t const& params)
{
    using scalar_type = typename Point::coordinate_type;
    std::vector<float> xyz;
    for (auto it = begin; it != end; ++it)
        pcp::detail::push_xyz(xyz, point_map(*it));
    std::vector<float> out(3 * params.I);
    detail::check(pcpx_wlop(xyz.data(), xyz.size() / 3, 12, nullptr, params.I, params.mu, params.h,
                            static_cast<std::uint32_t>(params.k), params.uniform ? 1 : 0,
                            params.seed, -1, out.data(), nullptr),
                  "pcpx_wlop");
    for (std::size_t i = 0; i < params.I; ++i)
        *out_begin++ = Point{static_cast<scalar_type>(out[3 * i]),
                             static_cast<scalar_type>(out[3 * i + 1]),
                             static_cast<scalar_type>(out[3 * i + 2])};
    return out_begin;
}
} // namespace wlop

} // namespace algorithm
} // namespace pcp

#endif // PCPX_PCP_HPP
