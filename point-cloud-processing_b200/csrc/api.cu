// The C ABI of libpcpx.so (include/pcpx.h): argument checking, host <-> device staging,
// timing.  All compute is in index.cu / query_body.inc; there is no CPU path.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <thread>
#include <vector>

#include "api_util.hpp"

using namespace pcpx;

// kernels a kNN-shaped call launches: main + retry for the register-list sizes; the heap
// kernel alone (rows) or followed by the inverse-order and row-reduction kernels (normals, means)
static uint32_t knn_shaped_launches(const pcpx_index& ix, uint32_t k, bool rows_only)
{
    return k <= kMaxK ? ix.query_launches.load() : (rows_only ? 1u : 3u);
}

// ---- several devices behind one handle (pcpx_index_params.devices) --------------------------
// The primary index plus one replica per further device.  A sharded call runs `fn(part_index,
// part)` for every device at once — the caller's thread takes the primary, one host thread per
// replica — and returns when all have finished (each launcher synchronises its own stream).
// The first error of any device is re-thrown.
template <class F>
static void on_every_device(pcpx_index& ix, F&& fn)
{
    size_t const nrep = ix.replicas.size();
    std::vector<std::thread> threads;
    std::vector<std::unique_ptr<Error>> errors(nrep);
    for (size_t r = 0; r < nrep; ++r)
        threads.emplace_back([&, r] {
            try
            {
                pcpx_index& rep = *ix.replicas[r];
                ScopedDevice guard(rep.device);
                CallStream call(rep);
                fn(rep, (uint32_t)r + 1u);
            }
            catch (Error const& e)
            {
                errors[r].reset(new Error(e));
            }
            catch (std::exception const& e)
            {
                errors[r].reset(new Error{PCPX_ERR_CUDA, e.what()});
            }
        });
    std::unique_ptr<Error> mine;
    try
    {
        fn(ix, 0u);
    }
    catch (Error const& e)
    {
        mine.reset(new Error(e));
    }
    for (auto& t : threads)
        t.join();
    if (mine)
        throw *mine;
    for (auto& e : errors)
        if (e)
            throw *e;
}

// a kNN-shaped call is spread over the replicas when there are any and k fits the register lists
static bool sharded(const pcpx_index& ix, uint32_t k) { return !ix.replicas.empty() && k <= kMaxK; }

// kernel time of a sharded call: the slowest device (each measures its own stream)
struct PartTimer
{
    std::vector<float> ms;
    explicit PartTimer(const pcpx_index& ix) : ms(ix.replicas.size() + 1, 0.f) {}
    template <class F>
    void run(pcpx_index& part_ix, uint32_t part, F&& launch)
    {
        Event a, b;
        a.record(part_ix.qstream());
        launch();
        b.record(part_ix.qstream());
        PCPX_CUDA(cudaStreamSynchronize(part_ix.qstream()));
        ms[part] = elapsed_ms(a, b);
    }
    float slowest() const { return *std::max_element(ms.begin(), ms.end()); }
};

// One output array of a sharded call.  The primary writes its rows in place; a replica fills a
// local buffer indexed by SORTED query position (QueryBatch::by_position) which the primary then
// reads in order over NVLink and scatters to the rows (launch_gather_rows) — rows written one by
// one across NVLink cost several times the kernel (4 devices: 2.2 ms per call against 0.6 ms
// of kernel).
template <typename T>
struct ShardedOut
{
    T* primary = nullptr;
    size_t rows = 0;
    uint32_t width = 0;
    std::vector<DevBuf<T>> local; // one per replica, on the replica's device

    ShardedOut(T* dst, size_t n_rows, uint32_t w, size_t n_replicas)
        : primary(dst), rows(n_rows), width(w), local(n_replicas)
    {
    }
    // the pointer the kernels of `part` write through (called on the part's own thread/device)
    T* target(uint32_t part)
    {
        if (!primary)
            return nullptr;
        if (part == 0)
            return primary;
        local[part - 1].alloc(std::max<size_t>(rows * width, 1));
        return local[part - 1].get();
    }
    void gather(const pcpx_index& ix, const QueryBatch& qb, const std::vector<ShardInfo>& shards)
    {
        if (!primary)
            return;
        for (size_t r = 0; r < local.size(); ++r)
            launch_gather_rows(ix, qb, shards[r + 1],
                               reinterpret_cast<const uint32_t*>(local[r].get()),
                               reinterpret_cast<uint32_t*>(primary), width);
    }
};

static void validate_devices(const pcpx_index_params& prm)
{
    if (prm.shard_mode != PCPX_SHARD_REPLICATED)
        fail(PCPX_ERR_UNSUPPORTED,
             "shard_mode %u: inside the library an index is replicated on its devices; slabs are "
             "one process per GPU (sharding.py, pcpx_extract_bands)", prm.shard_mode);
    if (prm.n_devices == 0)
        return;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        fail(PCPX_ERR_NO_DEVICE, "no CUDA device: libpcpx has no CPU path");
    if (prm.n_devices > 8)
        fail(PCPX_ERR_INVALID_ARG, "n_devices = %u (at most 8)", prm.n_devices);
    for (uint32_t i = 0; i < prm.n_devices; ++i)
    {
        if (prm.devices[i] < 0 || prm.devices[i] >= ndev)
            fail(PCPX_ERR_INVALID_ARG, "devices[%u] = %d out of range (%d devices)", i,
                 prm.devices[i], ndev);
        // (PCPX_TEST_SAME_DEVICE_REPLICAS=1: a device may be listed more than once, so that a
        // one-GPU box can exercise the sharded code path — tests only, it buys no speed)
        bool const allow_dup = std::getenv("PCPX_TEST_SAME_DEVICE_REPLICAS") != nullptr;
        for (uint32_t j = 0; j < i && !allow_dup; ++j)
            if (prm.devices[j] == prm.devices[i])
                fail(PCPX_ERR_INVALID_ARG, "device %d listed twice", prm.devices[i]);
    }
}

static void build_replicas(pcpx_index& ix, const float* xyz, size_t n, size_t stride_bytes,
                           const pcpx_index_params& prm)
{
    // every replica writes its rows into the primary's buffers (and reads its staged queries)
    for (uint32_t i = 1; i < prm.n_devices; ++i)
    {
        if (prm.devices[i] == ix.device)
            continue;
        int can = 0;
        PCPX_CUDA(cudaDeviceCanAccessPeer(&can, prm.devices[i], ix.device));
        if (!can)
            fail(PCPX_ERR_UNSUPPORTED, "device %d cannot access device %d's memory (no peer access)",
                 prm.devices[i], ix.device);
        // both ways: a replica reads the primary's staged queries, the primary reads the
        // replica's answers
        for (int dir = 0; dir < 2; ++dir)
        {
            int const from = dir ? ix.device : prm.devices[i], to = dir ? prm.devices[i] : ix.device;
            PCPX_CUDA(cudaDeviceCanAccessPeer(&can, from, to));
            if (!can)
                fail(PCPX_ERR_UNSUPPORTED, "device %d cannot access device %d's memory", from, to);
            ScopedDevice guard(from);
            cudaError_t const e = cudaDeviceEnablePeerAccess(to, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                fail(PCPX_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", from, to,
                     cudaGetErrorString(e));
            cudaGetLastError();
        }
    }
    size_t const nrep = prm.n_devices - 1;
    ix.replicas.assign(nrep, nullptr);
    std::vector<std::thread> threads;
    std::vector<std::unique_ptr<Error>> errors(nrep);
    for (size_t r = 0; r < nrep; ++r)
        threads.emplace_back([&, r] {
            try
            {
                pcpx_index_params p = prm;
                p.device            = prm.devices[r + 1];
                p.n_devices         = 0;
                ScopedDevice guard(p.device);
                if (!is_device_pointer(xyz))
                {
                    // host memory: the replica's build stages it on its own stream
                    ix.replicas[r] = build_index(xyz, n, stride_bytes, &p);
                    return;
                }
                // device memory (the primary's, usually): one packed copy over NVLink first, so
                // that the build's gathers stay local.  Stream-ordered: a synchronous cudaMemcpy
                // would not order the DMA against the build's non-blocking stream.
                DevBuf<float> local(std::max<size_t>(3 * n, 1));
                Stream copy_stream;
                if (n && (stride_bytes == 0 || stride_bytes == 12)) // packed rows: one DMA
                    PCPX_CUDA(cudaMemcpyAsync(local.get(), xyz, 12 * n, cudaMemcpyDefault,
                                              copy_stream.s));
                else if (n)
                    PCPX_CUDA(cudaMemcpy2DAsync(local.get(), 12, xyz, stride_bytes, 12, n,
                                                cudaMemcpyDefault, copy_stream.s));
                PCPX_CUDA(cudaStreamSynchronize(copy_stream.s));
                ix.replicas[r] = build_index(local.get(), n, 12, &p);
            }
            catch (Error const& e)
            {
                errors[r].reset(new Error(e));
            }
        });
    for (auto& t : threads)
        t.join();
    for (auto& e : errors)
        if (e)
            throw *e;
}

extern "C" {

int pcpx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess)
    {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char* pcpx_last_error(void) { return last_error_storage().c_str(); }

int pcpx_index_create(const float* xyz, size_t n, size_t stride_bytes,
                      const pcpx_index_params* params, pcpx_index** out_index)
{
    return guarded([&] {
        if (!out_index)
            fail(PCPX_ERR_INVALID_ARG, "out_index is NULL");
        *out_index = nullptr;
        pcpx_index_params prm{};
        if (params)
            prm = *params;
        validate_devices(prm);
        if (prm.n_devices >= 1)
            prm.device = prm.devices[0];
        std::unique_ptr<pcpx_index> ix(build_index(xyz, n, stride_bytes, &prm));
        if (prm.n_devices >= 2)
        {
            // replicas are built while nothing else uses the primary; a failure frees everything
            try
            {
                build_replicas(*ix, xyz, n, stride_bytes, prm);
            }
            catch (...)
            {
                ScopedDevice guard(ix->device);
                ix.reset();
                throw;
            }
        }
        *out_index = ix.release();
    });
}

void pcpx_index_destroy(pcpx_index* index)
{
    if (!index)
        return;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(index->device);
    delete index;
    if (prev >= 0)
        cudaSetDevice(prev);
}

int pcpx_index_info_get(const pcpx_index* index, pcpx_index_info* out)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out)
            fail(PCPX_ERR_INVALID_ARG, "out_info is NULL");
        std::memset(out, 0, sizeof *out);
        out->n_input   = ix.n_input;
        out->n_indexed = ix.n_indexed;
        for (int a = 0; a < 3; ++a)
            out->bbox_min[a] = ix.bbox_min[a], out->bbox_max[a] = ix.bbox_max[a];
        out->code_bits    = ix.code_bits;
        out->finest_level = (uint32_t)ix.grid.lfine;
        out->n_cells      = ix.n_cells;
        out->device_bytes = ix.device_bytes();
        out->device       = ix.device;
        out->build_ms     = ix.timings.build_ms;
        out->n_devices    = (uint32_t)ix.replicas.size() + 1u;
        for (pcpx_index const* r : ix.replicas)
            out->build_ms = std::max(out->build_ms, r->timings.build_ms);
    });
}

int pcpx_index_bbox(const pcpx_index* index, float out_min[3], float out_max[3])
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out_min || !out_max)
            fail(PCPX_ERR_INVALID_ARG, "out_min / out_max is NULL");
        for (int a = 0; a < 3; ++a)
            out_min[a] = ix.bbox_min[a], out_max[a] = ix.bbox_max[a];
    });
}

int pcpx_knn(const pcpx_index* index, const float* queries, size_t nq, size_t query_stride_bytes,
             uint32_t k, double eps, uint32_t* out_idx, float* out_d2, uint32_t* out_count)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (k == 0 || nq == 0) // octree/linked_octree_node.hpp:464: k == 0 -> {}
        {
            if (!queries && nq != ix.n_input && nq != 0)
                fail(PCPX_ERR_INVALID_ARG, "nq must equal the indexed cloud's size");
            return;
        }
        if (!out_idx)
            fail(PCPX_ERR_INVALID_ARG, "out_idx is NULL");
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        Batch batch;
        batch.prepare(ix, queries, nq, query_stride_bytes);
        OutBuf<uint32_t> idx, cnt;
        OutBuf<float> d2;
        idx.prepare(out_idx, nq * (size_t)k);
        d2.prepare(out_d2, nq * (size_t)k);
        cnt.prepare(out_count, nq);
        DevBuf<uint32_t> retries(1);
        PCPX_CUDA(cudaMemsetAsync(retries.get(), 0, 4, ix.qstream()));
        PartTimer parts(ix);
        timer.kernel_begin();
        if (sharded(ix, k))
        {
            PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // staged queries are in place
            size_t const nrep = ix.replicas.size();
            std::vector<ShardInfo> shards(nrep + 1);
            ShardedOut<uint32_t> s_idx(idx.d, nq, k, nrep), s_cnt(cnt.d, nq, 1, nrep);
            ShardedOut<float> s_d2(d2.d, nq, k, nrep);
            on_every_device(ix, [&](pcpx_index& dev_ix, uint32_t part) {
                QueryBatch qb = batch.qb;
                qb.part = part, qb.parts = (uint32_t)nrep + 1u;
                qb.by_position = part != 0, qb.shard_info = &shards[part];
                uint32_t* p_idx = s_idx.target(part);
                float* p_d2     = s_d2.target(part);
                uint32_t* p_cnt = s_cnt.target(part);
                parts.run(dev_ix, part, [&] {
                    launch_knn(dev_ix, qb, k, (float)eps, p_idx, p_d2, p_cnt,
                               part == 0 ? retries.get() : nullptr);
                });
            });
            s_idx.gather(ix, batch.qb, shards), s_d2.gather(ix, batch.qb, shards);
            s_cnt.gather(ix, batch.qb, shards);
            PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // before the replicas' buffers go
        }
        else
            launch_knn(ix, batch.qb, k, (float)eps, idx.d, d2.d, cnt.d, retries.get());
        timer.kernel_end();
        ix.timings.kernel_launches = knn_shaped_launches(ix, k, true);
        idx.finish(ix.qstream()), d2.finish(ix.qstream()), cnt.finish(ix.qstream());
        uint32_t h_retries = 0;
        timer.done();
        read_back(ix.qstream(), &h_retries, retries.get(), 4);
        if (sharded(ix, k))
            ix.timings.kernel_ms = parts.slowest();
        ix.timings.retry_queries = h_retries;
    });
}

int pcpx_radius_count(const pcpx_index* index, const float* queries, size_t nq,
                      size_t query_stride_bytes, const float* radii, float radius,
                      uint32_t* out_count)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (nq == 0)
            return;
        if (!out_count)
            fail(PCPX_ERR_INVALID_ARG, "out_count is NULL");
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        Batch batch;
        batch.prepare(ix, queries, nq, query_stride_bytes);
        InBuf rad;
        rad.stage(radii, nq, 4, 1, ix.qstream());
        OutBuf<uint32_t> cnt;
        cnt.prepare(out_count, nq);
        timer.kernel_begin();
        launch_radius_count(ix, batch.qb, rad.d, radius, cnt.d);
        timer.kernel_end();
        ix.timings.kernel_launches = 1;
        cnt.finish(ix.qstream());
        timer.done();
    });
}

int pcpx_radius_search(const pcpx_index* index, const float* queries, size_t nq,
                       size_t query_stride_bytes, const float* radii, float radius,
                       uint64_t* out_offsets, uint32_t** out_idx, int out_idx_device)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out_offsets || !out_idx)
            fail(PCPX_ERR_INVALID_ARG, "out_offsets / out_idx is NULL");
        *out_idx = nullptr;
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        Batch batch;
        batch.prepare(ix, queries, nq, query_stride_bytes);
        InBuf rad;
        rad.stage(radii, nq, 4, 1, ix.qstream());
        DevBuf<uint32_t> cnt(std::max<size_t>(nq, 1));
        OutBuf<uint64_t> off;
        off.prepare(out_offsets, nq + 1);
        timer.kernel_begin();
        launch_radius_count(ix, batch.qb, rad.d, radius, cnt.get());
        launch_exclusive_scan_u32(ix, cnt.get(), (uint32_t)nq, off.d);
        uint64_t total = 0;
        PCPX_CUDA(cudaMemcpyAsync(&total, off.d + nq, 8, cudaMemcpyDeviceToHost, ix.qstream()));
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
        DevBuf<uint32_t> lists(std::max<uint64_t>(total, 1));
        launch_radius_fill(ix, batch.qb, rad.d, radius, off.d, lists.get());
        if (out_idx_device & PCPX_RADIUS_SORTED)
            launch_sort_lists(ix, off.d, (uint32_t)nq, lists.get());
        timer.kernel_end();
        ix.timings.kernel_launches = (out_idx_device & PCPX_RADIUS_SORTED) ? 6 : 5;
        off.finish(ix.qstream());
        if (out_idx_device & PCPX_RADIUS_DEVICE)
        {
            timer.done();
            *out_idx = lists.detach();
        }
        else
        {
            uint32_t* host = (uint32_t*)std::malloc(std::max<uint64_t>(total, 1) * 4);
            if (!host)
                fail(PCPX_ERR_OUT_OF_MEMORY, "host allocation of %llu indices failed",
                     (unsigned long long)total);
            cudaError_t e = cudaMemcpyAsync(host, lists.get(), total * 4, cudaMemcpyDeviceToHost,
                                            ix.qstream());
            if (e == cudaSuccess)
                e = cudaStreamSynchronize(ix.qstream());
            if (e != cudaSuccess)
            {
                std::free(host);
                fail(PCPX_ERR_CUDA, "copying radius lists back failed: %s", cudaGetErrorString(e));
            }
            timer.done();
            *out_idx = host;
        }
    });
}

// the boxes of a box call, staged; bb = the index's bounding box (its voxel grid when it has one),
// which holds every indexed point
static BoxBatch box_batch(pcpx_index& ix, const float* boxes, size_t nb, size_t stride_bytes,
                          InBuf& in)
{
    if (nb >= 0xFFFFFFFFull)
        fail(PCPX_ERR_UNSUPPORTED, "more than 2^32 - 2 boxes in one call");
    if (nb && !boxes)
        fail(PCPX_ERR_INVALID_ARG, "boxes is NULL");
    in.stage(boxes, nb, stride_bytes, 6, ix.qstream());
    BoxBatch bx{in.d, in.stride_f, (uint32_t)nb, {}};
    for (int a = 0; a < 3; ++a)
        bx.bb[a] = ix.bbox_min[a], bx.bb[3 + a] = ix.bbox_max[a];
    return bx;
}

static void check_box_stride(size_t stride_bytes)
{
    if (stride_bytes < 24 || stride_bytes % 4)
        fail(PCPX_ERR_INVALID_ARG, "box_stride_bytes must be a multiple of 4 and >= 24");
}

int pcpx_box_count(const pcpx_index* index, const float* boxes, size_t nb,
                   size_t box_stride_bytes, uint32_t* out_count)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out_count)
            fail(PCPX_ERR_INVALID_ARG, "out_count is NULL");
        check_box_stride(box_stride_bytes);
        if (nb == 0)
            return;
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        InBuf in;
        BoxBatch const bx = box_batch(ix, boxes, nb, box_stride_bytes, in);
        OutBuf<uint32_t> cnt;
        cnt.prepare(out_count, nb);
        timer.kernel_begin();
        launch_box_count(ix, bx, cnt.d, nullptr);
        timer.kernel_end();
        ix.timings.kernel_launches = 1;
        cnt.finish(ix.qstream());
        timer.done();
    });
}

int pcpx_box_search(const pcpx_index* index, const float* boxes, size_t nb,
                    size_t box_stride_bytes, uint64_t* out_offsets, uint32_t** out_idx, int flags)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out_offsets || !out_idx)
            fail(PCPX_ERR_INVALID_ARG, "out_offsets / out_idx is NULL");
        *out_idx = nullptr;
        check_box_stride(box_stride_bytes);
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        InBuf in;
        BoxBatch const bx = box_batch(ix, boxes, nb, box_stride_bytes, in);
        DevBuf<uint32_t> cnt(std::max<size_t>(nb, 1));
        DevBuf<uint32_t> max_cnt(1);
        PCPX_CUDA(cudaMemsetAsync(max_cnt.get(), 0, 4, ix.qstream()));
        OutBuf<uint64_t> off;
        off.prepare(out_offsets, nb + 1);
        timer.kernel_begin();
        launch_box_count(ix, bx, cnt.get(), max_cnt.get());
        launch_exclusive_scan_u32(ix, cnt.get(), (uint32_t)nb, off.d);
        uint64_t total = 0;
        uint32_t longest = 0;
        PCPX_CUDA(cudaMemcpyAsync(&total, off.d + nb, 8, cudaMemcpyDeviceToHost, ix.qstream()));
        PCPX_CUDA(cudaMemcpyAsync(&longest, max_cnt.get(), 4, cudaMemcpyDeviceToHost, ix.qstream()));
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
        DevBuf<uint32_t> lists(std::max<uint64_t>(total, 1));
        // count + the scan's three kernels + fill and copy + the sort's
        uint32_t launches = nb ? 4 : 0;
        launches += launch_box_fill(ix, bx, off.d, total, lists.get());
        if (flags & PCPX_RADIUS_SORTED)
            launches += launch_box_sort(ix, off.d, (uint32_t)nb, total, longest, lists.get());
        timer.kernel_end();
        ix.timings.kernel_launches = launches;
        off.finish(ix.qstream());
        if (flags & PCPX_RADIUS_DEVICE)
        {
            timer.done();
            *out_idx = lists.detach();
        }
        else
        {
            uint32_t* host = (uint32_t*)std::malloc(std::max<uint64_t>(total, 1) * 4);
            if (!host)
                fail(PCPX_ERR_OUT_OF_MEMORY, "host allocation of %llu indices failed",
                     (unsigned long long)total);
            cudaError_t e = cudaMemcpyAsync(host, lists.get(), total * 4, cudaMemcpyDeviceToHost,
                                            ix.qstream());
            if (e == cudaSuccess)
                e = cudaStreamSynchronize(ix.qstream());
            if (e != cudaSuccess)
            {
                std::free(host);
                fail(PCPX_ERR_CUDA, "copying box lists back failed: %s", cudaGetErrorString(e));
            }
            timer.done();
            *out_idx = host;
        }
    });
}

void pcpx_free(void* p, int is_device)
{
    if (!p)
        return;
    if (is_device)
        cudaFree(p);
    else
        std::free(p);
}

static void normals_impl(const pcpx_index* index, const float* queries, size_t nq,
                         size_t query_stride_bytes, uint32_t k, double eps, float* out_points,
                         float* out_normals)
{
    pcpx_index& ix = checked(index);
    if (nq == 0)
        return;
    if (!out_normals)
        fail(PCPX_ERR_INVALID_ARG, "out_normals is NULL");
    ScopedDevice guard(ix.device);
    CallStream call(ix); // own stream: calls on one index may run concurrently
    CallTimer timer(ix);
    Batch batch;
    batch.prepare(ix, queries, nq, query_stride_bytes);
    OutBuf<float> nrm, ctr;
    nrm.prepare(out_normals, nq * 3);
    ctr.prepare(out_points, nq * 3);
    DevBuf<uint32_t> ties(1);
    PCPX_CUDA(cudaMemsetAsync(ties.get(), 0, 4, ix.qstream()));
    PartTimer parts(ix);
    timer.kernel_begin();
    if (sharded(ix, k))
    {
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // staged queries are in place
        size_t const nrep = ix.replicas.size();
        std::vector<ShardInfo> shards(nrep + 1);
        ShardedOut<float> s_nrm(nrm.d, nq, 3, nrep), s_ctr(ctr.d, nq, 3, nrep);
        on_every_device(ix, [&](pcpx_index& dev_ix, uint32_t part) {
            QueryBatch qb = batch.qb;
            qb.part = part, qb.parts = (uint32_t)nrep + 1u;
            qb.by_position = part != 0, qb.shard_info = &shards[part];
            float* p_ctr = s_ctr.target(part);
            float* p_nrm = s_nrm.target(part);
            parts.run(dev_ix, part, [&] {
                launch_normals(dev_ix, qb, k, (float)eps, p_ctr, p_nrm,
                               part == 0 ? ties.get() : nullptr);
            });
        });
        s_nrm.gather(ix, batch.qb, shards), s_ctr.gather(ix, batch.qb, shards);
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // before the replicas' buffers go
    }
    else
        launch_normals(ix, batch.qb, k, (float)eps, ctr.d, nrm.d, ties.get());
    timer.kernel_end();
    ix.timings.kernel_launches = knn_shaped_launches(ix, k, false);
    nrm.finish(ix.qstream()), ctr.finish(ix.qstream());
    uint32_t h_ties = 0;
    timer.done();
    read_back(ix.qstream(), &h_ties, ties.get(), 4);
    if (sharded(ix, k))
        ix.timings.kernel_ms = parts.slowest();
    ix.timings.retry_queries = h_ties;
}

int pcpx_estimate_normals(const pcpx_index* index, const float* queries, size_t nq,
                          size_t query_stride_bytes, uint32_t k, double eps, float* out_normals)
{
    return guarded(
        [&] { normals_impl(index, queries, nq, query_stride_bytes, k, eps, nullptr, out_normals); });
}

int pcpx_estimate_tangent_planes(const pcpx_index* index, const float* queries, size_t nq,
                                 size_t query_stride_bytes, uint32_t k, double eps,
                                 float* out_points, float* out_normals)
{
    return guarded([&] {
        if (nq && !out_points)
            fail(PCPX_ERR_INVALID_ARG, "out_points is NULL");
        normals_impl(index, queries, nq, query_stride_bytes, k, eps, out_points, out_normals);
    });
}

static void radius_normals_impl(const pcpx_index* index, const float* queries, size_t nq,
                                size_t query_stride_bytes, const float* radii, float radius,
                                float* out_points, float* out_normals, uint32_t* out_count)
{
    pcpx_index& ix = checked(index);
    if (nq == 0)
        return;
    if (!out_normals)
        fail(PCPX_ERR_INVALID_ARG, "out_normals is NULL");
    ScopedDevice guard(ix.device);
    CallStream call(ix); // own stream: calls on one index may run concurrently
    CallTimer timer(ix);
    Batch batch;
    batch.prepare(ix, queries, nq, query_stride_bytes);
    InBuf rad;
    rad.stage(radii, nq, 4, 1, ix.qstream());
    OutBuf<float> nrm, ctr;
    OutBuf<uint32_t> cnt;
    nrm.prepare(out_normals, nq * 3);
    ctr.prepare(out_points, nq * 3);
    cnt.prepare(out_count, nq);
    timer.kernel_begin();
    launch_radius_normals(ix, batch.qb, rad.d, radius, nrm.d, ctr.d, cnt.d);
    timer.kernel_end();
    ix.timings.kernel_launches = 1;
    nrm.finish(ix.qstream()), ctr.finish(ix.qstream()), cnt.finish(ix.qstream());
    timer.done();
}

int pcpx_estimate_normals_radius(const pcpx_index* index, const float* queries, size_t nq,
                                 size_t query_stride_bytes, const float* radii, float radius,
                                 float* out_normals, uint32_t* out_count)
{
    return guarded([&] {
        radius_normals_impl(index, queries, nq, query_stride_bytes, radii, radius, nullptr,
                            out_normals, out_count);
    });
}

int pcpx_estimate_tangent_planes_radius(const pcpx_index* index, const float* queries, size_t nq,
                                        size_t query_stride_bytes, const float* radii,
                                        float radius, float* out_points, float* out_normals,
                                        uint32_t* out_count)
{
    return guarded([&] {
        if (nq && !out_points)
            fail(PCPX_ERR_INVALID_ARG, "out_points is NULL");
        radius_normals_impl(index, queries, nq, query_stride_bytes, radii, radius, out_points,
                            out_normals, out_count);
    });
}

int pcpx_normals_from_neighbourhoods(const float* nbr_xyz, const uint64_t* offsets, size_t n,
                                     int device, float* out_normals)
{
    return guarded([&] {
        if (n == 0)
            return;
        if (!offsets || !out_normals)
            fail(PCPX_ERR_INVALID_ARG, "offsets / out_normals is NULL");
        if (n >= 0xFFFFFFFFull)
            fail(PCPX_ERR_UNSUPPORTED, "more than 2^32 - 2 neighbourhoods in one call");
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
            fail(PCPX_ERR_NO_DEVICE, "no CUDA device: libpcpx has no CPU path");
        if (device < 0)
            PCPX_CUDA(cudaGetDevice(&device));
        ScopedDevice guard(device);
        cudaStream_t stream = nullptr; // legacy default stream: this call owns no index
        DevBuf<uint64_t> d_off_buf;
        const uint64_t* d_off = offsets;
        uint64_t total        = 0;
        if (!is_device_pointer(offsets))
        {
            total = offsets[n];
            d_off_buf.alloc(n + 1);
            PCPX_CUDA(cudaMemcpyAsync(d_off_buf.get(), offsets, (n + 1) * 8,
                                      cudaMemcpyHostToDevice, stream));
            d_off = d_off_buf.get();
        }
        else
            PCPX_CUDA(cudaMemcpy(&total, offsets + n, 8, cudaMemcpyDeviceToHost));
        if (total && !nbr_xyz)
            fail(PCPX_ERR_INVALID_ARG, "nbr_xyz is NULL");
        InBuf pts;
        pts.stage(nbr_xyz, total, 12, 3, stream);
        OutBuf<float> out;
        out.prepare(out_normals, n * 3);
        launch_normals_from_neighbourhoods(stream, pts.d, d_off, (uint32_t)n, out.d);
        out.finish(stream);
        PCPX_CUDA(cudaStreamSynchronize(stream));
    });
}

int pcpx_mean_knn_distance(const pcpx_index* index, uint32_t k, double eps, float* out_per_point,
                           double* out_mean)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        size_t const n = ix.n_input;
        if (n == 0)
        {
            if (out_mean)
                *out_mean = std::nan("");
            return;
        }
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        QueryBatch qb{nullptr, 3u, nullptr, (uint32_t)n};
        OutBuf<float> means;
        DevBuf<float> scratch;
        if (out_per_point)
            means.prepare(out_per_point, n);
        else
        {
            scratch.alloc(n);
            means.d = scratch.get();
        }
        DevBuf<double> sum(1);
        DevBuf<uint32_t> valid(1);
        timer.kernel_begin();
        if (sharded(ix, k))
        {
            size_t const nrep = ix.replicas.size();
            std::vector<ShardInfo> shards(nrep + 1);
            ShardedOut<float> s_mean(means.d, n, 1, nrep);
            on_every_device(ix, [&](pcpx_index& dev_ix, uint32_t part) {
                QueryBatch q = qb;
                q.part = part, q.parts = (uint32_t)nrep + 1u;
                q.by_position = part != 0, q.shard_info = &shards[part];
                float* p_mean = s_mean.target(part);
                launch_mean_distance(dev_ix, q, k, (float)eps, p_mean);
            });
            s_mean.gather(ix, qb, shards);
            PCPX_CUDA(cudaStreamSynchronize(ix.qstream())); // before the replicas' buffers go
        }
        else
            launch_mean_distance(ix, qb, k, (float)eps, means.d);
        launch_mean_reduce(ix, means.d, (uint32_t)n, sum.get(), valid.get());
        timer.kernel_end();
        ix.timings.kernel_launches = knn_shaped_launches(ix, k, false) + 2u; // + the two-stage reduction
        means.finish(ix.qstream());
        double h_sum = 0;
        uint32_t h_valid = 0;
        timer.done();
        read_back(ix.qstream(), &h_sum, sum.get(), 8);
        read_back(ix.qstream(), &h_valid, valid.get(), 4);
        if (out_mean)
            *out_mean = h_valid == n ? h_sum / (double)n : std::nan("");
    });
}

int pcpx_density_filter(const pcpx_index* index, float radius, uint32_t threshold,
                        uint8_t* out_keep_mask, float* out_xyz, size_t* out_n)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        size_t const n = ix.n_input;
        if (out_n)
            *out_n = 0;
        if (n == 0)
            return;
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        OutBuf<uint8_t> keep;
        DevBuf<uint8_t> keep_scratch;
        if (out_keep_mask)
            keep.prepare(out_keep_mask, n);
        else
        {
            keep_scratch.alloc(n);
            keep.d = keep_scratch.get();
        }
        OutBuf<float> pts;
        pts.prepare(out_xyz, n * 3);
        DevBuf<uint64_t> scan(n + 1);
        timer.kernel_begin();
        launch_density_keep(ix, radius, threshold, keep.d);
        launch_exclusive_scan_u8(ix, keep.d, (uint32_t)n, scan.get());
        if (out_xyz)
            launch_compact_points(ix, keep.d, scan.get(), pts.d);
        timer.kernel_end();
        ix.timings.kernel_launches = out_xyz ? 5 : 4;
        uint64_t kept = 0;
        PCPX_CUDA(cudaMemcpyAsync(&kept, scan.get() + n, 8, cudaMemcpyDeviceToHost, ix.qstream()));
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
        keep.finish(ix.qstream());
        pts.finish(ix.qstream(), kept * 3);
        timer.done();
        if (out_n)
            *out_n = (size_t)kept;
    });
}

int pcpx_cluster_by_density(const pcpx_index* index, float radius, uint32_t min_points,
                            uint32_t* out_labels, uint64_t* out_n_clusters)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (std::isnan(radius))
            fail(PCPX_ERR_INVALID_ARG, "radius is NaN");
        if (out_n_clusters)
            *out_n_clusters = 0;
        size_t const n = ix.n_input;
        if (n == 0)
            return;
        if (!out_labels)
            fail(PCPX_ERR_INVALID_ARG, "out_labels is NULL");
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        OutBuf<uint32_t> labels;
        labels.prepare(out_labels, n);
        uint32_t launches = 0;
        timer.kernel_begin();
        uint64_t const n_clusters = launch_cluster_by_density(ix, radius, min_points, labels.d,
                                                              &launches);
        timer.kernel_end();
        ix.timings.kernel_launches = launches;
        labels.finish(ix.qstream());
        timer.done();
        if (out_n_clusters)
            *out_n_clusters = n_clusters;
    });
}

int pcpx_last_timings(const pcpx_index* index, pcpx_timings* out)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out)
            fail(PCPX_ERR_INVALID_ARG, "out is NULL");
        *out = ix.timings;
        out->deferred_queries = ix.deferred_queries;
        out->expanded_queries = ix.expanded_queries;
    });
}

int pcpx_set_tuning(const char* name, double value)
{
    return guarded([&] {
        if (!name)
            fail(PCPX_ERR_INVALID_ARG, "name is NULL");
        if (!std::strcmp(name, "success_margin"))
            tuning().success_margin = (float)value;
        else if (!std::strcmp(name, "pool_cap_mb"))
            DevicePool::instance().set_cap((size_t)std::max(0.0, value) << 20);
        else if (!std::strcmp(name, "tile"))
            tuning().tile = (int)value;
        else if (!std::strcmp(name, "warp_retry"))
            tuning().warp_retry = (int)value;
        else if (!std::strcmp(name, "warp_all"))
            tuning().warp_all = (int)value;
        else if (!std::strcmp(name, "tile_first_cap"))
            tuning().tile_first_cap = (int)value;
        else if (!std::strcmp(name, "tile_min_queries"))
            tuning().tile_min_queries = (int)value;
        else if (!std::strcmp(name, "tile_sub"))
            tuning().tile_sub = (int)value;
        else if (!std::strcmp(name, "tile_cap"))
            tuning().tile_cap = (float)value;
        else if (!std::strcmp(name, "tile_margin"))
            tuning().tile_margin = (float)value;
        else
            fail(PCPX_ERR_INVALID_ARG, "unknown tuning parameter '%s'", name);
    });
}

int pcpx_host_alloc(size_t bytes, void** out_ptr)
{
    return guarded([&] {
        if (!out_ptr)
            fail(PCPX_ERR_INVALID_ARG, "out_ptr is NULL");
        *out_ptr = nullptr;
        if (bytes == 0)
            return;
        if (pcpx_device_count() < 1)
            fail(PCPX_ERR_NO_DEVICE, "no CUDA device: libpcpx has no CPU path");
        PCPX_CUDA(cudaHostAlloc(out_ptr, bytes, cudaHostAllocPortable));
    });
}

void pcpx_host_free(void* ptr)
{
    if (ptr)
        cudaFreeHost(ptr);
}

int pcpx_trim(int device)
{
    return guarded([&] {
        int n = 0;
        PCPX_CUDA(cudaGetDeviceCount(&n));
        if (device < 0 || device >= n)
            fail(PCPX_ERR_INVALID_ARG, "device %d out of range", device);
        ScopedDevice guard(device);
        PCPX_CUDA(cudaDeviceSynchronize());
        DevicePool::instance().trim(device);
    });
}

int pcpx_debug_knn_stats(const pcpx_index* index, uint32_t k, double eps, uint64_t* out4)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        if (!out4)
            fail(PCPX_ERR_INVALID_ARG, "out4 is NULL");
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        DevBuf<unsigned long long> st(4);
        PCPX_CUDA(cudaMemsetAsync(st.get(), 0, 32, ix.qstream()));
        launch_knn_stats(ix, k, (float)eps, st.get());
        PCPX_CUDA(cudaMemcpyAsync(out4, st.get(), 32, cudaMemcpyDeviceToHost, ix.qstream()));
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
    });
}

} // extern "C"
