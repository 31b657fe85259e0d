// The GPU-resident index object behind the opaque pcpx_index handle.
#pragma once
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

#include "grid_core.cuh"
#include "host_util.hpp"

struct pcpx_index
{
    int device          = 0;
    cudaStream_t stream = nullptr;
    uint64_t n_input    = 0; // points handed in (sorted array length)
    uint64_t n_indexed  = 0; // points inside the root voxel
    float bbox_min[3]{}, bbox_max[3]{};
    uint32_t code_bits = 0;
    uint64_t n_cells   = 0;
    uint64_t cells_per_level[pcpx::kMaxLevel + 2] = {}; // occupied cells at each stored level
    pcpx::GridView grid{}; // device pointers into the buffers below
    pcpx::DevBuf<float4> pts;          // n_input entries, Morton order; w = original index
    pcpx::DevBuf<pcpx::HashSlot> table; // all levels
    pcpx::DevBuf<uint8_t> bnd;          // n_indexed entries: coarsest level at which sorted point i opens a new cell
    pcpx_timings timings{-1.f, -1.f, -1.f, -1.f, -1.f, 0u, 0u, 0u, 0u};
    // Concurrency.  The index is immutable once built, and the query entry points of the path
    // (kNN, radius, normals, mean distance, density filter) may be called from several host
    // threads at once: each call borrows its own stream (call_streams, below) and its own
    // temporaries, the lazily built tile lists are immutable once made, and the statistics of
    // "the last call" (`timings`, the counters below) are last-writer-wins: with calls in flight
    // from several threads pcpx_last_timings may mix fields of different calls.  `mtx` still serialises the calls that keep state
    // on the index's own stream (orientation, smoothing).
    std::mutex mtx;
    // tile list of one level (query.cu: ensure_tile_list), built on first use and kept for the
    // life of the index: starts[i] = first sorted position of tile i, starts[n_tiles] = n_indexed
    struct TileList
    {
        pcpx::DevBuf<uint32_t> starts, count, scratch;
        pcpx::DevBuf<uint64_t> xyz; // tile coordinates (tile_core.cuh: tile_pack)
        uint32_t capacity = 0;
        uint32_t region   = 0; // staged-region capacity that fits 97 % of the queries' tiles
    };
    mutable std::mutex tile_mtx;
    mutable std::map<int, std::unique_ptr<TileList>> tile_lists;
    mutable std::atomic<uint32_t> query_launches{0};   // kernels launched by the last kNN-shaped call
    mutable std::atomic<uint32_t> deferred_queries{0}; // ... queries its first pass handed on
    mutable std::atomic<uint32_t> expanded_queries{0}; // ... of those, not final at the first block
    cudaStream_t qstream() const; // the calling thread's stream for this index (index.hpp, below)
    // the same index on further devices (pcpx_index_params.devices[1..]); owned
    std::vector<pcpx_index*> replicas;

    ~pcpx_index()
    {
        for (pcpx_index* r : replicas)
        {
            cudaSetDevice(r->device);
            delete r;
        }
        cudaSetDevice(device);
        if (stream)
            cudaStreamDestroy(stream);
    }
    size_t device_bytes() const { return pts.bytes() + table.bytes() + bnd.bytes(); }
};

namespace pcpx {

// The stream a query call runs on: while a CallStream is alive on this thread for this index its
// borrowed stream, otherwise the index's own.
struct CallStreamSlot
{
    const pcpx_index* ix = nullptr;
    cudaStream_t s       = nullptr;
};
inline CallStreamSlot& call_stream_slot()
{
    static thread_local CallStreamSlot slot;
    return slot;
}
// Streams for concurrent calls are pooled per DEVICE for the life of the process (a serving loop
// that rebuilds its index for every cloud would otherwise create and destroy one per cloud).
struct CallStreamPool
{
    std::mutex m;
    std::map<int, std::vector<cudaStream_t>> idle;
    static CallStreamPool& instance()
    {
        static CallStreamPool* p = new CallStreamPool(); // (never destroyed: no teardown order issues)
        return *p;
    }
};
class CallStream
{
  public:
    explicit CallStream(const pcpx_index& ix) : device_(ix.device), prev_(call_stream_slot())
    {
        cudaStream_t s = nullptr;
        {
            CallStreamPool& pool = CallStreamPool::instance();
            std::lock_guard<std::mutex> lock(pool.m);
            auto& idle = pool.idle[device_];
            if (!idle.empty())
            {
                s = idle.back();
                idle.pop_back();
            }
        }
        if (!s)
            PCPX_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)); // (current device = ix.device)
        call_stream_slot() = CallStreamSlot{&ix, s};
    }
    ~CallStream()
    {
        cudaStream_t const s = call_stream_slot().s;
        call_stream_slot()   = prev_;
        CallStreamPool& pool = CallStreamPool::instance();
        std::lock_guard<std::mutex> lock(pool.m);
        pool.idle[device_].push_back(s);
    }
    CallStream(const CallStream&)            = delete;
    CallStream& operator=(const CallStream&) = delete;

  private:
    int device_;
    CallStreamSlot prev_;
};

// index.cu
pcpx_index* build_index(const float* xyz, size_t n, size_t stride_bytes,
                        const pcpx_index_params* params);

// Sort helper exported by index.cu for query batches: fills `order` (device, nq entries) with
// the query permutation sorted by fine Morton code of the query positions; adds the kernels it
// launched to *launches when given.
void sort_queries_by_cell(const pcpx_index& ix, const float* d_queries, uint32_t stride_floats,
                          uint32_t nq, uint32_t* d_order, uint32_t* launches = nullptr);

// Stable LSD radix sort (radix_sort.cuh) of n (key, value) pairs by key bits [0, n_bits), in
// place, on the calling thread's stream; adds the kernels it launched to *launches.
void sort_pairs_u64(const pcpx_index& ix, uint64_t* keys, uint32_t* vals, uint32_t n, int n_bits,
                    uint32_t* launches);

} // namespace pcpx

inline cudaStream_t pcpx_index::qstream() const
{
    pcpx::CallStreamSlot const& slot = pcpx::call_stream_slot();
    return slot.ix == this ? slot.s : stream;
}
