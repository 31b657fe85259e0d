// Rigid registration: pcpx_nearest_within (bounded nearest neighbour of transformed queries) and
// pcpx_icp (iterative closest point against the index), the bodies in icp_core.cuh, the host
// solve and the loop in icp_solve.hpp.  One correspondence pass on the device:
//   1. transform: y = T x in fp64, rounded once to fp32, into a packed buffer
//   2. sort the y by cell (sort_queries_by_cell), so that the lanes of a warp walk the same cells
//   3. one thread per sorted query: the nearest-within walk, then (ICP) the pair's terms of the
//      normal equations reduced over the block — warp butterflies in a fixed order, the warps
//      added in warp order — into one fp64 partial per block and term
//   4. one CTA per term adds the partials of all blocks with a fixed shape (strided, then a tree)
// The shapes depend on the number of queries alone, so the sums are bit-identical from run to run.
#include <cmath>

#include "api_util.hpp"
#include "icp_core.cuh"
#include "icp_solve.hpp"
#include "plan.hpp"

using namespace pcpx;

namespace {

constexpr int kIcpBlock = 128;
constexpr int kIcpFinal = 256;

uint32_t icp_blocks(uint32_t n, int block) { return std::max(1u, (n + block - 1) / block); }

__global__ void __launch_bounds__(256) icp_transform_kernel(const float* __restrict__ src,
                                                            uint32_t stride_f, uint32_t n,
                                                            Rigid34 T, float* __restrict__ y)
{
    uint32_t const i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n)
        return;
    const float* p = src + (size_t)i * stride_f;
    float o[3];
    rigid_apply(T, __ldg(p), __ldg(p + 1), __ldg(p + 2), o);
    y[3 * (size_t)i] = o[0], y[3 * (size_t)i + 1] = o[1], y[3 * (size_t)i + 2] = o[2];
}

__global__ void __launch_bounds__(kIcpBlock, 8) nearest_within_kernel(
    GridView g, int level, const float* __restrict__ y, uint32_t stride_f,
    const uint32_t* __restrict__ order, uint32_t n, float r, uint32_t* __restrict__ out_idx,
    float* __restrict__ out_d2)
{
    uint32_t const t = blockIdx.x * kIcpBlock + threadIdx.x;
    if (t >= n)
        return;
    uint32_t const row = order ? order[t] : t;
    const float* p     = y + (size_t)row * stride_f;
    uint32_t pos;
    uint64_t const key = nearest_within(g, level, __ldg(p), __ldg(p + 1), __ldg(p + 2), r, pos);
    out_idx[row] = key == kIcpNoKey ? kIcpNone : (uint32_t)key;
    if (out_d2)
        out_d2[row] = key == kIcpNoKey ? INFINITY : u2f((uint32_t)(key >> 32));
}

// partial[k * n_blocks + block] = term k summed over the block's pairs
template <uint32_t METRIC>
__global__ void __launch_bounds__(kIcpBlock) icp_pass_kernel(
    GridView g, int level, const float* __restrict__ y, const uint32_t* __restrict__ order,
    uint32_t n, float r, const float* __restrict__ normals, uint32_t normal_stride_f, double cx,
    double cy, double cz, double* __restrict__ partial, uint32_t* __restrict__ out_corr)
{
    constexpr int NT = METRIC == 0 ? kIcpPlaneTerms : kIcpPointTerms;
    uint32_t const t = blockIdx.x * kIcpBlock + threadIdx.x;
    IcpPair P{};
    bool valid = false;
    if (t < n)
    {
        uint32_t const row = order ? order[t] : t;
        float const yv[3]  = {__ldg(y + 3 * (size_t)row), __ldg(y + 3 * (size_t)row + 1),
                              __ldg(y + 3 * (size_t)row + 2)};
        uint32_t pos;
        uint64_t const key = nearest_within(g, level, yv[0], yv[1], yv[2], r, pos);
        uint32_t corr      = kIcpNone;
        if (key != kIcpNoKey)
        {
            uint32_t const orig = (uint32_t)key;
            float nrm[3]        = {0.f, 0.f, 0.f};
            if (METRIC == 0)
            {
                const float* np = normals + (size_t)orig * normal_stride_f;
                nrm[0] = __ldg(np), nrm[1] = __ldg(np + 1), nrm[2] = __ldg(np + 2);
            }
            if (icp_pair_valid(METRIC, nrm))
            {
                double const c[3] = {cx, cy, cz};
                P     = icp_pair(METRIC, yv, __ldg(g.pts + pos), nrm, c, u2f((uint32_t)(key >> 32)));
                valid = true;
                corr  = orig;
            }
        }
        if (out_corr)
            out_corr[row] = corr;
    }
    __shared__ double sh[kIcpBlock / 32][NT];
    int const lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NT; ++k)
    {
        double v = valid ? icp_term(METRIC, P, k) : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            v = dadd_x(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
        if (lane == 0)
            sh[warp][k] = v;
    }
    __syncthreads();
    if ((int)threadIdx.x < NT)
    {
        double s = sh[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < kIcpBlock / 32; ++w)
            s = dadd_x(s, sh[w][threadIdx.x]);
        partial[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = s;
    }
}

// block k: out[k] = sum of partial[k * n_blocks ...]: thread t adds blocks t, t + 256, ... in
// order, then a fixed tree over the threads
__global__ void __launch_bounds__(kIcpFinal) icp_final_kernel(const double* __restrict__ partial,
                                                              uint32_t n_blocks,
                                                              double* __restrict__ out)
{
    __shared__ double sh[kIcpFinal];
    const double* p = partial + (size_t)blockIdx.x * n_blocks;
    double s        = 0.0;
    for (uint32_t b = threadIdx.x; b < n_blocks; b += kIcpFinal)
        s = dadd_x(s, p[b]);
    sh[threadIdx.x] = s;
    __syncthreads();
#pragma unroll
    for (int o = kIcpFinal / 2; o > 0; o >>= 1)
    {
        if ((int)threadIdx.x < o)
            sh[threadIdx.x] = dadd_x(sh[threadIdx.x], sh[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0)
        out[blockIdx.x] = sh[0];
}

Rigid34 rigid34(const double T[16])
{
    Rigid34 r;
    for (int i = 0; i < 12; ++i)
        r.m[i] = T[i];
    return r;
}

void check_max_distance(float max_distance)
{
    if (!(max_distance > 0.f) || !(max_distance <= 3.402823466e38f))
        fail(PCPX_ERR_INVALID_ARG, "max_distance must be finite and > 0, got %g",
             (double)max_distance);
}

size_t checked_stride(size_t stride_bytes, const char* what)
{
    if (stride_bytes == 0)
        stride_bytes = 12;
    if (stride_bytes < 12 || stride_bytes % 4)
        fail(PCPX_ERR_INVALID_ARG, "%s must be a multiple of 4 and >= 12", what);
    return stride_bytes;
}

// the level a k = 1 search starts at: the kNN planner's
int nearest_level(const pcpx_index& ix)
{
    return choose_plan(ix.n_indexed, ix.cells_per_level, ix.grid.lfine, 1u,
                       (double)tuning().success_margin)
        .level;
}

// The transformed queries of a call, sorted by cell.  T == nullptr: the queries as they are.
struct IcpQueries
{
    DevBuf<float> y;
    DevBuf<uint32_t> order;
    const float* d    = nullptr;
    uint32_t stride_f = 3;
    uint32_t n        = 0;

    void prepare(pcpx_index& ix, const InBuf& in, uint32_t nq, const double* T, uint32_t* launches)
    {
        n = nq;
        d = in.d, stride_f = in.stride_f;
        if (T)
        {
            if (!y.get())
                y.alloc((size_t)nq * 3);
            icp_transform_kernel<<<icp_blocks(nq, 256), 256, 0, ix.qstream()>>>(
                in.d, in.stride_f, nq, rigid34(T), y.get());
            PCPX_CHECK_LAUNCH();
            *launches += 1;
            d = y.get(), stride_f = 3;
        }
        if (!order.get())
            order.alloc(nq);
        Event s0, s1;
        s0.record(ix.qstream());
        sort_queries_by_cell(ix, d, stride_f, nq, order.get(), launches);
        s1.record(ix.qstream());
        PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
        ix.timings.query_sort_ms += elapsed_ms(s0, s1);
    }
};

} // namespace

extern "C" {

int pcpx_nearest_within(const pcpx_index* index, const float* queries, size_t nq,
                        size_t query_stride_bytes, const double transform[16], float max_distance,
                        uint32_t* out_idx, float* out_d2)
{
    return guarded([&] {
        pcpx_index& ix = checked(index);
        check_max_distance(max_distance);
        size_t const stride = checked_stride(query_stride_bytes, "query_stride_bytes");
        if (nq == 0)
            return;
        if (nq >= 0xFFFFFFFFull)
            fail(PCPX_ERR_UNSUPPORTED, "more than 2^32 - 2 queries in one call");
        if (!queries || !out_idx)
            fail(PCPX_ERR_INVALID_ARG, "queries / out_idx is NULL");
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        InBuf in;
        in.stage(queries, nq, stride, 3, ix.qstream());
        OutBuf<uint32_t> idx;
        OutBuf<float> d2;
        idx.prepare(out_idx, nq);
        d2.prepare(out_d2, nq);
        uint32_t launches = 0;
        timer.kernel_begin();
        IcpQueries q;
        q.prepare(ix, in, (uint32_t)nq, transform, &launches);
        nearest_within_kernel<<<icp_blocks((uint32_t)nq, kIcpBlock), kIcpBlock, 0, ix.qstream()>>>(
            ix.grid, nearest_level(ix), q.d, q.stride_f, q.order.get(), (uint32_t)nq, max_distance,
            idx.d, d2.d);
        PCPX_CHECK_LAUNCH();
        timer.kernel_end();
        ix.timings.kernel_launches = launches + 1;
        idx.finish(ix.qstream()), d2.finish(ix.qstream());
        timer.done();
    });
}

int pcpx_icp(const pcpx_index* target, const float* target_normals, size_t normal_stride_bytes,
             const float* source, size_t ns, size_t source_stride_bytes,
             const pcpx_icp_params* params, const double init[16], double out_transform[16],
             pcpx_icp_result* out_result, uint32_t* out_correspondences)
{
    return guarded([&] {
        pcpx_index& ix = checked(target);
        if (!params || !out_transform)
            fail(PCPX_ERR_INVALID_ARG, "params / out_transform is NULL");
        pcpx_icp_params const prm = *params;
        if (prm.metric != PCPX_ICP_POINT_TO_PLANE && prm.metric != PCPX_ICP_POINT_TO_POINT)
            fail(PCPX_ERR_INVALID_ARG, "unknown metric %u", prm.metric);
        check_max_distance(prm.max_distance);
        uint32_t const metric = prm.metric;
        if (metric == PCPX_ICP_POINT_TO_PLANE && !target_normals)
            fail(PCPX_ERR_INVALID_ARG, "point-to-plane needs the target's normals");
        size_t const sstride = checked_stride(source_stride_bytes, "source_stride_bytes");
        size_t const nstride = checked_stride(normal_stride_bytes, "normal_stride_bytes");
        if (ns >= 0xFFFFFFFFull)
            fail(PCPX_ERR_UNSUPPORTED, "more than 2^32 - 2 source points in one call");
        if (ns && !source)
            fail(PCPX_ERR_INVALID_ARG, "source is NULL");
        double T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
        if (init)
            std::memcpy(T, init, sizeof T);
        uint32_t const max_it = prm.max_iterations ? prm.max_iterations : 30u;
        double const c[3] = {0.5 * ((double)ix.bbox_min[0] + (double)ix.bbox_max[0]),
                             0.5 * ((double)ix.bbox_min[1] + (double)ix.bbox_max[1]),
                             0.5 * ((double)ix.bbox_min[2] + (double)ix.bbox_max[2])};
        double diag = 0.0;
        for (int a = 0; a < 3; ++a)
        {
            double const e = (double)ix.bbox_max[a] - (double)ix.bbox_min[a];
            diag += e * e;
        }
        double const rot_tol   = prm.rotation_tolerance > 0.0 ? prm.rotation_tolerance : 1e-6;
        double const trans_tol = prm.translation_tolerance > 0.0 ? prm.translation_tolerance
                                                                  : 1e-6 * std::sqrt(diag);
        pcpx_icp_result res{0u, PCPX_ICP_TOO_FEW, 0u, 0.0, std::nan("")};
        ScopedDevice guard(ix.device);
        CallStream call(ix); // own stream: calls on one index may run concurrently
        CallTimer timer(ix);
        OutBuf<uint32_t> corr;
        corr.prepare(out_correspondences, ns);
        uint32_t launches = 0;
        timer.kernel_begin();
        if (ns && ix.n_indexed)
        {
            InBuf src, nrm;
            src.stage(source, ns, sstride, 3, ix.qstream());
            if (metric == PCPX_ICP_POINT_TO_PLANE)
                nrm.stage(target_normals, ix.n_input, nstride, 3, ix.qstream());
            uint32_t const n = (uint32_t)ns, nb = icp_blocks(n, kIcpBlock);
            int const nt = icp_terms(metric), level = nearest_level(ix);
            DevBuf<double> partial((size_t)nb * nt), sums(nt);
            IcpQueries q;
            auto pass = [&](const double* Tc, double* s, uint32_t* corr_d) {
                q.prepare(ix, src, n, Tc, &launches);
                if (metric == PCPX_ICP_POINT_TO_PLANE)
                    icp_pass_kernel<0><<<nb, kIcpBlock, 0, ix.qstream()>>>(
                        ix.grid, level, q.d, q.order.get(), n, prm.max_distance, nrm.d,
                        nrm.stride_f, c[0], c[1], c[2], partial.get(), corr_d);
                else
                    icp_pass_kernel<1><<<nb, kIcpBlock, 0, ix.qstream()>>>(
                        ix.grid, level, q.d, q.order.get(), n, prm.max_distance, nullptr, 0u,
                        c[0], c[1], c[2], partial.get(), corr_d);
                PCPX_CHECK_LAUNCH();
                icp_final_kernel<<<nt, kIcpFinal, 0, ix.qstream()>>>(partial.get(), nb, sums.get());
                PCPX_CHECK_LAUNCH();
                launches += 2;
                PCPX_CUDA(cudaMemcpyAsync(s, sums.get(), (size_t)nt * 8, cudaMemcpyDeviceToHost,
                                          ix.qstream()));
                PCPX_CUDA(cudaStreamSynchronize(ix.qstream()));
            };
            IcpLoopResult const lr =
                icp_loop(metric, max_it, rot_tol, trans_tol, c, T,
                         [&](const double* Tc, double* s) { pass(Tc, s, nullptr); });
            double s[kIcpMaxTerms];
            pass(T, s, corr.d); // the pairs of the returned transform
            double const pairs = icp_pairs(metric, s);
            res.iterations        = lr.iterations;
            res.stop_reason       = lr.stop_reason;
            res.n_correspondences = (uint64_t)pairs;
            res.fitness           = pairs / (double)ns;
            res.rmse = pairs > 0.0 ? std::sqrt(icp_sum_d2(metric, s) / pairs) : std::nan("");
        }
        else if (corr.d)
            PCPX_CUDA(cudaMemsetAsync(corr.d, 0xFF, ns * 4, ix.qstream()));
        timer.kernel_end();
        ix.timings.kernel_launches = launches;
        corr.finish(ix.qstream());
        timer.done();
        std::memcpy(out_transform, T, sizeof T);
        if (out_result)
            *out_result = res;
    });
}

} // extern "C"
