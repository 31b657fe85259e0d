// Rigid registration (pcpx_icp): the host side of one ICP iteration — the fp64 solve of the
// reduced normal equations, the rigid update, the stopping rules — and the iteration loop itself.
// Host-only C++ (no CUDA), so that the CPU emulation (tests/emu/emu_icp.cu) runs the same code
// as the library.  Compile with -ffp-contract=off: the results are specified bit for bit only
// for a given order of fp64 operations, and that order is the one written here.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

namespace pcpx {

// Layout of the reduced sums (icp_core.cuh writes them, everything here reads them).
//   point-to-plane: [0, 21) A = sum J^T J, upper triangle row by row; [21, 27) b = sum J^T r;
//                   27: sum d2; 28: pairs.  J = [(y - c) x n, n], r = (y - q) . n
//   point-to-point: [0, 3) sum (y - c); [3, 6) sum (q - c); [6, 15) sum (y - c)_a (q - c)_b,
//                   row a, column b; 15: sum d2; 16: pairs
constexpr int kIcpPlaneTerms = 29;
constexpr int kIcpPointTerms = 17;
constexpr int kIcpMaxTerms   = 29;

inline int icp_terms(uint32_t metric) { return metric == 0 ? kIcpPlaneTerms : kIcpPointTerms; }
inline double icp_pairs(uint32_t metric, const double* s) { return s[icp_terms(metric) - 1]; }
inline double icp_sum_d2(uint32_t metric, const double* s) { return s[icp_terms(metric) - 2]; }

// Symmetric eigendecomposition by cyclic Jacobi: a (n x n, row-major, destroyed) = V diag(w) V^T,
// eigenvector i in column i of v.  Rotations in the fixed order (p, q) = (0,1), (0,2), ...,
// (n-2, n-1); at most 50 sweeps, ending early once the off-diagonal part is exactly zero or
// negligible against the diagonal.
inline void jacobi_eigen(double* a, int n, double* w, double* v)
{
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
            v[i * n + j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 50; ++sweep)
    {
        double off = 0.0, diag = 0.0;
        for (int p = 0; p < n; ++p)
        {
            diag += a[p * n + p] * a[p * n + p];
            for (int q = p + 1; q < n; ++q)
                off += a[p * n + q] * a[p * n + q];
        }
        if (off == 0.0 || off <= 1e-60 * diag)
            break;
        for (int p = 0; p < n - 1; ++p)
            for (int q = p + 1; q < n; ++q)
            {
                double const apq = a[p * n + q];
                if (apq == 0.0)
                    continue;
                double const theta = (a[q * n + q] - a[p * n + p]) / (2.0 * apq);
                double const t     = (theta >= 0.0 ? 1.0 : -1.0) /
                                 (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                double const c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < n; ++k) // columns p, q
                {
                    double const akp = a[k * n + p], akq = a[k * n + q];
                    a[k * n + p] = c * akp - s * akq;
                    a[k * n + q] = s * akp + c * akq;
                }
                for (int k = 0; k < n; ++k) // rows p, q
                {
                    double const apk = a[p * n + k], aqk = a[q * n + k];
                    a[p * n + k] = c * apk - s * aqk;
                    a[q * n + k] = s * apk + c * aqk;
                }
                for (int k = 0; k < n; ++k)
                {
                    double const vkp = v[k * n + p], vkq = v[k * n + q];
                    v[k * n + p] = c * vkp - s * vkq;
                    v[k * n + q] = s * vkp + c * vkq;
                }
            }
    }
    for (int i = 0; i < n; ++i)
        w[i] = a[i * n + i];
}

// Point-to-plane step: x = (omega, v) = -A^+ b, A^+ the pseudo-inverse from the eigendecomposition
// with the eigenvalues <= 1e-12 * lambda_max dropped (a direction the pairs do not constrain —
// in-plane sliding of a plane — gets no motion instead of an arbitrary one).
inline void icp_solve_plane(const double* s, double x[6])
{
    double a[36], w[6], v[36];
    for (int i = 0, k = 0; i < 6; ++i)
        for (int j = i; j < 6; ++j, ++k)
            a[i * 6 + j] = a[j * 6 + i] = s[k];
    const double* b = s + 21;
    jacobi_eigen(a, 6, w, v);
    double lmax = 0.0;
    for (int i = 0; i < 6; ++i)
        lmax = std::fmax(lmax, w[i]);
    for (int j = 0; j < 6; ++j)
        x[j] = 0.0;
    for (int i = 0; i < 6; ++i)
    {
        if (!(w[i] > 1e-12 * lmax))
            continue;
        double vb = 0.0;
        for (int j = 0; j < 6; ++j)
            vb += v[j * 6 + i] * b[j];
        double const f = -vb / w[i];
        for (int j = 0; j < 6; ++j)
            x[j] += f * v[j * 6 + i];
    }
}

// Point-to-point step by Horn's closed-form quaternion method: the rotation is the unit
// eigenvector of the largest eigenvalue of Horn's 4 x 4 matrix of the centred cross-covariance,
// which is always a proper rotation (never a reflection).  Returned as the rotation vector omega
// (angle in [0, pi]) and v = mean(q - c) - R(omega) mean(y - c), so that y -> R (y - c) + c + v
// maps the centroid of the y onto the centroid of the q.
inline void rodrigues(const double w[3], double R[9]);

inline void icp_solve_point(const double* s, double x[6])
{
    double const n = s[16];
    double my[3], mq[3], S[9];
    for (int a = 0; a < 3; ++a)
        my[a] = s[a] / n, mq[a] = s[3 + a] / n;
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b)
            S[a * 3 + b] = s[6 + a * 3 + b] - n * my[a] * mq[b];
    double const xx = S[0], xy = S[1], xz = S[2], yx = S[3], yy = S[4], yz = S[5], zx = S[6],
                 zy = S[7], zz = S[8];
    double N[16] = {xx + yy + zz, yz - zy,       zx - xz,       xy - yx,
                    yz - zy,      xx - yy - zz,  xy + yx,       zx + xz,
                    zx - xz,      xy + yx,       -xx + yy - zz, yz + zy,
                    xy - yx,      zx + xz,       yz + zy,       -xx - yy + zz};
    double w[4], V[16];
    jacobi_eigen(N, 4, w, V);
    int best = 0;
    for (int i = 1; i < 4; ++i)
        if (w[i] > w[best])
            best = i;
    double q[4] = {V[0 * 4 + best], V[1 * 4 + best], V[2 * 4 + best], V[3 * 4 + best]};
    if (q[0] < 0.0)
        for (double& e : q)
            e = -e;
    double const sn = std::sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    double const angle = 2.0 * std::atan2(sn, q[0]);
    for (int a = 0; a < 3; ++a)
        x[a] = sn > 0.0 ? q[1 + a] / sn * angle : 0.0;
    double R[9];
    rodrigues(x, R);
    for (int a = 0; a < 3; ++a)
        x[3 + a] = mq[a] - ((R[a * 3] * my[0] + R[a * 3 + 1] * my[1]) + R[a * 3 + 2] * my[2]);
}

// R(omega) = I + sin(t) K + (1 - cos(t)) K^2, K the cross-product matrix of omega / t, t = |omega|
inline void rodrigues(const double w[3], double R[9])
{
    double const t = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
    for (int i = 0; i < 9; ++i)
        R[i] = (i % 4 == 0) ? 1.0 : 0.0;
    if (t == 0.0)
        return;
    double const k[3] = {w[0] / t, w[1] / t, w[2] / t};
    double const K[9] = {0.0, -k[2], k[1], k[2], 0.0, -k[0], -k[1], k[0], 0.0};
    double K2[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            K2[i * 3 + j] = (K[i * 3] * K[j]) + (K[i * 3 + 1] * K[3 + j]) + (K[i * 3 + 2] * K[6 + j]);
    double const st = std::sin(t), ct = 1.0 - std::cos(t);
    for (int i = 0; i < 9; ++i)
        R[i] += st * K[i] + ct * K2[i];
}

// T <- U o T with U(y) = R(omega) (y - c) + c + v; T row-major 4 x 4 with last row (0, 0, 0, 1)
inline void icp_update(double T[16], const double x[6], const double c[3])
{
    double R[9];
    rodrigues(x, R);
    double U[16] = {};
    for (int a = 0; a < 3; ++a)
    {
        for (int b = 0; b < 3; ++b)
            U[a * 4 + b] = R[a * 3 + b];
        U[a * 4 + 3] = c[a] + x[3 + a] - ((R[a * 3] * c[0] + R[a * 3 + 1] * c[1]) + R[a * 3 + 2] * c[2]);
    }
    U[15] = 1.0;
    double out[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j)
            out[i * 4 + j] = ((U[i * 4] * T[j] + U[i * 4 + 1] * T[4 + j]) + U[i * 4 + 2] * T[8 + j]) +
                             U[i * 4 + 3] * T[12 + j];
    std::memcpy(T, out, sizeof out);
}

struct IcpLoopResult
{
    uint32_t iterations;
    uint32_t stop_reason; // 0 converged, 1 max iterations, 2 too few pairs
};

// The iteration loop of pcpx_icp.  pass(T, sums) runs one correspondence pass under T and writes
// the reduced sums (layout above); T is updated in place.
template <class Pass>
IcpLoopResult icp_loop(uint32_t metric, uint32_t max_iterations, double rot_tol, double trans_tol,
                       const double c[3], double T[16], Pass&& pass)
{
    double const min_pairs = metric == 0 ? 6.0 : 3.0;
    double s[kIcpMaxTerms];
    for (uint32_t it = 0; it < max_iterations; ++it)
    {
        pass(T, s);
        if (icp_pairs(metric, s) < min_pairs)
            return IcpLoopResult{it, 2u};
        double x[6];
        if (metric == 0)
            icp_solve_plane(s, x);
        else
            icp_solve_point(s, x);
        icp_update(T, x, c);
        double const rw = std::sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
        double const rv = std::sqrt(x[3] * x[3] + x[4] * x[4] + x[5] * x[5]);
        if (rw <= rot_tol && rv <= trans_tol)
            return IcpLoopResult{it + 1, 0u};
    }
    return IcpLoopResult{max_iterations, 1u};
}

} // namespace pcpx
