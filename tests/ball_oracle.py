"""CPU checker of the ball PCA (pcpx_estimate_normals_radius / _tangent_planes_radius).

TEST INFRASTRUCTURE — never used by the product.  It composes what the oracle library already
restates from the reference: the octree sphere range search (oracle_radius, the reference's DFS
order, so that the fp32 sums run in the reference's order) and, per ball, the reference's
estimate_normal body (oracle_scatter_matrix / oracle_estimate_normal).  Its fp64 companion
`bruteforce_ball_normals` checks that composition independently.
"""
import numpy as np


def radius_normals(cloud, queries, r, radii=None, exact_prune=0):
    """(normals, centroids, gaps, counts) of every query's ball over an OracleCloud.
    An empty ball: normal (0,0,1), NaN centroid, gap 0, count 0 (oracle_scatter_matrix)."""
    off, idx = cloud.radius_search(queries, r, radii, exact_prune=exact_prune)
    nq = len(off) - 1
    o = cloud.o
    nrm = np.zeros((nq, 3), np.float32)
    ctr = np.zeros((nq, 3), np.float32)
    gap = np.zeros(nq, np.float32)
    pts = cloud.xyz[idx] if len(idx) else np.zeros((0, 3), np.float32)
    for i in range(nq):
        p = pts[off[i]:off[i + 1]]
        nrm[i], gap[i] = o.estimate_normal(p)
        ctr[i] = o.scatter_matrix(p)[1]
    return nrm, ctr, gap, np.diff(off.astype(np.int64)).astype(np.uint32)


def fp32_ball(xyz, q, r):
    """mask of the ball by the reference's predicate: fl(d2) <= fl(r * r), d2 without FMA"""
    d = xyz - q[None, :]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    return d2 <= np.float32(r) * np.float32(r)


def bruteforce_ball_normals(xyz, queries, r, radii=None):
    """numpy brute force: the ball by the fp32 predicate, fp64 mean and numpy.linalg.eigh.
    Returns (normals, centroids, gaps, counts); gap = (l1 - l0) / l2 as the oracle's."""
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    q = np.ascontiguousarray(queries, np.float32).reshape(-1, 3)
    nq = len(q)
    nrm = np.tile(np.array([0, 0, 1], np.float64), (nq, 1))
    ctr = np.full((nq, 3), np.nan)
    gap = np.zeros(nq)
    cnt = np.zeros(nq, np.uint32)
    for i in range(nq):
        rr = np.float32(r if radii is None else radii[i])
        p = xyz[fp32_ball(xyz, q[i], rr)].astype(np.float64)
        cnt[i] = len(p)
        if len(p) == 0:
            continue
        mu = p.mean(0)
        ctr[i] = mu
        c = p - mu
        w, v = np.linalg.eigh(c.T @ c)
        nrm[i] = v[:, 0]
        gap[i] = (w[1] - w[0]) / max(w[2], 1e-300)
    return nrm, ctr, gap, cnt


def normal_error(a, b):
    """1 - |cos| between rows of two normal arrays"""
    return 1.0 - np.abs((np.asarray(a, np.float64) * np.asarray(b, np.float64)).sum(1))


def centroid_tolerance(xyz):
    return 1e-5 * max(1.0, float(np.abs(xyz).max()))
