"""Measurement of density-based clustering (pcpx_cluster_by_density) on one GPU, in one command:

    python tools/cluster_probe.py [--out profiles/cluster_probe.json] [--calls 10]

Workloads, 10 M points each:
  * the noisy plane at r = 0.01, min_points 5: one giant component;
  * the 5 % noise mix at the density filter's radius (the mean 15-NN distance, as bench.py),
    min_points 5;
  * 10^4 separated Gaussian blobs of 1000 points (sigma 0.01, centres 1 apart), r = 0.005,
    min_points 5: many clusters.
For each: the device time of the call (CUDA events inside the library around its kernels,
median and min over `--calls` calls after warm-up), the host clock around the whole call with
device labels, the device time of each kernel (torch.profiler with CUDA activities, in a separate
run of the call), and the ratios to radius_count and to density_filter over the same balls,
timed the same way.  At 1 M points (the plane at the same density), also the host route the call
replaces: radius_search to host memory, then scipy's connected_components and the border rule in
numpy, timed on the host clock, with its labels checked against the call's.
"""
import argparse
import importlib
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pcpx = importlib.import_module("point-cloud-processing_b200")


def gpu_facts():
    import torch

    facts = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=60)
        facts["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        facts["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return facts


def timed(ix, fn, warmup, calls):
    import torch

    for _ in range(warmup):
        fn()
    dev, wall = [], []
    for _ in range(calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        wall.append(time.perf_counter() - t0)
        dev.append(ix.timings()["kernel_ms"])
    return {"device_median_ms": float(np.median(dev)), "device_min_ms": float(np.min(dev)),
            "call_median_ms": 1e3 * float(np.median(wall)), "calls": calls}


def per_kernel_ms(fn, calls):
    """mean device time per call of every kernel fn launches (torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile

    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            m = re.search(r"(\w+_kernel)", e.key)
            name = m.group(1) if m else e.key
            out[name] = out.get(name, 0.0) + t * 1e-3 / calls
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def workload(name, xyz, r, min_points, args):
    import torch

    n = len(xyz)
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    cnt = torch.empty(n, dtype=torch.int32, device="cuda")
    mask = torch.empty(n, dtype=torch.uint8, device="cuda")
    with pcpx.Index(torch.from_numpy(xyz).cuda()) as ix:
        if r is None:
            ix.mean_knn_distance(15)
            r = float(ix.mean_knn_distance(15)[1])
        _, nc = ix.cluster_by_density(r, min_points, out_labels=labels)
        lab = labels.cpu().numpy().view(np.uint32)
        noise = int((lab == pcpx.NOISE).sum())
        sizes = np.bincount(lab[lab != pcpx.NOISE]) if nc else np.zeros(1, np.int64)
        ix.radius_count(None, r, out_count=cnt)
        row = {"name": name, "points": n, "radius": r, "min_points": min_points,
               "mean_ball": float(cnt.double().mean().item()), "clusters": nc,
               "noise_points": noise, "largest_cluster": int(sizes.max())}
        t = timed(ix, lambda: ix.cluster_by_density(r, min_points, out_labels=labels),
                  args.warmup, args.calls)
        t["kernel_launches"] = ix.timings()["kernel_launches"]
        t["points_per_s"] = n / (t["device_median_ms"] * 1e-3)
        row["cluster_by_density"] = t
        row["radius_count"] = timed(ix, lambda: ix.radius_count(None, r, out_count=cnt),
                                    args.warmup, args.calls)
        row["density_filter"] = timed(
            ix, lambda: ix.density_filter(r, min_points, want_points=False, out_mask=mask),
            args.warmup, args.calls)
        dm = t["device_median_ms"]
        row["ratio_to_radius_count"] = dm / row["radius_count"]["device_median_ms"]
        row["ratio_to_density_filter"] = dm / row["density_filter"]["device_median_ms"]
        row["per_kernel_ms"] = per_kernel_ms(
            lambda: ix.cluster_by_density(r, min_points, out_labels=labels), args.calls)
    print(json.dumps({k: v for k, v in row.items() if k != "per_kernel_ms"}), flush=True)
    print(json.dumps(row["per_kernel_ms"]), flush=True)
    return row


def host_route(xyz, r, min_points, args):
    """radius_search to the host + scipy: what a caller did before this call"""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components

    n = len(xyz)
    walls = []
    with pcpx.Index(xyz) as ix:
        dev_labels, dev_nc = ix.cluster_by_density(r, min_points)
        dev = timed(ix, lambda: ix.cluster_by_density(r, min_points), 1, args.calls)
        for _ in range(3):
            t0 = time.perf_counter()
            off, idx = ix.radius_search(None, r)
            t1 = time.perf_counter()
            rows = np.repeat(np.arange(n, dtype=np.int32), np.diff(off).astype(np.int64))
            cols = idx.view(np.int32)
            core = np.diff(off) >= min_points
            keep = core[rows] & core[cols]
            g = csr_matrix((np.ones(int(keep.sum()), np.int8), (rows[keep], cols[keep])),
                           shape=(n, n))
            _, comp = connected_components(g, directed=False)
            labels = np.full(n, pcpx.NOISE, np.uint32)
            _, labels[core] = np.unique(comp[core], return_inverse=True)
            b = ~core[rows] & core[cols]
            bi, bj = rows[b], cols[b]
            d = xyz[bi] - xyz[bj]
            d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
            o = np.lexsort((bj, d2, bi))
            bi, bj = bi[o], bj[o]
            first = np.ones(len(bi), bool)
            first[1:] = bi[1:] != bi[:-1]
            labels[bi[first]] = labels[bj[first]]
            t2 = time.perf_counter()
            walls.append((t1 - t0, t2 - t1))
    same = bool(np.array_equal(labels, dev_labels))
    med = np.median(np.array(walls), axis=0)
    row = {"name": "host_route_plane_1M", "points": n, "radius": r, "min_points": min_points,
           "clusters": dev_nc, "labels_equal_to_call": same,
           "radius_search_to_host_median_s": float(med[0]),
           "scipy_components_and_border_median_s": float(med[1]),
           "host_route_median_s": float(med.sum()), "repeats": len(walls),
           "cluster_by_density_host_labels": dev,
           "host_route_over_call": float(med.sum()) / (dev["call_median_ms"] * 1e-3)}
    print(json.dumps(row), flush=True)
    assert same
    return row


def blobs(n_blobs, per_blob, sigma, seed=17):
    rng = np.random.default_rng(seed)
    side = int(np.ceil(n_blobs ** (1 / 3)))
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    centres = g[rng.permutation(len(g))[:n_blobs]].astype(np.float64)
    pts = np.repeat(centres, per_blob, 0) + sigma * rng.standard_normal((n_blobs * per_blob, 3))
    return np.ascontiguousarray(pts[rng.permutation(len(pts))].astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cluster_probe.json"))
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()

    res = {"facts": gpu_facts(), "workloads": []}
    n = 10_000_000
    res["workloads"].append(workload("plane_10M_r0.01_min5", pcpx.synth.noisy_plane(n), 0.01, 5,
                                     args))
    res["workloads"].append(workload("noise_mix_10M_density_radius_min5", pcpx.synth.noise_mix(n),
                                     None, 5, args))
    res["workloads"].append(workload("blobs_10M_1e4x1000_r0.005_min5", blobs(10_000, 1000, 0.01),
                                     0.005, 5, args))
    m = 1_000_000
    res["host_route"] = host_route(pcpx.synth.noisy_plane(m, extent=pcpx.synth.plane_extent(m)),
                                   0.01, 5, args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
