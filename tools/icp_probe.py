"""Measurement of rigid registration (pcpx_icp, pcpx_nearest_within) on one GPU, in one command:

    python tools/icp_probe.py [--out profiles/icp_probe.json] [--calls 5]

Target: synth.scan(10 M) with its estimate_normals(None, 15) normals.  Sources: the target moved
by 3 degrees and 0.5 % of the extent, all 10 M points and every tenth point (1 M).  For each:
  * pcpx_icp point-to-plane, max_distance 2 % of the extent, exactly 10 updates (tolerances of
    1e-300: 0 selects the defaults) plus the final pass: the host clock per call and the library's device
    time; per correspondence pass the device time of each kernel group (torch.profiler with CUDA
    activities, a separate run): transform, query sort, fused walk + block sums, final reduction;
  * pcpx_nearest_within against pcpx_knn(k = 1) over the same (moved) queries: device time of the
    kernels, of the query sort, and the host clock, on the same index;
  * the host loop the call replaces: per iteration knn(k = 1) into host memory, then the gather of
    target points and normals and the fp64 normal equations and solve in numpy, host clock.
The card's name, power limit and clock are read in the same run.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
pcpx = importlib.import_module("point-cloud-processing_b200")
from emu_icp_lib import np_solve, np_update, rigid, transform_f32  # noqa: E402

F32 = np.float32


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
    wall, dev, srt, ker = [], [], [], []
    for _ in range(calls):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
        t = ix.timings()
        dev.append(t["total_ms"]), srt.append(t["query_sort_ms"]), ker.append(t["kernel_ms"])
    return {"host_ms_median": float(np.median(wall)), "host_ms_min": float(np.min(wall)),
            "device_total_ms_median": float(np.median(dev)),
            "device_kernel_ms_median": float(np.median(ker)),
            "query_sort_ms_median": float(np.median(srt)),
            "kernel_launches": ix.timings()["kernel_launches"]}


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


def pass_groups(per_kernel, n_passes):
    """per-pass device time of transform, query sort, fused kernel and reduction; the copies and
    memsets (staging of the source and the normals, once per call) are listed per call apart"""
    groups = {"transform": 0.0, "sort": 0.0, "fused_walk_and_block_sums": 0.0,
              "final_reduction": 0.0, "copies_and_memsets_per_call": 0.0}
    for kname, ms in per_kernel.items():
        if kname.startswith("Memcpy") or kname.startswith("Memset"):
            groups["copies_and_memsets_per_call"] += ms
            continue
        g = ("transform" if "icp_transform" in kname else
             "fused_walk_and_block_sums" if "icp_pass" in kname else
             "final_reduction" if "icp_final" in kname else "sort")
        groups[g] += ms / n_passes
    return groups


def host_loop(ix, target, normals, src, r, iterations, centre):
    """knn(k = 1) to host + numpy normal equations and solve, per iteration (host clock)"""
    T = np.eye(4)
    times = []
    for _ in range(iterations):
        t0 = time.perf_counter()
        y = transform_f32(src, T)
        idx, d2, _ = ix.knn(y, 1, eps=0.0)
        idx, d2 = idx[:, 0], d2[:, 0]
        ok = d2 <= F32(r) * F32(r)
        yy = y[ok].astype(np.float64) - centre
        q = target[idx[ok]].astype(np.float64) - centre
        n = normals[idx[ok]].astype(np.float64)
        J = np.concatenate([np.cross(yy, n), n], axis=1)
        res = ((yy - q) * n).sum(1)
        A, b = J.T @ J, J.T @ res
        s = np.concatenate([A[np.triu_indices(6)], b, [0.0, float(ok.sum())]])
        T = np_update(T, np_solve(0, s), centre)
        times.append((time.perf_counter() - t0) * 1e3)
    return {"ms_per_iteration_median": float(np.median(times)), "iterations": iterations}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "icp_probe.json"))
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()

    res = {"facts": gpu_facts(), "workloads": []}
    target = pcpx.synth.scan(10_000_000)
    lo, hi = target.min(0).astype(np.float64), target.max(0).astype(np.float64)
    ext = float(np.linalg.norm(hi - lo))
    M = rigid(3, [1, 2, 3], 0.005 * ext * np.array([1, -1, 0]))
    moved = transform_f32(target, M)
    r = 0.02 * ext
    n_passes = 11
    with pcpx.Index(target, device=0) as ix:
        normals = ix.estimate_normals(None, 15)
        centre = 0.5 * (ix.bbox()[0].astype(np.float64) + ix.bbox()[1].astype(np.float64))
        for name, src in (("source_1M", np.ascontiguousarray(moved[::10])),
                          ("source_10M", moved)):
            def icp():
                return ix.icp(src, r, normals, max_iterations=10, rotation_tolerance=1e-300,
                              translation_tolerance=1e-300)

            row = {"workload": name, "target": "synth.scan(10M)", "ns": len(src),
                   "max_distance": r, "passes_per_call": n_passes}
            row["icp_call"] = timed(ix, icp, args.warmup, args.calls)
            T, info = icp()
            row["icp_result"] = info
            k = per_kernel_ms(icp, 2)
            row["per_pass_device_ms"] = pass_groups(k, n_passes)
            row["per_kernel_ms_per_call"] = k
            q = transform_f32(src, np.linalg.inv(M) @ np.eye(4))
            row["nearest_within"] = timed(ix, lambda: ix.nearest_within(q, r), args.warmup,
                                          args.calls)
            row["knn_k1"] = timed(ix, lambda: ix.knn(q, 1, eps=0.0), args.warmup, args.calls)
            row["host_loop"] = host_loop(ix, target, normals, src, r, 3, centre)
            res["workloads"].append(row)
            print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
