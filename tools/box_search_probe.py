"""Measurement of the box range search (pcpx_box_search) on one GPU, in one command:

    python tools/box_search_probe.py [--out profiles/box_search_probe.json] [--calls 20]

Workloads:
  * the reference benchmark's shape: 2^24 points of synth.uniform_cube(n, half=100) and 65 536
    cubes at random centres, with sides that hold about 32 and about 1000 points;
  * the 10 M-point noisy plane: 65 536 small boxes (about 40 points each), a slab 1 % of the
    cloud thick, a crop of half the cloud and a box over the whole cloud, each also sorted.
For each: the device time of the call (CUDA events inside the library from the count kernel to
the end of the fill / sort, median and min over `--calls` calls after warm-up), the whole call
(host clock around it, device boxes, device lists, ending in a synchronise), boxes/s and
results/s.  In the same run, the route the box overloads of pcp.hpp took before: pcpx_radius_search
over the circumscribed spheres with that route's slack, device time and its ratio to the box
call; skipped where one thread walks the whole cloud (slab, crop, whole cloud).  For the whole
cloud also a device-to-device copy of 4 B x n (cudaMemcpyAsync through torch), the floor of its
fill.
"""
import argparse
import ctypes as C
import importlib
import json
import os
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


def search(ix, d_boxes, nb, sorted_):
    """one pcpx_box_search with device boxes and device lists; returns the total"""
    off = np.zeros(nb + 1, np.uint64)
    p = C.c_void_p()
    rc = pcpx.lib().pcpx_box_search(ix._h, d_boxes.data_ptr(), nb, 24, off.ctypes.data,
                                    C.byref(p), 1 | (2 if sorted_ else 0))
    assert rc == 0, pcpx.lib().pcpx_last_error()
    pcpx.lib().pcpx_free(p, 1)
    return int(off[-1])


def spheres_search(ix, centres, radii):
    n = len(centres)
    off = np.zeros(n + 1, np.uint64)
    p = C.c_void_p()
    rc = pcpx.lib().pcpx_radius_search(ix._h, centres.data_ptr(), n, 12, radii.data_ptr(),
                                       C.c_float(0.0), off.ctypes.data, C.byref(p), 1)
    assert rc == 0, pcpx.lib().pcpx_last_error()
    pcpx.lib().pcpx_free(p, 1)
    return int(off[-1])


def circumscribed(boxes):
    """centre and radius of the route pcp.hpp used before (its slack formula)"""
    b = boxes.astype(np.float32)
    h = 0.5 * (b[:, 3:] - b[:, :3])
    c = b[:, :3] + h
    big = np.abs(b).max(1)
    r = np.sqrt((h * h).sum(1)) * np.float32(1.0001) + np.float32(8 * 1.1920929e-7) * big + np.float32(1e-30)
    return c.astype(np.float32), r.astype(np.float32)


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


def workload(ix, name, boxes, args, baseline=True):
    import torch

    nb = len(boxes)
    d_boxes = torch.from_numpy(np.ascontiguousarray(boxes, np.float32)).cuda()
    total = search(ix, d_boxes, nb, False)
    row = {"name": name, "boxes": nb, "results": total, "mean_per_box": total / nb}
    for sorted_ in (False, True):
        t = timed(ix, lambda: search(ix, d_boxes, nb, sorted_), args.warmup, args.calls)
        t["kernel_launches"] = ix.timings()["kernel_launches"]
        t["boxes_per_s"] = nb / (t["device_median_ms"] * 1e-3)
        t["results_per_s"] = total / (t["device_median_ms"] * 1e-3)
        row["sorted" if sorted_ else "unsorted"] = t
    cnt = torch.empty(nb, dtype=torch.int32, device="cuda")
    row["count_only"] = timed(ix, lambda: ix.box_count(d_boxes, out_count=cnt), args.warmup,
                              args.calls)
    if baseline:
        c, r = circumscribed(boxes)
        dc, dr = torch.from_numpy(c).cuda(), torch.from_numpy(r).cuda()
        sph_total = spheres_search(ix, dc, dr)
        t = timed(ix, lambda: spheres_search(ix, dc, dr), 1, max(3, args.calls // 4))
        t["results"] = sph_total
        t["ratio_to_box_call"] = t["device_median_ms"] / row["unsorted"]["device_median_ms"]
        row["circumscribed_sphere_baseline"] = t
    else:
        row["circumscribed_sphere_baseline"] = (
            "skipped: the sphere covers most of the cloud, and radius_level falls to level 0, "
            "where one thread walks the whole cloud")
    print(json.dumps({k: v for k, v in row.items() if k != "name"} | {"name": name}), flush=True)
    return row


def cubes(rng, nb, half, side):
    c = rng.uniform(-half, half, (nb, 3)).astype(np.float32)
    h = np.float32(side / 2)
    return np.concatenate([c - h, c + h], 1).astype(np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "box_search_probe.json"))
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch

    res = {"facts": gpu_facts(), "workloads": []}
    rng = np.random.default_rng(1)
    n = 1 << 24
    xyz = pcpx.synth.uniform_cube(n, half=100.0)
    with pcpx.Index(xyz) as ix:
        # side s holds n (s / 200)^3 points
        for m in (32, 1000):
            side = 200.0 * (m / n) ** (1 / 3)
            res["workloads"].append(workload(ix, "cube_2^24_65536_boxes_m%d" % m,
                                             cubes(rng, 65536, 100.0, side), args))
    del xyz
    n = 10_000_000
    xyz = pcpx.synth.noisy_plane(n)
    L = pcpx.synth.plane_extent(n)
    with pcpx.Index(xyz) as ix:
        c = np.concatenate([rng.uniform(0, L, (65536, 2)), np.zeros((65536, 1))], 1)
        small = np.concatenate([c - 0.01, c + 0.01], 1).astype(np.float32)
        res["workloads"].append(workload(ix, "plane_10M_65536_small_boxes", small, args))
        slab = np.array([[0.3 * L, -1, -1, 0.31 * L, L + 1, 1]], np.float32)
        res["workloads"].append(workload(ix, "plane_10M_slab_1pct", slab, args, baseline=False))
        half = np.array([[-1, -1, -1, 0.5 * L, L + 1, 1]], np.float32)
        res["workloads"].append(workload(ix, "plane_10M_half_crop", half, args, baseline=False))
        whole = np.array([[-np.inf] * 3 + [np.inf] * 3], np.float32)
        row = workload(ix, "plane_10M_whole_cloud", whole, args, baseline=False)
        src = torch.zeros(n, dtype=torch.int32, device="cuda")
        dst = torch.empty_like(src)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = []
        for i in range(args.warmup + args.calls):
            e0.record()
            dst.copy_(src)
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                ms.append(e0.elapsed_time(e1))
        row["d2d_copy_4B_x_n_median_ms"] = float(np.median(ms))
        row["unsorted_over_d2d"] = row["unsorted"]["device_median_ms"] / float(np.median(ms))
        res["workloads"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
