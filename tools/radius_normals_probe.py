"""Measurement of the fused ball PCA (pcpx_estimate_normals_radius) on one GPU, in one command:

    python tools/radius_normals_probe.py [--out profiles/radius_normals_probe.json] [--n 1e7]

Workloads (10 M points): the noisy plane at r = 0.01 (about 32 points per ball) and at the
radius that gives about 250, the noise mix at r = 0.01, and the plane with per-query radii of
twice the mean 15-NN distance.  For each: the kernel time of the fused call (CUDA events around
the kernel, inside the library; warm-up first, then `--calls` calls, median and min) and its
normals/s; pcpx_radius_count on the same input, which is the same walk without the epilogue;
the three-call composition radius_search -> gather -> normals_from_neighbourhoods (host clock
around the whole chain, ending in a device synchronise) where the neighbour lists fit; and the
bytes of the gather model, 12 + 12 m + 12 per query (query in, m neighbours of 12 B, normal out).
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


def kernel_ms(ix, fn, warmup, calls):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(calls):
        fn()
        ms.append(ix.timings()["kernel_ms"])
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "calls": calls}


def composition_s(ix, d_xyz, radius, radii, reps):
    """radius_search (host CSR) -> gather of the neighbours' xyz on the device ->
    normals_from_neighbourhoods on device buffers: the route the library offered before"""
    import torch

    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        off, idx = ix.radius_search(None, radius, radii=radii)
        d_idx = torch.from_numpy(idx.astype(np.int64)).cuda()
        nbr = d_xyz.index_select(0, d_idx)
        del d_idx
        d_off = torch.from_numpy(off.view(np.int64)).cuda()
        out = torch.empty((len(off) - 1, 3), dtype=torch.float32, device="cuda")
        rc = pcpx.lib().pcpx_normals_from_neighbourhoods(nbr.data_ptr(), d_off.data_ptr(),
                                                         len(off) - 1, 0, out.data_ptr())
        assert rc == 0
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        del nbr, d_off
    return {"median_s": float(np.median(times)), "min_s": float(np.min(times)), "reps": reps,
            "normals": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "radius_normals_probe.json"))
    ap.add_argument("--n", type=float, default=1e7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--max-composition-neighbours", type=float, default=6e8)
    a = ap.parse_args()
    import torch

    if pcpx.device_count() < 1 or not torch.cuda.is_available():
        sys.exit("radius_normals_probe: no CUDA device (nothing here runs on the CPU)")
    n = int(a.n)
    out = dict(gpu_facts(), n=n, warmup=a.warmup, calls=a.calls, workloads=[])
    plane = pcpx.synth.noisy_plane(n)
    mix = pcpx.synth.noise_mix(n)
    with pcpx.Index(plane) as ix:
        per15, _ = ix.mean_knn_distance(15)
    cases = [("plane r=0.01", plane, 0.01, None),
             ("plane m~250", plane, float(np.float32(0.01 * np.sqrt(250 / 31.4))), None),
             ("noise mix r=0.01", mix, 0.01, None),
             ("plane radii = 2 x mean 15-NN distance", plane, 0.0, (2 * per15).astype(np.float32))]
    for name, xyz, radius, radii in cases:
        d_xyz = torch.from_numpy(xyz).cuda()
        d_radii = None if radii is None else torch.from_numpy(radii).cuda()
        d_nrm = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        d_cnt = torch.empty(n, dtype=torch.int32, device="cuda")
        with pcpx.Index(d_xyz) as ix:
            fused = kernel_ms(ix, lambda: ix.estimate_normals_radius(
                None, radius, radii=d_radii, out=d_nrm, out_count=d_cnt), a.warmup, a.calls)
            count = kernel_ms(ix, lambda: ix.radius_count(None, radius, radii=d_radii,
                                                          out_count=d_cnt), a.warmup, a.calls)
            m = float(d_cnt.double().mean().item())
            total = float(d_cnt.double().sum().item())
            row = {"workload": name, "radius": radius, "mean_ball": m,
                   "fused_kernel": fused,
                   "fused_normals_per_s": n / (fused["median_ms"] * 1e-3),
                   "radius_count_kernel": count,
                   "fused_over_count": fused["median_ms"] / count["median_ms"],
                   "gather_model_bytes": n * (12 + 12 * m + 12),
                   "gather_model_GBps_at_fused_time":
                       n * (12 + 12 * m + 12) / (fused["median_ms"] * 1e-3) / 1e9}
            # end to end of the fused call on device buffers, same host clock as the composition
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                ix.estimate_normals_radius(None, radius, radii=d_radii, out=d_nrm)
            torch.cuda.synchronize()
            row["fused_call_s"] = (time.perf_counter() - t0) / 3
            if total <= a.max_composition_neighbours:
                comp = composition_s(ix, d_xyz, radius, radii, 3)
                got = comp.pop("normals")
                cos = (got * d_nrm).sum(1).abs()
                row["composition"] = comp
                row["composition_over_fused_call"] = comp["median_s"] / row["fused_call_s"]
                # rows where the two routes' normals differ by more than 1 - |cos| = 1e-4
                # (ill-conditioned balls, if any: no eigengap filter here)
                row["composition_rows_differing_1e-4"] = int(((1 - cos) > 1e-4).sum().item())
            else:
                row["composition"] = "not run: %.3g neighbours (limit %.3g)" % (
                    total, a.max_composition_neighbours)
        out["workloads"].append(row)
        print(json.dumps(row), flush=True)
        del d_xyz, d_radii, d_nrm, d_cnt
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
