#!/usr/bin/env python
"""bench.py — the hot path's headline metric on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], the one the metric is quoted on): k = 15 normal estimation
over a 10 M-point synthetic noisy plane (x, y ~ U[0, 10), z = 1e-3 N(0,1), seed 7).  ONE STEP =
the whole path over one cloud: build the spatial index on the device (bbox -> Morton -> radix
sort -> cell tables) + the fused kNN -> PCA normal kernel over all of its points.

  value   normals/s with the cloud already resident in HBM (device pointers in, normals left in
          HBM), whole job over all ranks, bracketed by barrier + synchronize, max over ranks.
  e2e     the same step through the public C ABI with HOST buffers: pinned xyz in (H2D inside
          the timed region), host normals out (D2H inside).  Clouds are processed as a stream:
          --e2e-threads host threads (default 4) each run whole blocking calls on their own
          index, so one cloud's copies overlap another's kernels; `e2e_serial` (extra key) is the
          same with one thread.
  roofline  the dominant kernel (the tile kNN -> normal kernel): algorithmic bytes (SURVEY.md §8d
          gather model: 12 + 12 k + 12 = 204 B per normal at k = 15) / its CUDA-event duration on
          the library's launching stream, against the measured HBM peak in MEASURED_PEAKS.json.
          `traffic` is the DRAM bytes of one launch from the committed ncu capture
          (profiles/normals_kernel_traffic.json), reported only while the kernel sources still
          hash to what was captured.
  cpu_baseline  the reference's own octree (oracle/_ref, unmodified headers) + the restated
          estimate_normal, on this box's host cores, on a bounded sample (rank 0, N = 1 only).
  extras  (extra keys, kernel times by CUDA events, each with units_per_s / kernel_ms / frac of
          its own gather-model roofline): knn_k15, radius_r0.01, build on the same 10 M plane;
          density_filter_mix (10 M points, 5 % uniform noise); knn_k8_sphere_10M — N = 1 only.
          For every N: scan100M_k30 (configs[3]: k = 30 normals over a 100 M-point scan cut into
          N slabs) and, for N > 1, strong (the ONE 10 M-point plane cut into N slabs) and
          replicated (the same plane through ONE C-ABI handle replicated on all N devices,
          pcpx_index_params.devices, driven by rank 0).

N > 1 ("weak" headline): every rank owns one 10 M-point slab of an N x 10 M-point plane plus a
0.05-wide halo of its neighbours' points; the halo strips are exchanged between neighbouring
ranks over NCCL inside every timed step (point-cloud-processing_b200/sharding.py:
exchange_halo) — the one real exchange of the sharded path; value = N x 10 M normals /
max-over-ranks time.

--impl reference: times the reference's CPU implementation of the same step (full-size octree
build + a bounded query sample, extrapolated linearly) on all host threads; rank 0 only.

--dump-outputs DIR: after the run, every rank saves the normals its last timed headline step
returned for the points it owns (halo rows left out), float32, rows in the order of its own
seeded slab: DIR/normals.npy on one GPU, DIR/normals_rank<r>.npy on N > 1.  Above
DUMP_ROWS / N owned points a rank keeps a fixed-seed sample of that many rows
(np.random.default_rng(0), sorted), so two builds of the library can be compared output for
output on identical inputs.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (which may be read-only)

N_POINTS = 10_000_000
K = 15
HALO = 0.05
ALGORITHMIC_BYTES_PER_NORMAL = 12 + 12 * K + 12  # SURVEY.md §8d: query + k winners + normal out
METRIC = "normals/sec (estimate_normals k=15, 10M-pt noisy plane; index build + fused kNN->PCA per step)"
DUMP_ROWS = 4_000_000  # 48 MB of float32 normals over all ranks: a dump stays under 64 MB


def dump_outputs(path, normals, max_rows):
    """Save `normals` (an (n, 3) CUDA tensor) as `path`: every row when n <= max_rows, else a
    sorted fixed-seed sample of max_rows rows."""
    import torch

    n = normals.shape[0]
    if n <= max_rows:
        sample = normals
    else:
        rows = np.sort(np.random.default_rng(0).choice(n, max_rows, replace=False))
        sample = normals[torch.from_numpy(rows).to(normals.device)]
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    np.save(path, sample.cpu().numpy().astype(np.float32))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def csrc_hash():
    """hash of the kernel sources (same recipe as tools/update_traffic.py)"""
    import hashlib

    d = os.path.join(ROOT, "point-cloud-processing_b200", "csrc")
    h = hashlib.sha256()
    for f in sorted(os.listdir(d)):
        p = os.path.join(d, f)
        if os.path.isfile(p) and f.endswith((".cu", ".cuh", ".hpp", ".inc")):
            h.update(f.encode())
            h.update(open(p, "rb").read())
    return h.hexdigest()[:16]


def recorded_traffic():
    """DRAM bytes of one launch of the dominant kernel from the committed ncu capture — only
    when the capture was taken from the kernel sources that are in the tree now.  Returns
    (bytes or None, provenance string)."""
    p = os.path.join(ROOT, "profiles", "normals_kernel_traffic.json")
    if not os.path.exists(p):
        return None, "no capture committed"
    try:
        rec = json.load(open(p))
        src = "%s, commit %s, %s" % (rec.get("source"), rec.get("commit"), rec.get("captured_at"))
        if rec.get("csrc_sha16") != csrc_hash():
            return None, "STALE capture (kernel sources changed since): " + src
        return float(rec["dram_bytes_per_launch"]), src
    except Exception as e:  # noqa: BLE001
        return None, "unreadable capture: %r" % (e,)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region: one long-running
    `nvidia-smi -lms 50` whose lines are collected while the context is open."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None
        self.t = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) >= 9:
                self.samples.append(f)

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.3)  # let the first samples arrive before the load starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            if self.t is not None:
                self.t.join(timeout=5)

    def summary(self):
        def num(x):
            try:
                return float(x)
            except ValueError:
                return None

        sm = [num(s[1]) for s in self.samples if num(s[1]) is not None]
        mx = [num(s[2]) for s in self.samples if num(s[2]) is not None]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for name, v in zip(names, s[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def bind_to_gpu_numa_node(local_rank):
    """Best effort: run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA
    node its GPU hangs off, so that N ranks do not all stage through one socket."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=10)
        bus = q.stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = "0000:" + bus[9:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def own_slab(pcpx, rank):
    """this rank's 10 M-point slab of the world x 10 M plane: x in [rank L, (rank + 1) L)"""
    L = pcpx.synth.plane_extent(N_POINTS)
    pts = pcpx.synth.noisy_plane(N_POINTS, seed=7 + rank, extent=L)
    pts[:, 0] += np.float32(rank * L)
    return pts, L


# ------------------------------------------------------------------------------------------
def cpu_reference_step(xyz, k, sample_size, seed=123):
    """The reference's CPU path for one step: full-size octree build (single thread: the
    insertion cannot be parallelised) + estimate_normals' body on a fixed-seed sample over all
    host threads, extrapolated linearly to the whole cloud."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    threads = max(1, os.cpu_count() or 1)
    rng = np.random.default_rng(seed)
    sample = np.sort(rng.choice(len(xyz), size=min(sample_size, len(xyz)), replace=False))
    if oracle_lib.have_ref():
        kind = "reference"
        ref = oracle_lib.RefBridge()
        t0 = time.perf_counter()
        cloud = ref.cloud(xyz, which=0)
        t_build = time.perf_counter() - t0
        t0 = time.perf_counter()
        cloud.normals_sample(0, sample.astype(np.uint32), k, nthreads=threads)
        t_query = time.perf_counter() - t0
    else:
        kind = "port"
        orc = oracle_lib.Oracle()
        t0 = time.perf_counter()
        cloud = orc.cloud(xyz)
        t_build = time.perf_counter() - t0
        t0 = time.perf_counter()
        cloud.normals(xyz[sample], k, nthreads=threads)
        t_query = time.perf_counter() - t0
    t_full = t_build + t_query * (len(xyz) / len(sample))
    desc = ("octree build over all %d points (1 thread, %.2f s) + estimate_normals body on a "
            "fixed-seed sample of %d points (%d threads, %.2f s), extrapolated linearly"
            % (len(xyz), t_build, len(sample), threads, t_query))
    return {"value": len(xyz) / t_full, "unit": "normals/s", "cores": threads, "kind": kind,
            "sample": desc, "build_s": t_build, "query_sample_s": t_query}


def headline_config(world, n_local, numa_node):
    """`config` of the JSON line — the same object for both arms (the reference arm runs this
    workload's one-GPU share on the host cores)."""
    return {
        "workload": "estimate_normals k=15 over a 10M-point noisy plane per GPU (seed 7+rank, "
                    "L=10, sigma_z=1e-3): device index build + fused kNN->PCA normal kernel",
        "n_points_per_gpu": N_POINTS, "k": K, "halo": HALO if world > 1 else 0.0,
        "local_points": n_local,
        "cache": "inputs larger than L2 (160 MB sorted float4 SoA + cell table vs 126 MB "
                 "L2); the index is rebuilt from scratch every step",
        "parallelism": "one process per GPU, spatial slabs; halo strips exchanged with the neighbouring ranks over NCCL (isend/irecv) inside the timed step",
        "numa_node_rank0": numa_node,
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    pcpx = importlib.import_module("point-cloud-processing_b200")
    xyz = pcpx.synth.noisy_plane(N_POINTS)
    times, last = [], None
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        last = cpu_reference_step(xyz, K, args.ref_sample)
        if it >= args.warmup:
            times.append(N_POINTS / last["value"])
    t = float(np.mean(times))
    value = N_POINTS / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "normals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the repo arm's config (same workload: rank 0's 10 M-point cloud, k = 15), answered by
        # the reference's own CPU path: octree build + kNN + PCA normal
        "config": headline_config(max(1, args.gpus), N_POINTS, None),
        "cpu_baseline": {k_: last[k_] for k_ in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": value, "unit": "normals/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    line["cpu_baseline"]["value"] = value
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------
def _timed(fn, steps, warmup, barrier, world, dist, torch):
    """K timed calls of fn bracketed by barrier + synchronize; max over ranks (seconds)"""
    for _ in range(warmup):
        fn()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    barrier()
    return dt


class ShardedCloud:
    """One rank's slab of a cloud cut along x, resident in HBM, with room behind it for the
    neighbours' halo strips; local() runs the exchange step and returns the local cloud."""

    def __init__(self, pcpx, torch, dist, pts, slab_lo, slab_hi, halo, rank, world):
        self.pcpx, self.torch, self.dist = pcpx, torch, dist
        self.rank, self.world, self.halo = rank, world, halo
        self.lo, self.hi = float(slab_lo), float(slab_hi)
        self.n_owned = len(pts)
        self.h_xyz = torch.from_numpy(pts).pin_memory()
        extent = max(self.hi - self.lo, 1e-9)
        # strips hold about n * halo / extent points; twice that (+ slack) is the capacity
        cap = 0 if world == 1 else int(2 * self.n_owned * halo / extent) + 65536
        self.buf = torch.empty((self.n_owned + 2 * cap, 3), dtype=torch.float32, device="cuda")
        self.own = self.buf[: self.n_owned]
        self.own.copy_(self.h_xyz)
        self.scratch = pcpx.sharding.HaloScratch(cap, "cuda") if world > 1 else None

    def local(self):
        if self.world == 1:
            return self.own
        return self.pcpx.sharding.exchange_halo(self.own, 0, self.lo, self.hi, self.halo,
                                                self.rank, self.world, self.dist, buffer=self.buf,
                                                scratch=self.scratch)[0]


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world,
                                device_id=torch.device("cuda", local_rank))
    pcpx = importlib.import_module("point-cloud-processing_b200")
    pcpx.lib()  # fail loudly now if the CUDA library is missing
    peak, peak_src = measured_peak_gbs()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # a host-side barrier (gloo): ranks waiting in it leave their GPU idle — an NCCL barrier is a
    # kernel that spins on the device, which would compete with rank 0's replicas on those GPUs
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None

    def host_barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---------------- the headline: weak, 10 M-point plane per rank --------------------------
    xyz, L = own_slab(pcpx, rank)
    cloud = ShardedCloud(pcpx, torch, dist, xyz, rank * L, (rank + 1) * L, HALO, rank, world)
    n_owned = cloud.n_owned
    n_local = int(cloud.local().shape[0])
    d_nrm = torch.empty((n_local + 65536, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()

    stats = {k_: [] for k_ in ("build_ms", "sort_ms", "kernel_ms", "launches", "retries")}

    def step_resident(cl=cloud, k=K, st=stats, out=d_nrm):
        d_xyz = cl.local()
        torch.cuda.synchronize()  # the library runs on its own stream
        ix = pcpx.Index(d_xyz, device=local_rank)
        tb = ix.timings()
        ix.estimate_normals(None, k, out=out[: ix.n])
        tq = ix.timings()
        ix.close()
        if st is not None:
            st["build_ms"].append(tb["build_ms"])
            st["sort_ms"].append(tb["sort_ms"])
            st["kernel_ms"].append(tq["kernel_ms"])
            st["launches"].append(tb["kernel_launches"] + tq["kernel_launches"])
            st["retries"].append(tq["retry_queries"])

    # end to end: pinned host buffers in and out.  N = 1: whole blocking C-ABI calls with HOST
    # pointers from T host threads (one cloud's copies overlap another's kernels).  N > 1: the
    # halo exchange is a collective step every rank must issue in the same order, so one thread
    # per rank pipelines the stream of clouds itself: the H2D of cloud i + 1 and the D2H of cloud
    # i - 1 run on side streams while cloud i is exchanged, indexed and answered (C-ABI calls
    # with device pointers); every cloud's 120 MB in and 120 MB out are inside the timed region.
    n_thr = max(1, args.e2e_threads)
    n_buf = n_thr if world == 1 else 2
    h_out = [torch.empty((n_local + 65536, 3), dtype=torch.float32).pin_memory() for _ in range(n_buf)]
    d_stage = d_res = None
    if world > 1:
        d_stage = [ShardedCloud(pcpx, torch, dist, xyz, rank * L, (rank + 1) * L, HALO, rank, world)
                   for _ in range(2)]
        d_res = [torch.empty((n_local + 65536, 3), dtype=torch.float32, device="cuda") for _ in range(2)]
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]

    def e2e_once(t):
        ix = pcpx.Index(cloud.h_xyz.numpy(), device=local_rank)  # host pointer: H2D inside
        ix.estimate_normals(None, K, out=h_out[t].numpy()[: ix.n])  # host pointer: D2H inside
        ix.close()

    def e2e_pipelined(total_steps, overlap=True):
        cur = torch.cuda.current_stream()

        def upload(b):
            with torch.cuda.stream(s_in):
                d_stage[b].own.copy_(cloud.h_xyz, non_blocking=True)
                ev_in[b].record(s_in)

        upload(0)
        for i in range(total_steps):
            b = i & 1
            if overlap and i + 1 < total_steps:
                upload(1 - b)  # (the step that last used this buffer has returned: calls block)
            ev_in[b].synchronize()
            d_xyz = d_stage[b].local()  # strip cut + NCCL exchange on the current stream
            cur.synchronize()
            if i >= 2:
                ev_out[b].synchronize()  # the copy that read d_res[b] two clouds ago is done
            ix = pcpx.Index(d_xyz, device=local_rank)
            ix.estimate_normals(None, K, out=d_res[b][: ix.n])
            nloc = ix.n
            ix.close()
            with torch.cuda.stream(s_out):
                h_out[b][:nloc].copy_(d_res[b][:nloc], non_blocking=True)
                ev_out[b].record(s_out)
            if not overlap:
                ev_out[b].synchronize()
                if i + 1 < total_steps:
                    upload(1 - b)
        torch.cuda.synchronize()

    def e2e_run(total_steps, threads):
        if world > 1:
            e2e_pipelined(total_steps, overlap=threads > 1)
            return
        if threads == 1:
            for _ in range(total_steps):
                e2e_once(0)
            return
        per = [total_steps // threads + (1 if i < total_steps % threads else 0) for i in range(threads)]
        errs = []

        def work(t):
            try:
                torch.cuda.set_device(local_rank)
                for _ in range(per[t]):
                    e2e_once(t)
            except Exception as e:  # noqa: BLE001
                errs.append(e)

        th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        if errs:
            raise errs[0]

    with ClockSampler(local_rank) as clocks:
        dt_res = _timed(step_resident, args.steps, args.warmup, barrier, world, dist, torch)
        del stats["build_ms"][: args.warmup], stats["sort_ms"][: args.warmup]
        del stats["kernel_ms"][: args.warmup], stats["retries"][: args.warmup]
        del stats["launches"][: args.warmup]
        e2e_steps = max(args.steps, 3 * n_thr)  # (every host thread gets a few clouds)
        # three timed repetitions of the whole stream, the median reported: one repetition is
        # ~40 ms of wall time, and a single cudaMalloc that lands inside it (the device pool's
        # best-fit choice depends on thread timing) would be a 3x outlier
        e2e_reps = [_timed(lambda: e2e_run(e2e_steps, n_thr if world == 1 else 2), 1, 1 if i == 0 else 0,
                           barrier, world, dist, torch) for i in range(3)]
        dt_e2e = float(np.median(e2e_reps))
        dt_e2e_serial = _timed(lambda: e2e_run(max(2, args.steps // 2), 1), 1, 0, barrier, world,
                               dist, torch)
    total_owned = n_owned * world
    value = total_owned * args.steps / dt_res
    e2e_value = total_owned * e2e_steps / dt_e2e
    e2e_serial_value = total_owned * max(2, args.steps // 2) / dt_e2e_serial

    kernel_ms = allmax(float(np.mean(stats["kernel_ms"])))
    traffic, traffic_src = recorded_traffic()
    achieved = ALGORITHMIC_BYTES_PER_NORMAL * n_local / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "tile_knn2_kernel<16, MODE_NORMALS, S=2, 96 threads> (+ tile list, + the "
                          "warp-per-query kernel for what the tile pass hands on)",
                "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": ALGORITHMIC_BYTES_PER_NORMAL * n_local,
                "peak_source": peak_src,
                "note": "gather-model bytes (12 + 12k + 12 per normal, SURVEY.md 8d); kernel_ms "
                        "is the CUDA-event time of everything the normals call launches"}

    # untimed: the halo is wide enough iff every owned point near an inner slab face has its k
    # nearest neighbours inside the local cloud, i.e. at least k + 1 local points (itself
    # included) within its distance to the outer face of the halo
    def halo_check(cl, own, lo, hi, k):
        if world == 1:
            return True
        d_xyz = cl.local()
        torch.cuda.synchronize()
        gap = np.full(len(own), np.inf, np.float32)
        if rank > 0:
            gap = np.minimum(gap, own[:, 0] - np.float32(lo - cl.halo))
        if rank < world - 1:
            gap = np.minimum(gap, np.float32(hi + cl.halo) - own[:, 0])
        near = np.flatnonzero(gap < 4 * cl.halo)
        ok = True
        if len(near):
            with pcpx.Index(d_xyz, device=local_rank) as ix:
                cnt = ix.radius_count(own[near], 0.0, radii=(gap[near] * np.float32(0.999)))
            ok = bool((cnt >= k + 1).all())
        t = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    halo_ok = halo_check(cloud, xyz, rank * L, (rank + 1) * L, K)

    # ---------------- extra legs ---------------------------------------------------------------
    extras = {}
    leg_steps, leg_warm = max(3, args.steps // 2), 2

    def kernel_leg(fn, ix, reps=5):
        ms = []
        for _ in range(reps):
            fn()
            ms.append(ix.timings()["kernel_ms"])
        return float(np.median(ms[1:])), float(min(ms[1:]))

    def frac_of(bytes_per_unit, units, ms):
        return bytes_per_unit * units / (ms * 1e-3) / 1e9 / peak

    if world == 1 and not args.no_extras:
        n = n_owned
        d_idx = torch.empty((n, K), dtype=torch.int32, device="cuda")
        d_d2 = torch.empty((n, K), dtype=torch.float32, device="cuda")
        d_cnt = torch.empty((n,), dtype=torch.int32, device="cuda")
        with pcpx.Index(cloud.own, device=local_rank) as ix:
            info = ix.info()
            med, best = kernel_leg(lambda: ix.knn(None, K, out_idx=d_idx, out_d2=d_d2,
                                                  out_count=d_cnt), ix)
            extras["knn_k15"] = {
                "workload": "batched kNN k=15 (indices + distances + counts) over the 10M-point plane, "
                            "queries = the cloud, index resident",
                "units_per_s": n / (med * 1e-3), "unit": "queries/s", "kernel_ms": med,
                "best_ms": best, "bytes_per_unit": 12 + 12 * K + 4 * K + 4 * K,
                "frac": frac_of(12 + 12 * K + 4 * K + 4 * K, n, med)}
            med, best = kernel_leg(lambda: ix.radius_count(None, 0.01, out_count=d_cnt), ix)
            mbar = float(d_cnt.to(torch.float64).mean().item())
            extras["radius_r0.01"] = {
                "workload": "radius count r=0.01 over the 10M-point plane, queries = the cloud",
                "units_per_s": n / (med * 1e-3), "unit": "queries/s", "kernel_ms": med,
                "best_ms": best, "mean_count": mbar, "bytes_per_unit": 12 + 12 * mbar + 4,
                "frac": frac_of(12 + 12 * mbar + 4, n, med)}
        build_ms = float(np.mean(stats["build_ms"]))
        bpp = 136 if info["code_bits"] <= 30 else 276
        extras["build"] = {
            "workload": "index build of the 10M-point plane (%d-bit codes), as inside every step" % info["code_bits"],
            "units_per_s": n / (build_ms * 1e-3), "unit": "points/s", "kernel_ms": build_ms,
            "sort_ms": float(np.mean(stats["sort_ms"])), "bytes_per_unit": bpp,
            "frac": frac_of(bpp, n, build_ms)}
        del d_idx, d_d2
        # configs[2]: density filter on 10 M points with 5 % uniform noise
        mix = torch.from_numpy(pcpx.synth.noise_mix(N_POINTS)).cuda()
        d_mask = torch.empty((N_POINTS,), dtype=torch.uint8, device="cuda")
        d_keep = torch.empty((N_POINTS, 3), dtype=torch.float32, device="cuda")
        with pcpx.Index(mix, device=local_rank) as ix:
            ix.mean_knn_distance(K)  # (first use: kernel module load, tile list)
            radius = float(ix.mean_knn_distance(K)[1])
            mean_ms = ix.timings()["kernel_ms"]
            mean_t = ix.timings()
            kept = [0]

            def flt():
                kept[0] = ix.density_filter(radius, 5, out_mask=d_mask, out_xyz=d_keep)[2]

            med, best = kernel_leg(flt, ix)
            ix.radius_count(None, radius, out_count=d_cnt)
            mbar = float(d_cnt.to(torch.float64).mean().item())
            a_flt = 12 + 12 * mbar + 1 + 12 * kept[0] / N_POINTS
            extras["density_filter_mix"] = {
                "workload": "density filter (radius = mean 15-NN distance, threshold 5) on 10M points with 5% uniform noise",
                "units_per_s": N_POINTS / (med * 1e-3), "unit": "points/s", "kernel_ms": med,
                "best_ms": best, "radius": radius, "mean_count": mbar, "kept": int(kept[0]),
                "mean_knn_distance_kernel_ms": mean_ms,
                "mean_knn_distance_handed_on": int(mean_t["deferred_queries"]),
                "bytes_per_unit": a_flt,
                "frac": frac_of(a_flt, N_POINTS, med)}
        del mix, d_mask, d_keep
        # configs[4], one point of the sweep: kNN k=8 over a 10 M-point noisy sphere
        sph = torch.from_numpy(pcpx.synth.noisy_sphere(N_POINTS)).cuda()
        d_idx8 = torch.empty((N_POINTS, 8), dtype=torch.int32, device="cuda")
        with pcpx.Index(sph, device=local_rank) as ix:
            sb = ix.info()["build_ms"]
            med, best = kernel_leg(lambda: ix.knn(None, 8, out_idx=d_idx8, out_d2=None,
                                                  out_count=d_cnt, want_d2=False), ix)
            extras["knn_k8_sphere_10M"] = {
                "workload": "kNN k=8 (indices + counts) over a 10M-point noisy sphere (sigma 0.005), queries = the cloud",
                "units_per_s": N_POINTS / (med * 1e-3), "unit": "queries/s", "kernel_ms": med,
                "best_ms": best, "build_ms": sb, "bytes_per_unit": 12 + 12 * 8 + 4 * 8,
                "frac": frac_of(12 + 12 * 8 + 4 * 8, N_POINTS, med)}
        del sph, d_idx8, d_cnt
        torch.cuda.empty_cache()

    def sharded_leg(pts, lo, hi, k, bytes_per_unit, what):
        cl = ShardedCloud(pcpx, torch, dist, pts, lo, hi, HALO, rank, world)
        nl = int(cl.local().shape[0])
        out = torch.empty((nl + 65536, 3), dtype=torch.float32, device="cuda")
        st = {k_: [] for k_ in ("build_ms", "sort_ms", "kernel_ms", "launches", "retries")}
        dt = _timed(lambda: step_resident(cl, k, st, out), leg_steps, leg_warm, barrier, world,
                    dist, torch)
        total = allsum(cl.n_owned)
        kms = allmax(float(np.mean(st["kernel_ms"][leg_warm:])))
        ok = halo_check(cl, pts, lo, hi, k)
        rec = {"workload": what, "units_per_s": total * leg_steps / dt, "unit": "normals/s",
               "total_points": int(total), "ms_per_step": dt / leg_steps * 1e3, "kernel_ms": kms,
               "build_ms": allmax(float(np.mean(st["build_ms"][leg_warm:]))),
               "bytes_per_unit": bytes_per_unit,
               "frac": bytes_per_unit * allmax(nl) / (kms * 1e-3) / 1e9 / peak,
               "halo_sufficient": ok, "n_gpus": world}
        del cl, out
        torch.cuda.empty_cache()
        return rec

    if not args.no_extras:
        if world > 1:
            # strong: the ONE seed-7 10 M-point plane, cut into `world` slabs along x
            full = pcpx.synth.noisy_plane(N_POINTS)
            edges = pcpx.sharding.slab_edges(0.0, L, world)
            own = np.ascontiguousarray(full[pcpx.sharding.owner_of(full[:, 0], edges) == rank])
            del full
            extras["strong"] = sharded_leg(
                own, edges[rank], edges[rank + 1], K, ALGORITHMIC_BYTES_PER_NORMAL,
                "strong scaling: estimate_normals k=15 over the ONE 10M-point noisy plane "
                "(seed 7) cut into %d slabs; index build + halo exchange + normals per step" % world)
        pts, side = pcpx.synth.scan_slab(100_000_000, rank / world, (rank + 1) / world)
        extras["scan100M_k30"] = sharded_leg(
            pts, side * rank / world, side * (rank + 1) / world, 30, 12 + 12 * 30 + 12,
            "estimate_normals k=30 over a 100M-point synthetic scan (height field + sphere), "
            "cut into %d slab(s) along x; index build + halo exchange + normals per step" % world)

    if not args.no_extras and world > 1:
        # replicated: ONE handle of the C ABI over all N devices (pcpx_index_params.devices): the
        # index of the seed-7 10 M-point plane is built on every device, the normals call is
        # sharded by tile range, device 0 gathers the replicas' answers over NVLink.  Rank 0 drives it from
        # one process while the other ranks wait; timed by the host around the blocking calls.
        host_barrier()
        if rank == 0:
            full = torch.from_numpy(pcpx.synth.noisy_plane(N_POINTS)).cuda()
            out1 = torch.empty((N_POINTS, 3), dtype=torch.float32, device="cuda")
            outn = torch.empty((N_POINTS, 3), dtype=torch.float32, device="cuda")
            with pcpx.Index(full, device=local_rank) as ix1:
                ix1.estimate_normals(None, K, out=out1)
            devs = [local_rank] + [d for d in range(world) if d != local_rank]
            t0 = time.perf_counter()
            ixn = pcpx.Index(full, devices=devs)
            first_build = (time.perf_counter() - t0) * 1e3
            ixn.close()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ixn = pcpx.Index(full, devices=devs)
            build_wall = (time.perf_counter() - t0) * 1e3
            wall, kern = [], []
            for _ in range(leg_steps + leg_warm):
                t0 = time.perf_counter()
                ixn.estimate_normals(None, K, out=outn)
                wall.append((time.perf_counter() - t0) * 1e3)
                kern.append(ixn.timings()["kernel_ms"])
            ixn.close()
            w = float(np.median(wall[leg_warm:]))
            extras["replicated"] = {
                "workload": "estimate_normals k=15 over the ONE 10M-point noisy plane through one C-ABI "
                            "handle replicated on %d devices (index resident, call sharded by tile "
                            "range, replicas answer into local buffers that device 0 gathers over NVLink); host-timed "
                            "blocking call" % world,
                "units_per_s": N_POINTS / (w * 1e-3), "unit": "normals/s", "call_ms": w,
                "kernel_ms_slowest_device": float(np.median(kern[leg_warm:])),
                "build_wall_ms": build_wall, "first_build_wall_ms": first_build,
                "equal_to_one_device": bool(torch.equal(out1, outn)), "n_gpus": world}
            del full, out1, outn
            torch.cuda.empty_cache()
        host_barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_step(xyz, K, args.ref_sample)
        cpu = {k_: cpu[k_] for k_ in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "normals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt_res / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": headline_config(world, n_local, numa_node),
            "e2e": {"value": e2e_value, "unit": "normals/s",
                    "h2d_bytes_per_step": int(n_owned * 12), "d2h_bytes_per_step": int(n_local * 12),
                    "ms_per_step": dt_e2e / e2e_steps * 1e3, "steps": e2e_steps,
                    "repetitions_ms_per_step": [t / e2e_steps * 1e3 for t in e2e_reps],
                    "host_threads": n_thr if world == 1 else 1,
                    "mode": ("%d host threads, each whole blocking C-ABI calls with host pointers" % n_thr)
                    if world == 1 else
                    "one thread per rank; H2D of the next cloud and D2H of the previous one on side "
                    "streams while the current one is exchanged, indexed and answered"},
            "e2e_serial": {"value": e2e_serial_value, "unit": "normals/s",
                           "ms_per_step": dt_e2e_serial / max(2, args.steps // 2) * 1e3},
            "gpu_launches": int(np.sum(stats["launches"])),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "clocks": clocks.summary(),
            "breakdown_ms": {"build": float(np.mean(stats["build_ms"])),
                             "sort": float(np.mean(stats["sort_ms"])),
                             "normals_kernel": float(np.mean(stats["kernel_ms"]))},
            "exact_fallback_queries_per_step": float(np.mean(stats["retries"])),
            "halo_sufficient": halo_ok,
        }
        line.update(extras)
        print(json.dumps(line))
    if args.dump_outputs:
        # d_nrm is untouched since the last timed step; its first n_owned rows are this rank's
        # own points (the halo strips sit behind them)
        name = "normals.npy" if world == 1 else "normals_rank%d.npy" % rank
        dump_outputs(os.path.join(args.dump_outputs, name), d_nrm[:n_owned], DUMP_ROWS // world)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-sample", type=int, default=100_000,
                    help="queries in the CPU reference's bounded sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra legs (knn, radius, filter, sweep point, strong, scan100M)")
    ap.add_argument("--e2e-threads", type=int, default=4,
                    help="host threads streaming clouds through the C ABI in the e2e leg (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="save the normals of the last timed step as DIR/normals.npy, one file "
                         "per rank on N > 1 (a fixed-seed sample of %d rows over all ranks above "
                         "that size)" % DUMP_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs saves what the GPU path computed: it needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
