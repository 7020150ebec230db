#!/usr/bin/env python
"""bench.py — headline benchmark of the registration hot path (BASELINE.json metric: scans/sec,
100 k-pt 64-beam scan vs 10 M-pt map, full LIO iterate-to-converge).

One "step" = one pass of the per-scan LIO hot path (lsd_lio_scan): voxel-grid downsample (K1) ->
iterated ESKF update with fused k-NN + plane + residual/Jacobian + J^T J reduction per iteration
(K3-K5, host 23x23 algebra in double) -> map_incremental insert (K2).  Every step visits a
different 120 m x 80 m block of the map, so the map lines it touches are cold (the table + points
are far larger than L2).

  python bench.py [--gpus N] [--steps K] [--warmup W]          our CUDA path (C ABI)
  python bench.py --impl reference ...                         the CPU reference arm

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

_T0 = time.time()   # process start: the experimental legs' wall-clock budget counts from here
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")


class _QuietStdout:
    """Route fd 1 to stderr while libraries may chat (NCCL prints its version banner with printf at the first
    communicator), and give it back for the one JSON line: stdout must carry nothing else."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCKS_X, BLOCKS_Y, SPACING = 13, 13, 0.5   # 169 blocks x ~60 k pts = ~10.1 M map points
N_AZ = 1920                                  # 64 x 1920 = 122 880 rays, ~100 k returns (sky rays miss)
MAP_SEED, SCAN_SEED = 20260922 + 2, 20260922 + 102
WORKLOAD = "config[1]: 100k-pt 64-beam synthetic scan vs 10M-pt map, full LIO iterate-to-converge"


def load_synth():
    """The seeded generators (lidar-slam-detection_b200/synth.py, numpy only) loaded BY PATH: the reference arm must not import the
    product package (importing it dlopens liblsdreg.so)."""
    import importlib.util
    if "lsd_bench_synth" in sys.modules:
        return sys.modules["lsd_bench_synth"]
    spec = importlib.util.spec_from_file_location("lsd_bench_synth", os.path.join(ROOT, "lidar-slam-detection_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["lsd_bench_synth"] = mod
    spec.loader.exec_module(mod)
    return mod


REF_POSES = os.path.join(os.environ.get("TMPDIR", "/tmp"), "lsdreg_bench_reference_poses.json")


def workload_config(map_points, scan_points, n_down):
    """The `config` object: properties of the WORKLOAD only, so that both arms print the same keys and — the inputs being the
    same seeded scans and the downsample being the same function — the same values.  Everything that describes how an arm
    runs it goes to `impl_config`."""
    return {"workload": WORKLOAD, "map_points": int(map_points), "scan_rays": 64 * N_AZ, "scan_points": float(scan_points),
            "downsampled_points": float(n_down), "l2": "every step visits a different 120x80 m map block; table+points 4.3 GB >> 126 MB L2"}


def step_block(s: int):
    return (s * 5 + 2) % BLOCKS_X, (s * 7 + 3) % BLOCKS_Y


def make_step(s: int):
    """Scan s: ground-truth pose inside block step_block(s), the scan seen from it, and a prior
    perturbed by |t| <= 0.3 m, |theta| <= 1 deg (SURVEY.md §8d)."""
    synth = load_synth()
    bi, bj = step_block(s)
    rng = np.random.default_rng([SCAN_SEED, s])
    Rgt = synth.rot_from_rpy(*np.deg2rad(rng.uniform(-2, 2, 2)), rng.uniform(-np.pi, np.pi))
    tgt = synth.block_center(bi, bj) + np.append(rng.uniform(-3, 3, 2), 0.0)
    scan = synth.scan64(SCAN_SEED + s, N_AZ, Rgt, tgt, bi, bj)
    dR, dt = synth.perturb(SCAN_SEED + 1000 + s)
    return scan, Rgt, tgt, Rgt @ dR, tgt + dt


def quat_from_R(R):
    t = np.trace(R)
    q = np.zeros(4)
    if t > 0:
        t = np.sqrt(t + 1.0); q[3] = 0.5 * t; t = 0.5 / t
        q[0] = (R[2, 1] - R[1, 2]) * t; q[1] = (R[0, 2] - R[2, 0]) * t; q[2] = (R[1, 0] - R[0, 1]) * t
    else:
        i = int(np.argmax(np.diag(R))); j, k = (i + 1) % 3, (i + 2) % 3
        t = np.sqrt(R[i, i] - R[j, j] - R[k, k] + 1.0); q[i] = 0.5 * t; t = 0.5 / t
        q[3] = (R[k, j] - R[j, k]) * t; q[j] = (R[j, i] + R[i, j]) * t; q[k] = (R[k, i] + R[i, k]) * t
    return q


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.rows, self.index, self.proc = [], index, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def pin_to_gpu_numa(index: int):
    """Bind this process to the CPUs NVML reports as local to GPU `index` (what `numactl
    --cpunodebind` does in a deployment): pinned buffers then live on the GPU's NUMA node and the
    H2D copy / completion polling do not cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = [64 * w + b for w in range(n) for b in range(64) if (mask[w] >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


SWEEP_CACHE = os.path.join(os.environ.get("TMPDIR", "/tmp"), "lsdreg_bench_thread_sweep.json")


def sweep_child(cores, W, K):
    """Child process of the reference arm (bench.py --impl reference --sweep-only): every candidate thread count timed on
    THREE COLD blocks (one scan each, like the timed steps) of a reference map of its own; prints {threads: median seconds}."""
    from oracle import eskf
    from oracle import fastlio as FL
    synth = load_synth()
    m = synth.block_map(MAP_SEED, BLOCKS_X, BLOCKS_Y, SPACING)
    ref = FL.RefFastLioBench(capacity=1 << 30, threads=8)
    ref.add_map_points(m)
    cands = sorted({t for t in (4, 8, 16, 32, 64, cores) if t <= cores})
    if os.environ.get("LSD_BENCH_SWEEP_CANDS"):     # the second (FMA-build) child times only the winner's neighbourhood
        cands = sorted({int(t) for t in os.environ["LSD_BENCH_SWEEP_CANDS"].split(",") if 0 < int(t) <= cores}) or cands
    reps, nxt = 3, 2 * (W + K) + 64
    out = {}
    for ci, nt in enumerate(cands):
        ref.set_threads(nt)
        ts = []
        for r in range(reps):
            scan0, _, _, Rp0, tp0 = make_step(nxt + ci * reps + r)
            x = eskf.State(); x.rot = eskf.R_to_quat(Rp0); x.pos = tp0.copy()
            t1 = time.perf_counter()
            ref.process_scan(scan0, x, eskf.init_P())
            ts.append(time.perf_counter() - t1)
        out[str(nt)] = float(np.median(ts))
    print(json.dumps({"sweep_s": out, "cores": cores}))


FMA_SWEEP = {}     # {threads: median seconds} of the FMA-target build of the same sources, filled by thread_sweep


def thread_sweep(cores, W, K):
    """-> ({threads: median seconds}, how).  LSD_BENCH_REF_THREADS fixes the count; a sweep of this boot (same core count,
    younger than an hour: the reference arm runs right before the product arm) is reused; else a child process measures."""
    fixed = os.environ.get("LSD_BENCH_REF_THREADS")
    if fixed:
        return {int(fixed): 0.0}, "fixed by LSD_BENCH_REF_THREADS"
    try:
        with open(SWEEP_CACHE) as f:
            c = json.load(f)
        if c.get("cores") == cores and time.time() - c.get("when", 0) < 3600:
            FMA_SWEEP.clear(); FMA_SWEEP.update({int(k): v for k, v in c.get("fma_build_sweep_s", {}).items()})
            return {int(k): v for k, v in c["sweep_s"].items()}, "median of 3 cold-block scans per candidate in a child process (reused from the reference arm's run on this box); best median used"
    except Exception:
        pass
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--sweep-only", "--steps", str(K), "--warmup", str(W)],
                           cwd=ROOT, capture_output=True, text=True, timeout=600)
        row = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{") and "sweep_s" in ln][-1]
        sweep = {int(k): v for k, v in row["sweep_s"].items()}
        # The same sources built for an FMA target (oracle/_ref/libref_fastlio_fma.so, -O3 -march=x86-64-v3): SURVEY 8d's "fair
        # speed baseline".  Timing only, in a child of its own; the arm's value and poses stay the reference-flags build's.
        fma_lib = os.path.join(ROOT, "oracle", "_ref", "libref_fastlio_fma.so")
        if os.path.exists(fma_lib):
            try:
                best = min(sweep, key=sweep.get)
                cands = sorted({t for t in (best // 2, best, best * 2) if 4 <= t <= cores})
                r2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--sweep-only", "--steps", str(K), "--warmup", str(W)],
                                    cwd=ROOT, capture_output=True, text=True, timeout=300,
                                    env=dict(os.environ, LSD_REF_FASTLIO_LIB=fma_lib, LSD_BENCH_SWEEP_CANDS=",".join(map(str, cands))))
                row["fma_build_sweep_s"] = [json.loads(ln) for ln in r2.stdout.splitlines() if ln.startswith("{") and "sweep_s" in ln][-1]["sweep_s"]
            except Exception:  # noqa: BLE001
                pass
        try:
            with open(SWEEP_CACHE, "w") as f:
                json.dump(dict(row, when=time.time()), f)
        except OSError:
            pass
        FMA_SWEEP.clear(); FMA_SWEEP.update({int(k): v for k, v in row.get("fma_build_sweep_s", {}).items()})
        return sweep, "median of 3 cold-block scans per candidate in a child process (own map: the timed steps' map history is untouched); best median used"
    except Exception as e:  # noqa: BLE001
        return {8: 0.0}, f"sweep child failed ({type(e).__name__}): the reference's own MP_PROC_NUM = 8"


def run_cpu_fastlio(args, FL, eskf, synth, cores, dump_poses=None):
    """The reference's OWN per-scan code: laserMapping.cpp compiled unmodified with its build's -DMP_EN (oracle/_ref/
    libref_fastlio.so); each step runs the statements of fastlio_main that follow ImuProcess — pcl::VoxelGrid (the one
    restated stage, PCL being external), kf.update_iterated_dyn_share_modified with h_share_model_geometric, and
    map_incremental — on the 10 M-point map held by the reference's iVox (capacity raised, SURVEY.md section 8a row a2).

    Thread count: the reference build hard-codes MP_PROC_NUM = 8 on x86_64 (fastlio/CMakeLists.txt:20-25); "all the host
    threads it can use" is not monotone on a many-core host, so every candidate count is timed on THREE COLD blocks (blocks no
    timed step visits, one scan each, like the timed steps) and the best median wins; the sweep is reported."""
    t0 = time.time()
    m = synth.block_map(MAP_SEED, BLOCKS_X, BLOCKS_Y, SPACING)
    ref = FL.RefFastLioBench(capacity=1 << 30, threads=8)
    ref.add_map_points(m)
    setup_s = time.time() - t0
    W, K = args.warmup, args.steps
    steps = [make_step(s) for s in range(W + K)]

    def prior_of(Rp, tp):
        x = eskf.State(); x.rot = eskf.R_to_quat(Rp); x.pos = tp.copy()
        return x
    # The sweep registers scans of its own, which would leave their inserts and Nearest_Points rows in the (process-global)
    # reference state and move the poses of the timed steps by millimetres — so it runs in a CHILD process (own map) and
    # only its verdict comes back; the steps timed here see exactly the map history the product arm's steps see.
    sweep, how = thread_sweep(cores, W, K)
    ref.set_threads(min(sweep, key=sweep.get))
    times, poses, n_downs = [], [], []
    for s, (scan, Rgt, tgt, Rp, tp) in enumerate(steps):
        t1 = time.perf_counter()
        x, P, n_down = ref.process_scan(scan, prior_of(Rp, tp), eskf.init_P())
        dt = time.perf_counter() - t1
        poses.append(x.to_vec()[:7].tolist())
        if s >= W:
            times.append(dt); n_downs.append(n_down)
            err = float(np.abs(x.pos - tgt).max())
            assert n_down > 0 and err < 0.1, f"reference LIO did not converge at step {s}: {err}"
    if dump_poses:      # the product arm compares its poses of the same steps with these (pose_parity in its JSON line)
        try:
            with open(dump_poses, "w") as f:
                json.dump({"steps": K, "warmup": W, "map_seed": MAP_SEED, "scan_seed": SCAN_SEED, "map_points": int(m.shape[0]),
                           "pose7_pos_xyz_quat_xyzw": poses}, f)
        except OSError:
            pass
    total = float(np.sum(times))
    return dict(value=K / total, ms_per_step=1e3 * total / K, cores=ref.threads, host_cores=cores,
                step_ms={"median": 1e3 * float(np.median(times)), "p95": 1e3 * float(np.percentile(times, 95)), "min": 1e3 * float(np.min(times)), "max": 1e3 * float(np.max(times))},
                thread_sweep_ms={str(k): round(v * 1e3, 2) for k, v in sweep.items()},
                thread_sweep=how,
                fma_build=({"flags": "-O3 -march=x86-64-v3 (AVX2 + FMA; the arm's value and poses are the reference-flags build's)",
                            "ms_per_scan": round(1e3 * min(FMA_SWEEP.values()), 2), "threads": min(FMA_SWEEP, key=FMA_SWEEP.get),
                            "sample": "median of 3 cold-block scans per thread count, child process"} if FMA_SWEEP else None),
                kind="reference", setup_s=setup_s, poses=poses,
                iters=None, map_points=int(m.shape[0]), scan_points=float(np.mean([st[0].shape[0] for st in steps[W:]])), n_down=float(np.mean(n_downs)),
                what="laserMapping.cpp compiled unmodified (-DMP_EN): VoxelGrid -> update_iterated_dyn_share_modified -> map_incremental")


def pin_to_one_socket():
    """The CPU arm runs on ONE socket (BASELINE.json north_star: "the reference single-socket CPU scans/sec"): bind this process
    (and the sweep child it spawns) to the CPUs of one NUMA node, so that OpenMP threads and the 10 M-point iVox stay on one
    memory controller — across two sockets the same code measured anything from 20 to 54 ms per scan on the same box."""
    try:
        have = os.sched_getaffinity(0)
        best = None
        for d in sorted(os.listdir("/sys/devices/system/node")):
            if not d.startswith("node") or not d[4:].isdigit():
                continue
            cpus = set()
            for part in open(f"/sys/devices/system/node/{d}/cpulist").read().strip().split(","):
                if "-" in part:
                    a, b = part.split("-"); cpus.update(range(int(a), int(b) + 1))
                elif part:
                    cpus.add(int(part))
            cpus &= have
            if cpus and (best is None or len(cpus) > len(best)):
                best = cpus
        if best and len(best) < len(have):
            os.sched_setaffinity(0, best)
        return len(os.sched_getaffinity(0))
    except Exception:
        return 0


def run_cpu(args, rank, world, dump_poses=None):
    """Reference arm / cpu_baseline: the reference's CPU path on the host cores.  Uses oracle/_ref
    (laserMapping.cpp compiled unmodified) when it exists, else the plain-C port.  Imports nothing of the product."""
    from oracle import eskf
    from oracle.lio import OracleLio
    from oracle import oracle as O
    from oracle import fastlio as FL
    synth = load_synth()
    pin_to_one_socket()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if FL.HAVE_REF_FASTLIO and not os.environ.get("LSD_BENCH_CPU_RESTATED"):
        return run_cpu_fastlio(args, FL, eskf, synth, cores, dump_poses)
    kind = "reference" if (O.HAVE_REF and hasattr(O.ref, "ref_lio_hmodel")) else "port"
    t0 = time.time()
    m = synth.block_map(MAP_SEED, BLOCKS_X, BLOCKS_Y, SPACING)
    lio = OracleLio(18, expected_cells=1 << 24, nthreads=cores, backend=kind) if "backend" in OracleLio.__init__.__code__.co_varnames \
        else OracleLio(18, expected_cells=1 << 24, nthreads=cores)
    lio.add_map_points(m)
    setup_s = time.time() - t0
    W, K = args.warmup, args.steps
    steps = [make_step(s) for s in range(W + K)]
    # OpenMP thread count: the reference hard-codes MP_PROC_NUM = 8 (fastlio/CMakeLists.txt:17-25);
    # "all the host threads it can use" is not monotone on a many-core host, so sweep and keep the best.
    sweep = {}
    scan0, _, _, Rp0, tp0 = steps[0]
    for nt in sorted({t for t in (4, 8, 16, 32, 64, cores) if t <= cores}):
        lio.nthreads = nt
        best = 1e9
        for _ in range(2):
            prior = eskf.State(); prior.rot = eskf.R_to_quat(Rp0); prior.pos = tp0.copy()
            t1 = time.perf_counter()
            lio.process_scan(scan0, prior, eskf.init_P(), update_map=False)
            best = min(best, time.perf_counter() - t1)
        sweep[nt] = best
    lio.nthreads = min(sweep, key=sweep.get)
    times, iters = [], []
    for s, (scan, Rgt, tgt, Rp, tp) in enumerate(steps):
        prior = eskf.State(); prior.rot = eskf.R_to_quat(Rp); prior.pos = tp.copy()
        t1 = time.perf_counter()
        r = lio.process_scan(scan, prior, eskf.init_P())
        dt = time.perf_counter() - t1
        if s >= W:
            times.append(dt); iters.append(r["iters"])
            err = float(np.abs(lio.x.pos - tgt).max())
            assert err < 0.1, f"CPU LIO did not converge at step {s}: {err}"
    total = float(np.sum(times))
    value = K / total
    return dict(value=value, ms_per_step=1e3 * total / K, cores=lio.nthreads, host_cores=cores,
                step_ms={"median": 1e3 * float(np.median(times)), "p95": 1e3 * float(np.percentile(times, 95)), "min": 1e3 * float(np.min(times)), "max": 1e3 * float(np.max(times))},
                thread_sweep_ms={str(k): round(v * 1e3, 2) for k, v in sweep.items()}, kind=kind, setup_s=setup_s, poses=None,
                iters=float(np.mean(iters)), map_points=int(m.shape[0]), scan_points=float(np.mean([st[0].shape[0] for st in steps[W:]])), n_down=None)


def run_knn_batch(torch, hmap, m, dev, nq):
    """5-NN (NEARBY18, d2 < 5) for nq queries against the resident map through lsd_knn_query_dev, timed with CUDA
    events on the library's stream (the whole call: for the brick shape that is the three binning kernels + the search).
    Queries = map points + N(0, 0.1 m) noise: 'random' = random order over the whole 10 M-point map (every query's
    cell lines are cold), 'sorted' = the same queries in voxel order.  L2 is flushed before every launch.
    Shapes: the batch default (brick pages staged through TMA, csrc/brick.cuh) and, for reference, round 1's
    thread-per-query kernel over the voxel lines; the two must return identical bits."""
    rng = np.random.default_rng(99)
    sel = rng.integers(0, m.shape[0], nq)
    q = m[sel].copy()
    q[:, :3] += rng.normal(0.0, 0.1, (nq, 3)).astype(np.float32)
    cell = np.round(q[:, :3] / 0.5).astype(np.int64)
    order = np.lexsort((cell[:, 0], cell[:, 1], cell[:, 2]))
    stream = torch.cuda.ExternalStream(hmap.stream(), device=dev)
    t0 = time.perf_counter()
    hmap.enable_bricks(19)          # copies the 10 M points of the populated map into their brick pages
    torch.cuda.synchronize()
    brick_build_s = time.perf_counter() - t0
    bst = hmap.brick_stats()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"queries": nq, "k": 5, "stencil": "NEARBY18", "shape": "brick pages, TMA-staged (lsd_knn_set_shape 3 = the batch default)",
           "brick_pages": bst["pages"], "brick_replicas": bst["replicas"], "brick_dropped": bst["dropped"], "brick_build_s": brick_build_s}
    res = {}
    for shape, tag in ((3, ""), (2, "thread_")):
        hmap.set_knn_shape(shape)
        for name, qq in (("random", q), ("sorted", q[order])):
            qd = torch.from_numpy(np.ascontiguousarray(qq)).to(dev)
            idx = torch.empty((nq, 5), dtype=torch.int32, device=dev)
            d2 = torch.empty((nq, 5), dtype=torch.float32, device=dev)
            cnt = torch.empty(nq, dtype=torch.int32, device=dev)
            times = []
            for rep in range(6):
                flush.fill_(rep)                      # > L2: the next launch starts from HBM
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                hmap.knn_dev(qd, idx, d2, cnt, k=5, max_sq=5.0)
                e1.record(stream)
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1) * 1e3)
            out[tag + name + "_us"] = float(np.median(times[2:]))
            res[(shape, name)] = (idx, d2, cnt)
            if shape == 3:
                out[name + "_found5"] = float((cnt == 5).float().mean().item())
    hmap.set_knn_shape(0)
    out["identical_to_thread_shape"] = bool(all(torch.equal(a, b) for n in ("random", "sorted") for a, b in zip(res[(3, n)], res[(2, n)])))
    return out


def finish_knn_batch(kb, bytes_per_query, peak):
    out = dict(kb, bytes_per_query=bytes_per_query, peak=peak)
    for k in list(kb):
        if k.endswith("_us") and kb[k]:
            gbs = kb["queries"] * bytes_per_query / (kb[k] * 1e-6) / 1e9
            out[k[:-3] + "_gbs"] = gbs
            out[k[:-3] + "_frac"] = gbs / peak
    return out


def run_streams(torch, lsdreg, local, m, steps, dev_scans, W, K, S, prior_vec, P0):
    """S host threads, each with its own LioFrontend (own map replica, own CUDA stream), all registering the same K
    device-resident scans concurrently.  ctypes releases the GIL inside the C calls."""
    import threading
    handles = []
    for _ in range(S):
        h = lsdreg.LioFrontend(map_log2_lines=25, max_scan_points=131072, max_points=100000, async_map_insert=1)
        h.map.insert(m, 0)
        h.set_next_id(m.shape[0])
        handles.append(h)
    start = threading.Barrier(S + 1)
    done = threading.Barrier(S + 1)
    errs = [0.0] * S

    def worker(k):
        lsdreg.init(local)
        h = handles[k]
        for s in range(W):
            h.scan(dev_scans[s], prior_vec(steps[s]), P0)
        h.sync()
        start.wait()
        worst = 0.0
        for s in range(W, W + K):
            x, P, info = h.scan(dev_scans[s], prior_vec(steps[s]), P0)
            worst = max(worst, float(np.abs(x[:3] - steps[s][2]).max()))
        h.sync()
        errs[k] = worst
        done.wait()

    ths = [threading.Thread(target=worker, args=(k,)) for k in range(S)]
    for t in ths:
        t.start()
    start.wait()
    t0 = time.perf_counter()
    done.wait()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    for t in ths:
        t.join()
    for h in handles:
        h.close()
    return {"streams": S, "value": S * K / wall, "unit": "scans/s", "ms_per_scan_per_stream": 1e3 * wall / K,
            "pos_err_max_m": max(errs), "note": "independent streams, one map replica and one handle each, same GPU"}


def step_stats(ts):
    ts = np.asarray(ts, np.float64) * 1e3
    return {"median": float(np.median(ts)), "p95": float(np.percentile(ts, 95)), "min": float(ts.min()), "max": float(ts.max())}


def pose_delta(x_ours, pose7_ref):
    """|dpos| (m, max over axes) and the rotation angle (rad) between two (pos, quat xyzw) poses."""
    pa, pb = np.asarray(x_ours[:3]), np.asarray(pose7_ref[:3])
    qa, qb = np.asarray(x_ours[3:7]), np.asarray(pose7_ref[3:7])
    dot = abs(float(np.dot(qa / np.linalg.norm(qa), qb / np.linalg.norm(qb))))
    return float(np.abs(pa - pb).max()), float(2.0 * np.arccos(min(1.0, dot)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=3, help="scans timed for cpu_baseline (N=1, rank 0)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-knn-batch", action="store_true")
    ap.add_argument("--no-shard-leg", action="store_true", help="N>1: skip the tile-sharded leg (replicas only)")
    ap.add_argument("--no-reference-order-leg", action="store_true", help="N=1: skip the extra leg with lsd_lio_set_reference_order off (sorted rows)")
    ap.add_argument("--sweep-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--streams", type=int, default=4, help="extra leg (N=1): this many independent scan streams, each with "
                    "its own map replica and handle, registered concurrently on the one GPU (0/1 = skip)")
    ap.add_argument("--no-prefetch", action="store_true", help="e2e leg: upload each scan inside lsd_lio_scan instead of one scan ahead")
    ap.add_argument("--knn-batch", type=int, default=1 << 21, help="queries in the batched k-NN leg (N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned for its last step (state vector "
                    "and covariance, float64) as DIR/<name>.npy, to compare two builds output for output")
    ap.add_argument("--mg-mode", default="replicas", choices=["replicas", "shard"],
                    help="N>1, what `value` / `e2e` report: 'replicas' = one map replica and one independent scan stream per GPU "
                         "(weak scaling, no collective); 'shard' = ONE scan stream, map tile-sharded across the GPUs, normal equations "
                         "all-reduced through peer memory inside the reduction kernel (strong scaling).  The other mode is "
                         "always reported beside it (`shard` / `replicas` object of the line)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        if rank != 0:
            return 0
        if args.sweep_only:
            pin_to_one_socket()
            cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            sweep_child(cores, args.warmup, args.steps)
            return 0
        r = run_cpu(args, rank, world, dump_poses=REF_POSES)
        line = {"impl": "reference", "metric": "scans/sec", "value": r["value"], "unit": "scans/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(r["map_points"], r["scan_points"], r["n_down"] if r["n_down"] is not None else -1),
                "impl_config": {"parallelism": f"{r['cores']} OpenMP threads on one socket ({r['host_cores']} CPUs of {os.cpu_count()} on the box)", "what": r.get("what", "restated loop on the compiled reference iVox / esti_plane"),
                                "thread_sweep_ms": r["thread_sweep_ms"], "thread_sweep": r.get("thread_sweep"), "fma_build": r.get("fma_build"),
                                "timing": "host wall clock around each fastlio_main pass (ref_fastlio_pass), summed over the K timed steps"},
                "step_ms": r["step_ms"],
                "cpu_baseline": {"value": r["value"], "unit": "scans/s", "cores": r["cores"], "kind": r["kind"],
                                 "host_cores": r["host_cores"], "thread_sweep_ms": r["thread_sweep_ms"], "fma_build": r.get("fma_build"), "what": r.get("what", "restated loop on the compiled reference iVox / esti_plane"),
                                 "sample": f"{args.steps} full scans of the workload after {args.warmup} warm-up scans"},
                "e2e": {"value": r["value"], "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "mean_iterations": r["iters"], "poses_written_to": REF_POSES}
        print(json.dumps(line))
        return 0

    numa_cpus = pin_to_gpu_numa(local)
    import torch
    import lsdreg
    synth = load_synth()
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    lsdreg.init(local)
    dev = torch.device("cuda", local)
    W, K = args.warmup, args.steps
    n_prof = 5
    P0 = lsdreg.init_cov()
    m = synth.block_map(MAP_SEED, BLOCKS_X, BLOCKS_Y, SPACING)

    def prior_vec(stp):
        return lsdreg.make_state(pos=stp[4], rot_xyzw=quat_from_R(stp[3]))

    def lio_is_sharded(lio):
        return bool(getattr(lio, "_bench_sharded", False))

    def run_steps(lio, steps, scans, timed_from, prefetch=False):
        """Returns (wall seconds of the timed part, per-step infos incl. host wall time per call, poses of ALL steps, and the
        state vector and covariance the last step returned).
        Bracketed by sync + barrier.  prefetch: the next scan is announced before the current one is registered (host
        scans: its H2D copy runs on the copy stream; any scan: its voxel grid is pipelined under the running scan)."""
        # Per-step inputs and outputs are laid out before the timed region (the priors are the workload's, not the path's);
        # inside it the loop is: announce scan s+1, register scan s in place, keep a copy of the pose.
        n = len(steps)
        states = [np.array(prior_vec(stp), np.float64) for stp in steps]
        covs = [np.array(P0, np.float64) for _ in steps]
        cinfos = [lsdreg.capi.LioInfo() for _ in steps]
        call_s = np.zeros(n)
        status = [0] * n
        t_start = None
        clock = time.perf_counter
        if prefetch:
            lio.prefetch(scans[0])
        for s in range(n):
            if s == timed_from:
                torch.cuda.synchronize()
                if dist is not None:
                    dist.barrier()
                if lio_is_sharded(lio):
                    lio.shard_exchange_stats()     # reset: warm-up evaluations (ranks out of step) are not the exchange's cost
                t_start = clock()
            t1 = clock()
            if prefetch and s + 1 < n:
                lio.prefetch(scans[s + 1])
            status[s] = lio.scan_into(scans[s], states[s], covs[s], cinfos[s])
            call_s[s] = clock() - t1
        last_ms, _ = lio.sync()
        torch.cuda.synchronize()
        wall = clock() - t_start
        infos, poses = [], [x[:7].copy() for x in states]
        for s in range(timed_from, n):
            info = dict(cinfos[s].as_dict(), status=status[s])
            info["call_s"] = float(call_s[s])
            info["pos_err"] = float(np.abs(states[s][:3] - steps[s][2]).max())
            infos.append(info)
            if len(infos) >= 2:
                infos[-2]["gpu_ms"] = info["gpu_ms"]  # async insert: device time is reported one scan late
        infos[-1]["gpu_ms"] = last_ms
        return wall, infos, poses, (states[-1], covs[-1])

    def run_mode(sharded):
        """The value leg (scans resident in HBM) and the e2e leg (pinned host scans, H2D inside) of one multi-GPU mode."""
        lio = lsdreg.LioFrontend(map_log2_lines=25, max_scan_points=131072, max_points=100000, async_map_insert=1)
        t0 = time.perf_counter()
        if sharded:
            from lsdreg import shard as shardlib
            shardlib.connect(lio, rank, world, tile_cells=shardlib.TILE_CELLS, reach_cells=1)
            lio._bench_sharded = True
        lio.map.insert(m, 0)
        build_s = time.perf_counter() - t0
        lio.set_next_id(m.shape[0])
        st = lio.map.stats()
        base = 0 if sharded else rank * (2 * (W + K) + n_prof)  # shard mode: every rank sees the same scans
        steps_a = [make_step(base + s) for s in range(W + K)]
        steps_b = [make_step(base + W + K + s) for s in range(W + K)]
        dev_scans = [torch.from_numpy(stp[0]).to(dev) for stp in steps_a]
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.3)
        wall_a, infos_a, poses_a, last_a = run_steps(lio, steps_a, dev_scans, W, prefetch=True)
        clocks = sampler.stop()
        xchg = lio.shard_exchange_stats() if sharded else None     # over the timed steps of the value leg
        host_scans = [torch.from_numpy(stp[0]).pin_memory() for stp in steps_b]
        scratch = torch.empty((131072, 4), dtype=torch.float32, device=dev)
        for hs in host_scans:  # first DMA from a freshly pinned buffer pays a one-off mapping cost: take it here
            scratch[:hs.shape[0]].copy_(hs, non_blocking=True)
        torch.cuda.synchronize()
        wall_b, infos_b, _, _ = run_steps(lio, steps_b, host_scans, W, prefetch=not args.no_prefetch)
        dev_ms = float(np.sum([i["gpu_ms"] for i in infos_a]))
        t = torch.tensor([wall_a, wall_b, dev_ms * 1e-3], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall_a, wall_b, dev_s = [float(v) for v in t.cpu()]
        for i in infos_a + infos_b:
            assert i["pos_err"] < 0.1, f"LIO did not converge: {i}"
        streams = 1 if sharded else world
        return dict(xchg=xchg, lio=lio, st=st, build_s=build_s, steps_a=steps_a, steps_b=steps_b, dev_scans=dev_scans, host_scans=host_scans,
                    infos_a=infos_a, infos_b=infos_b, poses_a=poses_a, last_a=last_a, clocks=clocks, wall_a=wall_a, wall_b=wall_b, dev_s=dev_s,
                    value=streams * K / wall_a, e2e=streams * K / wall_b, base=base)

    want_shard = world > 1 and args.mg_mode == "shard"
    main_run = run_mode(want_shard)
    other = None
    if world > 1 and not args.no_shard_leg:      # the other mode, reported beside the headline in the same line
        other = run_mode(not want_shard)
        other["lio"].close(); other["lio"] = None
    R = main_run
    lio, st, infos_a, infos_b = R["lio"], R["st"], R["infos_a"], R["infos_b"]
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        state, cov = R["last_a"]
        np.save(os.path.join(args.dump_outputs, "state.npy"), np.asarray(state, np.float64))
        np.save(os.path.join(args.dump_outputs, "cov.npy"), np.asarray(cov, np.float64))
    rho = st["points"] / max(st["cells"], 1)

    # H2D probe: what this box's PCIe path gives a 1.6 MB pinned copy (explains e2e - value)
    probe_src = R["host_scans"][0]
    probe_dst = torch.empty(probe_src.shape, dtype=probe_src.dtype, device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        probe_dst.copy_(probe_src, non_blocking=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(10):
        probe_dst.copy_(probe_src, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    h2d_us = ev0.elapsed_time(ev1) * 1e3 / 10
    # ---------------- per-kernel timing pass for the roofline (not part of any throughput number)
    steps_p = [make_step(R["base"] + 2 * (W + K) + s) for s in range(n_prof)]
    lio.set_profile(True)
    n_down_p = []
    for stp in steps_p:
        x, P, info = lio.scan(torch.from_numpy(stp[0]).to(dev), prior_vec(stp), P0)
        n_down_p.append(info["n_down"])
    prof = lio.get_profile()
    lio.set_profile(False)

    # ---------------- batched k-NN (BASELINE metric "kNN GB/s vs HBM peak"): many scans' worth of queries in flight
    knn_batch = None
    if world == 1 and not args.no_knn_batch:
        knn_batch = run_knn_batch(torch, lio.map, m, dev, args.knn_batch)

    # ---------------- several independent scan streams on ONE GPU (a fleet server): what the GPU sustains when a
    # single stream's latency chain no longer leaves it idle.  Reported beside the headline, never instead of it.
    multi_stream = None
    if world == 1 and args.streams > 1:
        multi_stream = run_streams(torch, lsdreg, local, m, R["steps_a"], R["dev_scans"], W, K, args.streams, prior_vec, P0)

    # ---------------- the same K steps with Nearest_Points sorted by distance instead of in the reference's own order
    # (lsd_lio_set_reference_order(0)): what exactness against laserMapping.cpp costs.  Reported beside the headline.
    ref_order_leg = None
    if world == 1 and not args.no_reference_order_leg:
        h = lsdreg.LioFrontend(map_log2_lines=25, max_scan_points=131072, max_points=100000, async_map_insert=1)
        h.map.insert(m, 0)
        h.set_next_id(m.shape[0])
        h.set_reference_order(False)
        wall_r, infos_r, poses_r, _ = run_steps(h, R["steps_a"], R["dev_scans"], W, prefetch=True)
        ref_order_leg = {"value": K / wall_r, "unit": "scans/s", "ms_per_step": 1e3 * wall_r / K,
                         "device_ms_per_step": float(np.sum([i["gpu_ms"] for i in infos_r])) / K,
                         "vs_this_lines_value": (K / wall_r) / R["value"],
                         "pos_err_max_m": max(i["pos_err"] for i in infos_r), "poses": poses_r,
                         "what": "lsd_lio_set_reference_order(0): Nearest_Points rows in ascending (d2, id) order instead of the order "
                                 "IVox::GetClosestPoint returns them in (the default, which the headline runs)"}
        h.close()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    hs = prof["hmodel_search"]
    n_q = float(np.mean(n_down_p))
    bytes_per_query = 56 + 19 * (8 + 16 * rho)   # SURVEY.md §8d: K3 algorithmic bytes, S = 19, k = 5
    alg_bytes = n_q * bytes_per_query
    dur_s = hs["ms"] / max(hs["count"], 1) * 1e-3
    achieved = alg_bytes / dur_s / 1e9 if dur_s > 0 else 0.0
    peak, peak_src = 6650.0, "fallback"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak, peak_src = float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        pass
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f).get("lio_hmodel_search_bytes_per_launch")
    except Exception:
        pass

    # ---------------- pose parity with the reference arm: the poses laserMapping.cpp (compiled unmodified) computed for the
    # SAME steps — from the file `bench.py --impl reference` left behind on this box when it ran before us with the same
    # K / W, else from the in-process cpu_baseline sample below.  This is parity, not accuracy (pos_err_max_m is vs truth).
    pose_parity = None

    def compare(ref_poses, source, ours=None):
        ours = R["poses_a"] if ours is None else ours
        n = min(len(ref_poses), len(ours))
        dm = [pose_delta(ours[s], ref_poses[s]) for s in range(n)]
        out = {"max_m": max(d[0] for d in dm), "max_rad": max(d[1] for d in dm),
               "median_m": float(np.median([d[0] for d in dm])), "median_rad": float(np.median([d[1] for d in dm])),
               "steps_within_bar": int(sum(1 for d in dm if d[0] < 1e-4 and d[1] < 1e-5)), "steps_compared": n, "against": source,
               "bar": "1e-4 m / 1e-5 rad (BASELINE.json north_star)", "within_bar": bool(max(d[0] for d in dm) < 1e-4 and max(d[1] for d in dm) < 1e-5)}
        try:     # the reference's own build-to-build spread on these steps (tools/ref_build_sensitivity.py, run where the reference tree is)
            with open(os.path.join(ROOT, "profiles", "r02_ref_build_sensitivity.json")) as f:
                sens = json.load(f)["variants"]
            worst = max(sens, key=lambda k: sens[k]["max_rad"])
            out["reference_vs_itself"] = {"build": worst, "max_m": sens[worst]["max_m"], "max_rad": sens[worst]["max_rad"],
                                          "steps_over_bar": sens[worst]["steps_over_bar"],
                                          "what": "the same unmodified sources compiled for another x86 target vs the build compared here, same steps "
                                                  "(profiles/r02_ref_build_sensitivity.json): the bar sits at the reference's own reproducibility"}
        except Exception:
            pass
        return out
    if True:     # rank 0 registers steps 0.. in either mode
        try:
            with open(REF_POSES) as f:
                rp = json.load(f)
            if rp.get("steps") == K and rp.get("warmup") == W and rp.get("map_seed") == MAP_SEED and rp.get("scan_seed") == SCAN_SEED:
                pose_parity = compare(rp["pose7_pos_xyz_quat_xyzw"], f"bench.py --impl reference on this box ({REF_POSES}): laserMapping.cpp compiled unmodified, all {W}+{K} steps")
                if ref_order_leg is not None:
                    pp = compare(rp["pose7_pos_xyz_quat_xyzw"], "the same reference poses", ours=ref_order_leg["poses"])
                    pp.pop("reference_vs_itself", None)
                    ref_order_leg["pose_parity"] = pp
        except Exception:
            pass

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        a2 = argparse.Namespace(steps=args.cpu_sample, warmup=1)
        r = run_cpu(a2, 0, 1)
        cpu = {"value": r["value"], "unit": "scans/s", "cores": r["cores"], "kind": r["kind"],
               "host_cores": r["host_cores"], "thread_sweep_ms": r["thread_sweep_ms"], "thread_sweep": r.get("thread_sweep"), "fma_build": r.get("fma_build"),
               "what": r.get("what", "restated loop on the compiled reference iVox / esti_plane"),
               "sample": f"{args.cpu_sample} full scans of the same workload (same map, same generator) after 1 warm-up scan",
               "ms_per_scan": r["ms_per_step"], "mean_iterations": r["iters"]}
        if pose_parity is None and r.get("poses"):
            pose_parity = compare(r["poses"], f"in-process cpu_baseline: laserMapping.cpp compiled unmodified, steps 0..{args.cpu_sample}")

    def mode_summary(X, sharded):
        return {"mode": "shard" if sharded else "replicas", "scaling": "strong" if sharded else "weak",
                "value": X["value"], "e2e": X["e2e"], "unit": "scans/s", "ms_per_step": 1e3 * X["wall_a"] / K, "e2e_ms_per_step": 1e3 * X["wall_b"] / K,
                "device_ms_per_step": 1e3 * X["dev_s"] / K, "pos_err_max_m": float(np.max([i["pos_err"] for i in X["infos_a"]])),
                "map_points_this_rank": int(X["st"]["points"]), "gpu_launches": int(np.sum([i["kernel_launches"] for i in X["infos_a"]])),
                "in_kernel_exchange": X.get("xchg") and dict(X["xchg"], what="mean us per h-model evaluation between this rank's partial sums being ready and every peer's having arrived (clock64 in grid_finalize, rank 0)"),
                "parallelism": (f"map tile-sharded over {world} GPUs, ONE scan stream, peer-memory all-reduce of the normal equations inside the reduction kernel"
                                if sharded else f"{world} replicas, independent scan streams, no collective")}

    iters = float(np.mean([i["iterations"] for i in infos_a]))
    h2d = int(np.mean([stp[0].shape[0] for stp in R["steps_b"][W:]]) * 16)
    d2h = int(iters * (32 + 8) * 8 + 4)
    line = {
        "metric": "scans/sec", "value": R["value"], "unit": "scans/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * R["wall_a"] / K, "higher_is_better": True, "scaling": "strong" if want_shard else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(m.shape[0], np.mean([stp[0].shape[0] for stp in R["steps_a"][W:]]), np.mean([i["n_down"] for i in infos_a])),
        "impl_config": {"map_voxels": int(st["cells"]), "mean_iterations": iters,
                        "parallelism": "1 GPU" if world == 1 else mode_summary(R, want_shard)["parallelism"],
                        "shard_points_this_rank": int(st["points"]),
                        "pipeline_vg": os.environ.get("LSD_PIPELINE_VG", "1")[:1] != "0",   # voxel grid of scan s+1 on the copy stream under scan s (default on)
                        "pdl": os.environ.get("LSD_PDL", "0")[:1] == "1",                   # programmatic dependent launch (opt-in)
                        "stale_rows": True,
                        "reference_order": os.environ.get("LSD_REF_ORDER", "1")[:1] != "0",   # neighbours in the reference's own order (default; the `sorted_order` leg measures the alternative)
                        "reference_order_fallbacks": lio.reference_order_fallbacks(),
                        "voxelgrid_sums": "fixed-point" if os.environ.get("LSD_VG_SUMS", "")[:1] == "f" else "fp32, input order (the restated pcl::VoxelGrid's arithmetic)",
                        "timing": "wall clock around K steps bracketed by cuda sync (+barrier), max over ranks; device_ms_per_step = CUDA events on the library stream; "
                                  "step_ms = host wall time of each lsd_lio_scan call (what the caller waits for)"},
        "device_ms_per_step": 1e3 * R["dev_s"] / K,
        "step_ms": step_stats([i["call_s"] for i in infos_a]),
        "e2e": {"value": R["e2e"], "unit": "scans/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * R["wall_b"] / K, "step_ms": step_stats([i["call_s"] for i in infos_b]), "h2d_probe_us": h2d_us,
                "h2d_probe_gbs": probe_src.numel() * 4 / (h2d_us * 1e-6) / 1e9,
                "host_binding": f"{numa_cpus} CPUs local to the GPU (NVML affinity)" if numa_cpus else "unbound",
                "ingest": "serial: H2D inside lsd_lio_scan" if args.no_prefetch else
                          "double-buffered: lsd_lio_prefetch uploads scan k+1 on a copy stream while scan k is registered; "
                          "every scan's H2D copy and result read-back are inside the timed region"},
        "gpu_launches": int(np.sum([i["kernel_launches"] for i in infos_a])),
        "pose_parity": pose_parity,
        "roofline": {"kernel": "lio_knn_kernel + lio_hmodel_kernel<search> (one search evaluation)", "bound": "hbm", "achieved": achieved, "peak": peak,
                     "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_query": bytes_per_query, "rho": rho,
                     "queries_per_launch": n_q, "us_per_launch": dur_s * 1e6, "launches_timed": hs["count"]},
        "kernels_ms": {k: (v["ms"] / max(v["count"], 1)) for k, v in prof.items()},
        "knn_batch": knn_batch and finish_knn_batch(knn_batch, bytes_per_query, peak),
        "multi_stream": multi_stream,
        "sorted_order": ({k: v for k, v in ref_order_leg.items() if k != "poses"} if ref_order_leg else None),
        "cpu_baseline": cpu, "clocks": R["clocks"], "map_build_s": R["build_s"],
        "pos_err_max_m": float(np.max([i["pos_err"] for i in infos_a])),
    }
    if other is not None:
        line["shard" if not want_shard else "replicas"] = mode_summary(other, not want_shard)
        line[("shard" if not want_shard else "replicas")]["vs_this_lines_value"] = other["value"] / R["value"]
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    import contextlib
    import io
    buf = io.StringIO()
    with _QuietStdout():
        with contextlib.redirect_stdout(buf):      # main() prints the JSON line: hold it until fd 1 is ours again
            rc = main()
    sys.stdout.write(buf.getvalue())
    sys.stdout.flush()
    sys.exit(rc)
