#!/usr/bin/env python
"""bench.py — pairwise registrations/sec of the map_merge_3d hot path on B200 (and the CPU reference arm).

A "step" is one whole estimateMapsTransforms() over the workload: the per-map feature pipeline (voxel grid, outlier
removal, normals, keypoints, descriptors) for every map plus the all-pairs loop (reciprocal k-NN matching, RANSAC, ICP
refine, scoring) and the host pose graph.

Workloads (BASELINE.json configs):
  c3 (default)  32 synthetic maps x 1M points, SIFT + FPFH, 496 pairs — the configuration the headline metric is quoted on
  c2            8 maps x 500k points, SIFT + FPFH, 28 pairs
  c4            16 maps x 500k points, Harris3D + SHOT-1344, inlier_threshold 0.2, 120 pairs
  c5            composeMaps of 4 maps x 10M points at output_resolution 0.05 (metric: input points/s)

  value : pairs/s, inputs already resident in HBM when the timed region starts (CUDA events, max over ranks); per-kernel
          profiling is OFF in this region — the roofline / kernel table come from a separate profiled pass
  e2e   : pairs/s through the C-ABI call with HOST buffers (pinned), H2D of the clouds and D2H of the transforms inside the
          timed region
  N > 1 : one process per GPU (torchrun).  The whole multi-GPU step runs inside the library (mm3d_estimate_*_dist,
          csrc/dist.cu): maps sharded for the feature pipeline, NCCL exchange of features, LPT-sharded pair list, results
          all-reduced into the reference's pair order, host graph on every rank.  torch.distributed only hands the NCCL id
          around and provides the barrier / max-over-ranks.  Same workload at every N => "scaling": "strong".
  --impl reference : the CPU restatement of the reference (oracle/, all host threads), bounded sample per step.

  --dump-outputs DIR : after the timed steps, what the last timed step returned to its caller is saved as DIR/<name>.npy
          (transforms.npy, or composed_points.npy for c5), at most 64 MB in all; the inputs are seeded, so two builds run
          with the same arguments can be compared output for output.
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

# the benchmark runs from the tree as built and writes nothing into it (the tree may be read-only)
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pairwise_registrations_per_sec"
UNIT = "pairs/s"

# roofline denominator: HBM copy bandwidth (read + write) measured on an NVIDIA B200 at SM max 1965 MHz, power limit not
# recorded (BASELINE.md section 2)
HBM_PEAK_GBS = 6453.7
HBM_PEAK_SOURCE = "HBM copy bandwidth measured on a B200 (BASELINE.md section 2)"

DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this many bytes of files in all

WORKLOADS = {
    "c2": dict(params=dict(descriptor_type="FPFH"), what="SIFT+FPFH, MATCHING+ICP"),
    "c3": dict(params=dict(descriptor_type="FPFH"), what="SIFT+FPFH, MATCHING+ICP"),
    "c4": dict(params=dict(keypoint_type="HARRIS", keypoint_threshold=0.0, descriptor_type="SHOT", inlier_threshold=0.2),
               what="Harris3D+SHOT-1344, inlier_threshold 0.2, MATCHING+ICP"),
    "tiny": dict(params=dict(descriptor_type="FPFH"), what="SIFT+FPFH, MATCHING+ICP"),
    "small": dict(params=dict(descriptor_type="FPFH"), what="SIFT+FPFH, MATCHING+ICP"),
}


def synth_mod():
    import mm3d_pkg
    return mm3d_pkg.load_synth()


def n_pairs_of(m: int) -> int:
    return m * (m - 1) // 2


def workload_label(name, cfg):
    m = cfg["n_maps"]
    return f"{name}: {m} maps x {cfg['n_points']} pts, {WORKLOADS[name]['what']}, {n_pairs_of(m)} pairs"


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Saves every array as <out_dir>/<name>.npy, the files ``budget`` bytes at most in all.  An array larger than its share
    is cut to a fixed, seeded sample of its rows, kept in their original order, so that the files of two runs line up row
    for row."""
    os.makedirs(out_dir, exist_ok=True)
    share = budget // len(arrays) - 4096  # room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if a.nbytes > share:
            rows = share // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), rows, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """SM clock + throttle reasons sampled during the timed region through NVML in a background thread (pynvml; an
    `nvidia-smi -lms 100` child process was measured to slow the host side of short steps by up to 2x while it polls, and
    100 ms NVML polling the c3 step by up to 30 %: the queries contend with CUDA calls for the driver lock)."""

    PERIOD = 1.0  # seconds between samples: a query can hold the driver lock for tens of ms, so few of them fall into a step

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # no NVML: fall back to one nvidia-smi query at the end
            self.err = str(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.perf_counter(), sm, reasons))
            except Exception as e:
                self.err = str(e)
                return
            self.stop_flag.wait(self.PERIOD)  # NVML queries contend with CUDA calls for the driver lock: 100 ms polling cost up to 30 % of a step

    def stop(self, t0=None, t1=None):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=2)
        if not self.samples:
            return self._smi_once()
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        sel = [x for x in self.samples if t0 is None or (t0 <= x[0] <= t1 + 0.15)] or self.samples
        reasons = sorted(k for k, b in bits.items() if any(x[2] & b for x in sel))
        return {"sm_mhz": float(np.median([x[1] for x in sel])), "sm_max_mhz": self.max_sm, "samples": len(sel), "reasons": reasons,
                "source": f"NVML, {self.PERIOD:g} s period, samples inside the timed region"}

    def _smi_once(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
            parts = [p.strip() for p in out.split(",")]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            return {"sm_mhz": float(parts[0]), "sm_max_mhz": float(parts[1]), "samples": 1,
                    "reasons": [n for n, v in zip(names, parts[2:6]) if v.lower().startswith("active")],
                    "source": f"one nvidia-smi query after the timed region (NVML thread unavailable: {self.err})"}
        except Exception as e:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": [f"clock sampling unavailable: {e}"]}


# ---------------------------------------------------------------------------------------------- CPU arms
def oracle_params(oracle_py, name):
    kw = dict(WORKLOADS[name]["params"])
    conv = dict(descriptor_type=dict(PFH=0, PFHRGB=1, FPFH=2, RSD=3, SHOT=4, SC3D=5), keypoint_type=dict(SIFT=0, HARRIS=1))
    for k in list(kw):
        if k in conv and isinstance(kw[k], str):
            kw[k] = conv[k][kw[k]]
    return oracle_py.default_params(**kw)


def oracle_sample_job(O, maps, p):
    """The reference's loops (map_merging.cpp:212-269) on the CPU restatement: stage-major over the sample maps, then the
    pair loop, sequential like the reference, each stage's per-point loop on all host threads.  Returns per-map and
    per-pair seconds and the results."""
    r = O.estimate_maps_transforms(maps, p)
    st = r["stage_times"]
    feat = sum(st[k] for k in ("downsampling", "removing outliers", "normals computation", "keypoints detection", "descriptors computation"))
    pair = sum(st[k] for k in ("finding correspondences", "initial alignment", "ICP alignment", "scoring"))
    n_pairs = max(len(r["pairs"]), 1)
    return feat / len(maps), pair / n_pairs, r


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "c5":
        return run_reference_compose(args)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    O = oracle_py.Oracle()
    threads = O.set_threads(0)
    synth = synth_mod()
    cfg = dict(synth.CONFIGS[args.workload])
    M = cfg["n_maps"]
    P = n_pairs_of(M)
    sample = min(2, M)
    maps, _ = synth.make_maps(**cfg, only=range(sample))
    sub = maps[:sample]
    p = oracle_params(oracle_py, args.workload)
    total_steps = args.steps + args.warmup
    feats, pairs = [], []
    t_run = time.perf_counter()
    done = 0
    for s in range(total_steps):
        f, g, r = oracle_sample_job(O, sub, p)
        done += 1
        if s >= args.warmup:
            feats.append(f); pairs.append(g)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"transforms": r["transforms"]})
    full = M * float(np.mean(feats)) + P * float(np.mean(pairs))
    value = P / full
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": full * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(args.workload, cfg), "seed": cfg["seed"]},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": (f"per step: maps 0-{sample - 1} of the workload through the whole path ({n_pairs_of(sample)} of {P} pairs), the "
                                    f"reference's sequential map / pair loops with every per-point loop on {threads} host threads (OpenMP); "
                                    f"per-map ({np.mean(feats):.2f} s) and per-pair ({np.mean(pairs):.2f} s) times extrapolated to {M} maps / {P} pairs; "
                                    f"{(time.perf_counter() - t_run):.0f} s of CPU wall for {done} steps"),
                         "what": "CPU restatement of the reference's algorithm (oracle/, grid-hash neighbour search) — not PCL/FLANN itself, "
                                 "which cannot be built in this image"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()


def run_reference_compose(args):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    O = oracle_py.Oracle()
    synth = synth_mod()
    cfg = dict(synth.CONFIGS["c5"])
    M = cfg["n_maps"]
    maps, truth = synth.make_maps(**cfg, only=[0])
    T = np.eye(4, dtype=np.float32)[None]
    times = []
    for s in range(args.steps + args.warmup):
        t0 = time.perf_counter()
        out = O.compose_maps(maps[:1], T, 0.05)
        if s >= args.warmup:
            times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"composed_points": out})
    per_map = float(np.mean(times))
    value = cfg["n_points"] / per_map
    line = {"impl": "reference", "metric": "compose_maps_points_per_sec", "value": value, "unit": "points/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_map * M * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"c5: composeMaps of {M} maps x {cfg['n_points']} pts at output_resolution 0.05", "seed": cfg["seed"]},
            "cpu_baseline": {"value": value, "unit": "points/s", "cores": 1, "kind": "port",
                             "sample": f"map 0 of the workload composed alone per step ({per_map:.2f} s), scaled to {M} maps"},
            "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()


def cpu_baseline_and_parity(job, maps, name, M, P):
    """N = 1 only: the CPU restatement on maps 0-1 of the workload (one pair) — timed as the cpu_baseline, and its results
    compared with the CUDA path on the same two maps (the `parity` object)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    O = oracle_py.Oracle()
    threads = O.set_threads(0)
    p = oracle_params(oracle_py, name)
    t0 = time.perf_counter()
    feat, pair, ref = oracle_sample_job(O, maps[:2], p)
    wall = time.perf_counter() - t0
    full = M * feat + P * pair
    cb = {"value": P / full, "unit": UNIT, "cores": threads, "kind": "port",
          "sample": f"maps 0-1 of the workload through the whole path (1 of {P} pairs), {wall:.1f} s on {threads} host threads (OpenMP inside each "
                    f"stage, the reference's sequential map / pair loops); per-map ({feat:.2f} s) and per-pair ({pair:.2f} s) times "
                    f"extrapolated to {M} maps / {P} pairs",
          "stage_seconds_sample": {k: round(v, 4) for k, v in ref["stage_times"].items()}}
    # parity: the same two maps through the CUDA path, stage outputs that the oracle reports compared bit for bit
    ctx, mm = job.ctx, job.mm
    dm = ctx.maps_upload(maps[:2])
    f = ctx.features_compute(dm, 0, 2, job.p)
    npt, nk, dim = f.sizes()
    ij = np.array([[0, 1]], np.int32)
    T, conf, stats = ctx.register_pairs(f, ij, job.p) if (nk > 0).all() else (np.zeros((0, 4, 4), np.float32), np.zeros(0), np.zeros((0, 4), np.int32))
    G = ctx.estimate_resident(dm, job.p)
    checks = {}
    want_T = np.asarray(ref["pair_T"], np.float32).reshape(-1, 4, 4)
    checks["pair_list"] = [list(map(int, r[:2])) for r in ref["pairs"]] == [[0, 1]][:len(T)]
    if len(T) and len(want_T):
        checks["pair_transform_bits"] = bool(np.array_equal(T[0].view(np.uint32), want_T[0].view(np.uint32)))
        checks["confidence_bits"] = bool(np.float64(conf[0]).view(np.uint64) == np.float64(ref["pair_conf"][0]).view(np.uint64))
        checks["n_correspondences"] = int(stats[0, 0]) == int(ref["pairs"][0][2])
        checks["n_ransac_inliers"] = int(stats[0, 1]) == int(ref["pairs"][0][3])
    checks["global_transforms_1e-5"] = bool(G.shape == np.asarray(ref["transforms"]).shape and
                                            np.allclose(G, ref["transforms"], rtol=0, atol=1e-5))
    parity = {"pairs": int(len(T)), "maps": 2, "bit_exact": bool(all(checks.values())), "checks": checks,
              "points_after_filter": [int(x) for x in npt], "keypoints": [int(x) for x in nk],
              "what": "maps 0-1 of this workload: CUDA path vs the CPU restatement (oracle/) — pairwise transform and confidence bit for "
                      "bit, correspondence and RANSAC inlier counts equal, global transforms within 1e-5"}
    f.free(); dm.free()
    return cb, parity


# ---------------------------------------------------------------------------------------------- GPU arm
class Job:
    """One rank of the job.  All the multi-GPU logic is inside libmm3d (csrc/dist.cu); this class only owns the buffers."""

    def __init__(self, args):
        import torch
        import mm3d_pkg
        self.torch = torch
        self.mm = mm3d_pkg.load()
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.phases_on = os.environ.get("MM3D_BENCH_PHASES") == "1"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=self.dev)
        self.ctx = self.mm.Context(self.local, stream=torch.cuda.current_stream().cuda_stream)
        self.comm = None
        if self.world > 1:
            # rank 0's ncclUniqueId travels through torch.distributed; the communicator itself belongs to the library
            idt = torch.zeros(self.mm.COMM_ID_BYTES, dtype=torch.uint8, device=self.dev)
            if self.rank == 0:
                idt.copy_(torch.frombuffer(bytearray(self.mm.comm_id()), dtype=torch.uint8))
            self.dist.broadcast(idt, 0)
            self.comm = self.ctx.comm_create(self.rank, self.world, bytes(idt.cpu().numpy().tobytes()))
        synth = synth_mod()
        self.name = args.workload
        self.cfg = dict(synth.CONFIGS[self.name])
        self.M = self.cfg["n_maps"]
        self.P = n_pairs_of(self.M)
        self.first, self.count = self.mm.dist_block(self.rank, self.world, self.M)
        t0 = time.perf_counter()
        self.maps, _ = synth.make_maps(**self.cfg, only=range(self.first, self.first + self.count))
        self.gen_s = time.perf_counter() - t0
        # pinned host copies of this rank's maps (e2e path) and resident device copies (value path)
        self.host = [None] * self.M
        for m in range(self.first, self.first + self.count):
            t = torch.empty((len(self.maps[m]), 4), dtype=torch.float32, pin_memory=True)
            t.numpy()[:] = self.maps[m]
            self.host[m] = t
        self.host_np = [t.numpy() if t is not None else None for t in self.host]
        self.resident = self.ctx.maps_upload([self.host_np[m] for m in range(self.first, self.first + self.count)])
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)
        self.h2d_bytes = sum(int(self.host[m].numel()) * 4 for m in range(self.first, self.first + self.count))
        self.phase_ms = {}
        if self.name != "c5":
            self.p = self.mm.default_params(**WORKLOADS[self.name]["params"])

    def step(self, from_host: bool):
        if self.world == 1:
            if from_host:
                return self.ctx.estimate_maps_transforms(self.host_np, self.p)
            if self.phases_on:
                G, st = self.ctx.estimate_resident(self.resident, self.p, stage_times=True)
                for k, v in st.items():
                    self.phase_ms[k] = self.phase_ms.get(k, 0.0) + v
                return G
            return self.ctx.estimate_resident(self.resident, self.p)
        if from_host:
            return self.ctx.estimate_maps_transforms_dist(self.comm, self.host_np, self.p)
        if self.phases_on:
            G, ph = self.ctx.estimate_resident_dist(self.comm, self.M, self.resident, self.p, phases=True)
            for k, v in ph.items():
                self.phase_ms[k] = self.phase_ms.get(k, 0.0) + v
            return G
        return self.ctx.estimate_resident_dist(self.comm, self.M, self.resident, self.p)

    def compose_step(self, from_host: bool, T):
        loc = slice(self.first, self.first + self.count)
        if from_host:
            return self.ctx.compose_maps_dist(self.comm, self.host_np[loc], T[loc], 0.05)
        return self.ctx.compose_resident_dist(self.comm, self.resident, T[loc], 0.05)

    def timed(self, steps: int, fn, profile: bool = False):
        torch, dist = self.torch, self.dist
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = self.ctx.launches
        if profile:
            self.ctx.profile_begin()
        w0 = time.perf_counter()
        ev0.record()
        out = None
        for _ in range(steps):
            self.flush.zero_()  # evict the previous step's working set from L2
            out = fn()
        ev1.record()
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        prof = self.ctx.profile_end() if profile else None
        if self.world > 1:
            dist.barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), self.ctx.launches - l0, prof, out, (w0, w1)


def settle(job, fn, seconds: float = 1.0):
    """Untimed steps (the same number on every rank) while the clock sampler starts up.  A step is collective at N > 1
    (NCCL inside the library), so EVERY rank runs the first step — a rank that timed it alone would wait for the others inside
    the step while they wait for its broadcast — and rank 0's duration decides how many more follow."""
    t0 = time.perf_counter()
    fn()
    dt = max(time.perf_counter() - t0, 1e-3)
    n = max(1, min(20, int(seconds / dt)))
    if job.world > 1:
        t = job.torch.tensor([n], dtype=job.torch.int64, device=job.dev)
        job.dist.broadcast(t, 0)
        n = int(t.item())
    for _ in range(n - 1):
        fn()


def roofline_of(prof, steps, peak, peak_src):
    """Dominant kernel of the profiled pass.  achieved = its algorithmic bytes / its CUDA-event time (per-launch averages)."""
    prof = sorted(prof, key=lambda k: -k["ms"])
    total_kernel_ms = sum(k["ms"] for k in prof)
    top = prof[0]
    roof = {"bound": "hbm", "kernel": top["kernel"], "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
            "peak_source": peak_src, "launches_per_step": top["launches"] / steps, "avg_launch_ms": top["ms"] / max(top["launches"], 1),
            "share_of_kernel_time": top["ms"] / max(total_kernel_ms, 1e-9),
            "note": "achieved = algorithmic bytes per launch (DESIGN.md §3, SURVEY.md 8d) / CUDA-event launch time, averaged over the "
                    "kernel's launches in the profiled pass"}
    if top["algorithmic_bytes"] > 0 and top["ms_annotated"] > 0:
        roof["achieved"] = top["algorithmic_bytes"] / (top["ms_annotated"] * 1e-3) / 1e9
        roof["frac"] = roof["achieved"] / peak
        roof["algorithmic_bytes_per_launch"] = top["algorithmic_bytes"] / top["launches"]
    # DRAM traffic of the same kernel from the committed ncu captures (profiles/r02_traffic.json, profiles/README.md).  ncu
    # replays every kernel ~40 times, so the captures ran an 8-map subset of the workload: the capture's DRAM bytes are
    # reported next to the algorithmic bytes of the SAME capture (like for like), and `traffic` — which would have to be per
    # launch of THIS run — stays null.
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as fh:
            tr = json.load(fh).get(top["kernel"])
        if tr:
            roof["traffic_capture"] = {"dram_bytes_per_launch": tr["dram_bytes_per_launch"],
                                       "algorithmic_bytes_per_launch": tr["algorithmic_bytes_per_launch"],
                                       "dram_over_algorithmic": tr["dram_bytes_per_launch"] / tr["algorithmic_bytes_per_launch"],
                                       "workload": tr["workload"], "ncu": tr.get("ncu"), "remark": tr.get("remark")}
    except Exception:
        pass
    kernels = [{"kernel": k["kernel"], "launches_per_step": k["launches"] / steps, "ms_per_step": k["ms"] / steps,
                "gbps": (k["algorithmic_bytes"] / (k["ms_annotated"] * 1e-3) / 1e9) if k["ms_annotated"] > 0 else None,
                "hbm_frac": (k["algorithmic_bytes"] / (k["ms_annotated"] * 1e-3) / 1e9 / peak) if k["ms_annotated"] > 0 else None}
               for k in prof[:16]]
    return roof, kernels


def run_gpu(args):
    job = Job(args)
    if args.workload == "c5":
        return run_gpu_compose(args, job)
    M, P = job.M, job.P
    W = max(args.warmup, 3)
    for _ in range(W):
        job.step(False)
    sampler = ClockSampler(job.local)
    if job.rank == 0:
        sampler.start()
    settle(job, lambda: job.step(False))  # nvidia-smi initialises NVML for ~0.5 s and stalls driver calls meanwhile: keep that out of the timed region
    job.phase_ms = {}
    ms, launches, _, out, (w0, w1) = job.timed(args.steps, lambda: job.step(False))
    if job.phases_on:
        print(f"[phases] rank {job.rank}: " + ", ".join(f"{k} {v / args.steps:.2f} ms" for k, v in job.phase_ms.items()) +
              f"; step {ms / args.steps:.2f} ms", file=sys.stderr, flush=True)
    clocks = sampler.stop(w0, w1) if job.rank == 0 else None
    # end to end from pinned host buffers (two warm host steps first: the stream-ordered pool grows to the host path's peak)
    job.step(True)
    job.step(True)
    ms_e2e, _, _, out_e2e, _ = job.timed(args.steps, lambda: job.step(True))
    # separate profiled pass (CUDA events around every launch) for the kernel table and the roofline
    psteps = min(args.steps, 3)
    _, _, prof, _, _ = job.timed(psteps, lambda: job.step(False), profile=True)
    if job.rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"transforms": out})  # every rank holds all transforms
    value = P * args.steps / (ms * 1e-3)
    e2e = P * args.steps / (ms_e2e * 1e-3)
    roof, kernels = roofline_of(prof, psteps, HBM_PEAK_GBS, HBM_PEAK_SOURCE)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": job.world, "steps": args.steps, "warmup": W,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(job.name, job.cfg), "seed": job.cfg["seed"],
                   "l2": f"256 MiB memset between steps (inputs are {M * job.cfg['n_points'] * 16 // 1000000} MB)",
                   "parallelism": "single GPU" if job.world == 1 else
                   f"maps and pairs sharded over {job.world} ranks inside libmm3d (NCCL feature exchange, LPT pair plan)"},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(job.h2d_bytes), "d2h_bytes_per_step": int(M * 64),
                "ms_per_step": ms_e2e / args.steps, "same_result_as_resident": bool(np.array_equal(out, out_e2e))},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "kernels": kernels,
        "transforms_estimated": int(len(out)),
    }
    if job.world == 1 and not args.no_cpu_baseline:
        cb, parity = cpu_baseline_and_parity(job, job.maps, job.name, M, P)
        line["cpu_baseline"] = cb
        line["parity"] = parity
    else:
        line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "timed at N=1 only"}
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()
    if job.comm:
        job.comm.free()
    if job.world > 1:
        job.dist.destroy_process_group()


def run_gpu_compose(args, job):
    """c5: composeMaps (map_merging.cpp:277-305) of 4 x 10M points at 0.05 m, maps sharded over the ranks."""
    M = job.M
    n_in = M * job.cfg["n_points"]
    T = np.stack([np.eye(4, dtype=np.float32)] * M)  # the maps are composed in their own frames: the voxel work is the same
    W = max(args.warmup, 3)
    for _ in range(W):
        job.compose_step(False, T)
    sampler = ClockSampler(job.local)
    if job.rank == 0:
        sampler.start()
    settle(job, lambda: job.compose_step(False, T))
    ms, launches, _, out, (w0, w1) = job.timed(args.steps, lambda: job.compose_step(False, T))
    clocks = sampler.stop(w0, w1) if job.rank == 0 else None
    job.compose_step(True, T)
    ms_e2e, _, _, _, _ = job.timed(args.steps, lambda: job.compose_step(True, T))
    psteps = min(args.steps, 3)
    _, _, prof, _, _ = job.timed(psteps, lambda: job.compose_step(False, T), profile=True)
    n_out = job.torch.tensor([len(out)], dtype=job.torch.int64, device=job.dev)
    if job.world > 1:
        job.dist.all_reduce(n_out)
    if args.dump_outputs:
        # each rank returns its own key range of the composed map
        name = "composed_points" if job.world == 1 else f"composed_points_rank{job.rank}"
        dump_outputs(args.dump_outputs, {name: out}, DUMP_BYTES // job.world)
    if job.rank != 0:
        return
    peak = HBM_PEAK_GBS
    roof, kernels = roofline_of(prof, psteps, peak, HBM_PEAK_SOURCE)
    # whole-step roofline: every input point read once, transformed copy written and read once, output written once
    step_bytes = 48.0 * n_in / job.world + 16.0 * len(out)
    kernel_ms = sum(k["ms"] for k in prof) / psteps
    roof["step"] = {"algorithmic_bytes_per_rank": step_bytes, "kernel_ms_per_step": kernel_ms,
                    "achieved_gbps": step_bytes / (kernel_ms * 1e-3) / 1e9, "frac": step_bytes / (kernel_ms * 1e-3) / 1e9 / peak}
    line = {"metric": "compose_maps_points_per_sec", "value": n_in * args.steps / (ms * 1e-3), "unit": "points/s", "n_gpus": job.world,
            "steps": args.steps, "warmup": W, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"c5: composeMaps of {M} maps x {job.cfg['n_points']} pts at output_resolution 0.05",
                       "seed": job.cfg["seed"], "l2": "256 MiB memset between steps (inputs are 640 MB)",
                       "parallelism": "single GPU" if job.world == 1 else f"maps sharded over {job.world} ranks, all-to-all of raw points by voxel key range",
                       "output_points": int(n_out.item())},
            "e2e": {"value": n_in * args.steps / (ms_e2e * 1e-3), "unit": "points/s", "h2d_bytes_per_step": int(job.h2d_bytes),
                    "d2h_bytes_per_step": int(len(out) * 16), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "kernels": kernels,
            "cpu_baseline": {"value": None, "unit": "points/s", "cores": 0, "kind": "port", "sample": "see --impl reference --workload c5"}}
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()
    if job.comm:
        job.comm.free()
    if job.world > 1:
        job.dist.destroy_process_group()


_OUT = sys.stdout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mm3d", choices=["mm3d", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(set(WORKLOADS) | {"c5"}))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="save what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    # stdout carries exactly one JSON line: keep a private handle to it and point fd 1 at stderr, so that anything a
    # library writes to stdout (NCCL prints its version banner there) cannot get in front of the line
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
