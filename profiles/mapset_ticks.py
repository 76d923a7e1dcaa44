"""The map set (mm3d_mapset) on a node-like timeline, against the stateless calls, on one GPU.

Config 3 (32 x 1M points, SIFT + FPFH as in bench.py), records in the pcl::PointXYZRGB layout (32 bytes a point):
  1  stateless       mm3d_estimate_maps_transforms_layout on all 32 maps
  2  first estimate  a new map set: update all 32 slots, estimate (every map and pair computed)
  3  one map         slot 17 replaced (alternately by a map drawn from another seed and by the original), estimate
  4  unchanged       all 32 maps sent again as they are, estimate
Config 5 (4 x 10M points, 0.05 m): mm3d_compose_maps_layout against mm3d_mapset_compose, PCL records in and out.

Each step runs once to warm up, then reps times alternating with the stateless call; times are a host clock around calls
that end in a device synchronise (median, min, max).  Every map-set result is compared bit for bit with the stateless
call on the same clouds.  One extra profiled pass (CUDA events per kernel, not part of the timings) gives the kernel time
of step 3's estimate and of the change check in step 4's update.  Needs a GPU and a prior __graft_entry__.build().

  python profiles/mapset_ticks.py --out <dir>/r04_mapset_ticks.json [--reps 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBM_PEAK_GBS = 6453.7  # bench.py's roofline peak
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    first = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = first.partition(",")
    return {"name": name.strip() or None, "power_limit": power.strip() or None}


def stats(v):
    return {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "runs_ms": v}


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t0) * 1e3


def to_records(pts, layout):
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
    w = np.tile(np.frombuffer(layout.template_bytes, np.uint32), (len(pts), 1))
    src = pts.view(np.uint32)
    for k, off in enumerate((layout.offset_x, layout.offset_y, layout.offset_z, layout.offset_rgba)):
        w[:, off // 4] = src[:, k]
    return np.ascontiguousarray(w).view(np.uint8)


def same(a, b):
    return a is not None and b is not None and a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint8),
                                                                                   np.ascontiguousarray(b).view(np.uint8))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import mm3d_pkg
    mm = mm3d_pkg.load()
    synth = mm3d_pkg.load_synth()
    ctx = mm.Context(0)
    pcl = mm.PCL_XYZRGB
    res = {"card": card(), "reps": args.reps, "layout": "pcl::PointXYZRGB (32 bytes a point)", "hbm_peak_gbs": HBM_PEAK_GBS}

    # ---- config 3 estimate timeline
    cfg = dict(synth.CONFIGS["c3"])
    maps, _ = synth.make_maps(**cfg)
    recs = [to_records(m, pcl) for m in maps]
    del maps
    alt17 = to_records(synth.make_maps(**dict(cfg, seed=cfg["seed"] + 100), only=[17])[0][17], pcl)
    orig17 = recs[17]
    p = mm.default_params(descriptor_type="FPFH")
    everything = {i: r for i, r in enumerate(recs)}

    def stateless():
        return ctx.estimate_maps_transforms_layout(recs, pcl, p)

    ok = {}
    t_stateless, t_first_update, t_first_est, t_one_update, t_one_est, t_same_update, t_same_est = [], [], [], [], [], [], []
    work = {}
    want = stateless()  # warm-up
    ms = ctx.mapset()
    ms.update(everything, pcl)
    ms.estimate(p)  # warm-up of the map-set path
    ok["first"] = ok["one_map"] = ok["unchanged"] = True
    launches_unchanged = []
    for r in range(args.reps + 1):
        warm = r == 0
        want, ts = timed(stateless)
        fresh = ctx.mapset()
        _, tu = timed(lambda: fresh.update(everything, pcl))
        (got, w), te = timed(lambda: fresh.estimate(p, work=True))
        fresh.free()
        ok["first"] &= same(got, want)
        work["first"] = w
        if not warm:
            t_stateless.append(ts); t_first_update.append(tu); t_first_est.append(te)
    for r in range(args.reps + 1):
        warm = r == 0
        recs[17] = alt17 if r % 2 == 0 else orig17
        want, _ = timed(stateless)
        ch, tu = timed(lambda: ms.update({17: recs[17]}, pcl))
        (got, w), te = timed(lambda: ms.estimate(p, work=True))
        ok["one_map"] &= same(got, want) and ch == [True]
        work["one_map"] = w
        if not warm:
            t_one_update.append(tu); t_one_est.append(te)
    everything = {i: r for i, r in enumerate(recs)}
    want = stateless()
    for r in range(args.reps + 1):
        warm = r == 0
        ch, tu = timed(lambda: ms.update(everything, pcl))
        l0 = ctx.launches
        (got, w), te = timed(lambda: ms.estimate(p, work=True))
        launches_unchanged.append(ctx.launches - l0)
        ok["unchanged"] &= same(got, want) and ch == [False] * len(recs)
        work["unchanged"] = w
        if not warm:
            t_same_update.append(tu); t_same_est.append(te)

    # profiled pass (CUDA events per kernel): step 3 and step 4's update
    recs[17] = alt17 if recs[17] is orig17 else orig17
    ms.update({17: recs[17]}, pcl)
    ctx.profile_begin()
    ms.estimate(p)
    prof3 = ctx.profile_end()
    ctx.profile_begin()
    ms.update({i: r for i, r in enumerate(recs)}, pcl)
    prof4 = ctx.profile_end()
    ok["one_map"] &= same(ms.estimate(p), stateless())
    ms.free()
    cmp = [k for k in prof4 if k["kernel"] == "mapset_compare_kernel"]
    cmp_ms = sum(k["ms"] for k in cmp)
    cmp_bytes = sum(k["algorithmic_bytes"] for k in cmp)
    res["c3"] = {
        "maps": 32, "points_per_map": 1_000_000, "pairs": 496, "params": "SIFT + FPFH, MATCHING + ICP (bench.py config 3)",
        "1_stateless_estimate": stats(t_stateless),
        "2_first_mapset": {"update": stats(t_first_update), "estimate": stats(t_first_est), "work": work["first"]},
        "3_one_map_replaced": {"update": stats(t_one_update), "estimate": stats(t_one_est), "work": work["one_map"],
                               "estimate_kernel_ms": sum(k["ms"] for k in prof3),
                               "estimate_kernel_launches": sum(k["launches"] for k in prof3)},
        "4_all_sent_unchanged": {"update": stats(t_same_update), "estimate": stats(t_same_est), "work": work["unchanged"],
                                 "estimate_kernel_launches": launches_unchanged,
                                 "compare_kernel": {"launches": sum(k["launches"] for k in cmp), "ms": cmp_ms, "algorithmic_bytes": cmp_bytes,
                                                    "gbs": cmp_bytes / (cmp_ms * 1e-3) / 1e9 if cmp_ms > 0 else None}},
        "identical_bits": ok,
    }
    if res["c3"]["4_all_sent_unchanged"]["compare_kernel"]["gbs"]:
        res["c3"]["4_all_sent_unchanged"]["compare_kernel"]["hbm_frac"] = res["c3"]["4_all_sent_unchanged"]["compare_kernel"]["gbs"] / HBM_PEAK_GBS
    del recs, everything, alt17, orig17

    # ---- config 5 compose
    cfg5 = dict(synth.CONFIGS["c5"])
    maps5, truth5 = synth.make_maps(**cfg5)
    recs5 = [to_records(m, pcl) for m in maps5]
    del maps5
    T = np.stack([np.linalg.inv(truth5[0]) @ t for t in truth5]).astype(np.float32)
    res5 = 0.05
    ms5 = ctx.mapset()
    ms5.update({i: r for i, r in enumerate(recs5)}, pcl)
    t_a, t_b, ok5 = [], [], True
    n_out = None
    for r in range(args.reps + 1):
        a, ta = timed(lambda: ctx.compose_maps_layout(recs5, T, res5, pcl, pcl))
        b, tb = timed(lambda: ms5.compose(T, res5, pcl))
        ok5 &= same(a, b)
        n_out = len(b)
        del a, b
        if r:
            t_a.append(ta); t_b.append(tb)
    ms5.free()
    res["c5_compose"] = {"maps": 4, "points_per_map": 10_000_000, "resolution": res5, "output_points": n_out,
                         "stateless_compose_maps_layout": stats(t_a), "mapset_compose": stats(t_b), "identical_bits": ok5}
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res)[:4000])
    good = all(ok.values()) and ok5
    print("identical bits at every step:", good)
    return 0 if good else 1


if __name__ == "__main__":
    sys.exit(main())
