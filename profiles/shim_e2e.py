"""End-to-end cost of the C++ API (host/shim.cpp) against the C ABI, on config 3 (estimateMapsTransforms, 32 x 1M points)
and config 5 (composeMaps, 4 x 10M points at 0.05 m).

Builds profiles/shim_e2e_harness.cpp into a temporary directory (never into the tree), writes the seeded synthetic maps
there, and runs the harness once per workload; each run alternates three variants after one warm-up call each:
  a  the previous shim path: single-thread pack() into pageable vectors, the packed C ABI call (+ unpack() for composeMaps)
  b  map_merge_3d::estimateMapsTransforms / composeMaps as they are now (records handed over as they lie, converted on the GPU)
  c  the C ABI from pinned, pre-packed points (bench.py's e2e path)
A third harness run breaks the staged upload inside b down into host copy, host-to-device copy and unpack kernel time.
Times are a host clock around calls that end in a device synchronise.  Needs a GPU and a prior __graft_entry__.build().

  python profiles/shim_e2e.py --out <dir>/shim_e2e.json [--reps 5]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "map-merge_b200")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
HBM_PEAK_GBS = 6453.7  # bench.py's roofline peak
sys.path.insert(0, ROOT)


def stats(v):
    return {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "runs_ms": v}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    first = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    name, _, power = first.partition(",")
    return {"name": name.strip() or None, "power_limit": power.strip() or None}


def write_maps(d, tag, maps):
    files = []
    for i, m in enumerate(maps):
        f = os.path.join(d, f"{tag}_{i}.bin")
        np.ascontiguousarray(m, np.float32).tofile(f)
        files.append(f)
    return files


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import mm3d_pkg
    synth = mm3d_pkg.load_synth()
    env = dict(os.environ, MM3D_DEVICE="0")  # the shim on one GPU, like the C ABI context it is compared with
    env.pop("MM3D_DEVICES", None)
    res = {"card": card(), "reps": args.reps, "hbm_peak_gbs": HBM_PEAK_GBS}
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "shim_e2e_harness")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(PKG, "host"),
                               "-I" + os.path.join(CUDA, "include"), "-o", exe, os.path.join(ROOT, "profiles", "shim_e2e_harness.cpp"),
                               "-L" + PKG, "-lmm3d_shim", "-lmm3d", "-L" + os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + PKG])

        def harness(mode, files, extra_env=None):
            r = subprocess.run([exe, mode, str(args.reps)] + files, capture_output=True, text=True, env=dict(env, **(extra_env or {})))
            if r.returncode != 0:
                raise SystemExit(f"harness {mode} failed ({r.returncode}): {r.stdout[-2000:]} {r.stderr[-2000:]}")
            return json.loads(r.stdout.strip().splitlines()[-1]), r.stderr

        c3, _ = synth.make_maps(**synth.CONFIGS["c3"])
        f3 = write_maps(d, "c3", c3)
        del c3
        est, _ = harness("estimate", f3)
        up, trace = harness("upload", f3, {"MM3D_HOST_TRACE": "1"})
        c5, _ = synth.make_maps(**synth.CONFIGS["c5"])
        f5 = write_maps(d, "c5", c5)
        del c5
        comp, _ = harness("compose", f5)
    for name, r in (("c3_estimate", est), ("c5_compose", comp)):
        r["a"], r["b"], r["c"] = stats(r.pop("a_ms")), stats(r.pop("b_ms")), stats(r.pop("c_ms"))
        r["b_over_c"] = r["b"]["median_ms"] / r["c"]["median_ms"]
        r["b_over_a"] = r["b"]["median_ms"] / r["a"]["median_ms"]
        res[name] = r
    # breakdown of b's staged upload on config 3
    copies = [(float(a), float(b), int(t)) for a, b, t in
              re.findall(r"\[mm3d staging\].*enqueue wall ([\d.]+) ms, host copy ([\d.]+) ms.*over (\d+) threads", trace)]
    unpack = [k for k in up["profile"] if k["kernel"].startswith("unpack_records")]
    k_ms = sum(k["ms"] for k in unpack)
    k_bytes = sum(k["algorithmic_bytes"] for k in unpack)
    gbs = k_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None
    res["c3_upload_breakdown"] = {
        "what": "mm3d_maps_upload_layout of config 3's 32 x 1M pcl::PointXYZRGB records from pageable memory (the upload inside b)",
        "record_bytes": up["record_bytes"],
        "upload": stats(up["upload_ms"]),
        "host_copy_ms_per_thread": [c / t for _, c, t in copies[1:args.reps + 1]],
        "host_copy_threads": copies[-1][2] if copies else None,
        "h2d_copy_ms": stats(up["h2d_copy_ms"]),
        "h2d_copy_gbs": up["record_bytes"] / (statistics.median(up["h2d_copy_ms"]) * 1e-3) / 1e9,
        "unpack_kernel": {"launches": sum(k["launches"] for k in unpack), "ms": k_ms, "algorithmic_bytes": k_bytes, "gbs": gbs,
                          "hbm_frac": gbs / HBM_PEAK_GBS if gbs else None},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk not in ("runs_ms",)}) for k, v in res.items()}))
    ok = est["bit_identical"] and comp["bit_identical"]
    print("bit-identical a == b == c:", ok)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
