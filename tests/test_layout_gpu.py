"""Point clouds in the caller's record layout (mm3d_layout): the GPU conversion against the packed path, bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "map-merge_b200")
ERR_ARG = -3


def to_records(pts, layout, rng=None):
    """float32[n, 4] (x, y, z, rgba bits) -> uint8[n, point_step]; bytes outside the four fields are random garbage."""
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
    n, step = len(pts), layout.point_step
    rng = rng or np.random.default_rng(0)
    rec = rng.integers(0, 256, size=(n, step), dtype=np.uint8)
    w = rec.view(np.uint32)
    src = pts.view(np.uint32)
    for k, off in enumerate((layout.offset_x, layout.offset_y, layout.offset_z, layout.offset_rgba)):
        w[:, off // 4] = src[:, k]
    return rec


def expected_records(pts, layout):
    """What a composed record must hold: the layout's template with x, y, z and rgba written over it."""
    n = len(pts)
    w = np.tile(np.frombuffer(layout.template_bytes, np.uint32), (n, 1))
    src = np.ascontiguousarray(pts, np.float32).view(np.uint32)
    for k, off in enumerate((layout.offset_x, layout.offset_y, layout.offset_z, layout.offset_rgba)):
        w[:, off // 4] = src[:, k]
    return w


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def scrambled(mm):
    return mm.Layout(48, 20, 8, 36, 0, np.random.default_rng(7).integers(0, 256, 48, dtype=np.uint8).tobytes())


@pytest.mark.parametrize("cfg", ["tiny", "small"])
@pytest.mark.parametrize("desc", ["FPFH", "PFHRGB"])
def test_estimate_layout_matches_packed(ctx, mm, synth, scrambled, cfg, desc):
    maps, _ = synth.make_maps(**synth.CONFIGS[cfg])
    p = mm.default_params(descriptor_type=desc)
    want = ctx.estimate_maps_transforms(maps, p)
    assert len(want) == len(maps)
    for layout in (mm.PCL_XYZRGB, scrambled):
        got = ctx.estimate_maps_transforms_layout([to_records(m, layout) for m in maps], layout, p)
        assert np.array_equal(bits(got), bits(want)), (cfg, desc, layout.point_step)


def _with_special_values(m, seed):
    """A copy with NaNs (two payloads), infinities and negative zeros in place of some coordinates."""
    m = m.copy()
    rng = np.random.default_rng(seed)
    w = m.view(np.uint32)
    idx = rng.choice(len(m), 40, replace=False)
    w[idx[0:10], 0] = 0x7fc00001
    w[idx[10:20], 1] = 0xffa5a5a5
    m[idx[20:25], 2] = np.inf
    m[idx[25:30], 0] = -np.inf
    m[idx[30:40], 0:3] = -0.0
    return m


def test_compose_layout_staging(ctx, mm, synth, scrambled):
    """4 x 2M points (several staging slots each, not whole slots), a null, an empty and a one-point map in the middle,
    non-finite and -0.0 coordinates; resolution 1e-4 takes the overflow-guard path (the output is the concatenation)."""
    maps, truth = synth.make_maps(seed=5, n_maps=4, n_points=2_000_000, size_x=28.0, size_y=20.0, rooms_x=2, rooms_y=2)
    maps = [_with_special_values(m, i) for i, m in enumerate(maps)]
    clouds = [maps[0], maps[1], None, np.zeros((0, 4), np.float32), maps[2][:1].copy(), maps[2], maps[3]]
    T = np.stack([np.linalg.inv(truth[0]) @ truth[i] for i in (0, 1, 0, 0, 2, 2, 3)]).astype(np.float32)
    pcl = mm.PCL_XYZRGB
    recs = [to_records(c, pcl) if c is not None else None for c in clouds]
    for res in (0.05, 0.2, 1e-4):
        want = ctx.compose_maps(clouds, T, res)
        got = ctx.compose_maps_layout(recs, T, res, pcl, pcl)
        assert got.shape == (len(want), 32), res
        assert np.array_equal(got.view(np.uint32), expected_records(want, pcl)), res
        if res == 0.2:  # another output layout, garbage template
            got48 = ctx.compose_maps_layout(recs, T, res, pcl, scrambled)
            assert np.array_equal(got48.view(np.uint32), expected_records(want, scrambled))
            recs48 = [to_records(c, scrambled) if c is not None else None for c in clouds]
            assert np.array_equal(ctx.compose_maps_layout(recs48, T, res, scrambled, pcl).view(np.uint32), got.view(np.uint32))
    assert ctx.compose_maps_layout([], [], 0.05, pcl, pcl) is None
    empty = ctx.compose_maps_layout([None, np.zeros((0, 32), np.uint8)], np.stack([np.eye(4)] * 2), 0.05, pcl, pcl)
    assert empty.shape == (0, 32)


def test_malformed_layouts_launch_nothing(ctx, mm, tiny_maps):
    maps, _ = tiny_maps
    p = mm.default_params(descriptor_type="FPFH")
    T = np.stack([np.eye(4)] * len(maps)).astype(np.float32)
    bad = [mm.Layout(12, 0, 4, 8, 8), mm.Layout(32, 2, 4, 8, 16), mm.Layout(32, 0, 4, 8, 32), mm.Layout(20, 0, 4, 8, 18),
           mm.Layout(32, 0, -4, 8, 16), mm.Layout(18, 0, 4, 8, 12)]
    for layout in bad:
        recs = [np.zeros((len(m), layout.point_step), np.uint8) for m in maps]
        l0 = ctx.launches
        with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
            ctx.estimate_maps_transforms_layout(recs, layout, p)
        with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
            ctx.compose_maps_layout(recs, T, 0.05, layout, mm.PCL_XYZRGB)
        good = [to_records(m, mm.PCL_XYZRGB) for m in maps]
        with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
            ctx.compose_maps_layout(good, T, 0.05, mm.PCL_XYZRGB, layout)
        with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
            ctx.maps_upload_layout(recs, layout)
        assert ctx.launches == l0, layout.point_step
    # a NULL layout, through the C ABI directly
    L = ctx.L
    arrs, ptrs, ns = ctx._record_args([to_records(m, mm.PCL_XYZRGB) for m in maps], mm.PCL_XYZRGB)
    out = np.zeros((len(maps), 16), np.float32); no = C.c_int(); h = C.c_void_p(); o = C.c_void_p(); n = C.c_uint64()
    l0 = ctx.launches
    assert L.mm3d_estimate_maps_transforms_layout(ctx.h, len(maps), ptrs, ns, None, C.byref(p), out.ctypes.data_as(C.POINTER(C.c_float)),
                                                  C.byref(no)) == ERR_ARG
    assert L.mm3d_maps_upload_layout(ctx.h, len(maps), ptrs, ns, None, C.byref(h)) == ERR_ARG
    assert L.mm3d_compose_maps_layout(ctx.h, len(maps), ptrs, ns, None, len(T), T.ctypes.data_as(C.POINTER(C.c_float)), C.c_double(0.05),
                                      C.byref(mm.PCL_XYZRGB), C.byref(o), C.byref(n)) == ERR_ARG
    assert ctx.launches == l0


def test_conversion_runs_on_the_gpu(ctx, mm, tiny_maps):
    torch = pytest.importorskip("torch")
    maps, _ = tiny_maps
    p = mm.default_params(descriptor_type="FPFH")
    pcl = mm.PCL_XYZRGB
    recs = [to_records(m, pcl) for m in maps]
    ctx.profile_begin()
    pageable = ctx.estimate_maps_transforms_layout(recs, pcl, p)
    prof = ctx.profile_end()
    unpack = [k for k in prof if k["kernel"].startswith("unpack_records")]
    assert unpack, [k["kernel"] for k in prof]
    assert sum(k["algorithmic_bytes"] for k in unpack) == sum(len(m) for m in maps) * (32 + 16)
    pinned = []
    for r in recs:
        t = torch.empty(r.shape, dtype=torch.uint8, pin_memory=True)
        t.numpy()[:] = r
        pinned.append(t)
    got = ctx.estimate_maps_transforms_layout([t.numpy() for t in pinned], pcl, p)
    assert np.array_equal(bits(got), bits(pageable))
    assert np.array_equal(bits(pageable), bits(ctx.estimate_maps_transforms(maps, p)))


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_two_gpus_layout_matches_one_gpu_packed(mm, small_maps):
    maps, truth = small_maps
    p = mm.default_params(descriptor_type="FPFH")
    pcl = mm.PCL_XYZRGB
    one = mm.Context(0)
    two = mm.Context(devices=[0, 1])
    recs = [to_records(m, pcl) for m in maps]
    assert np.array_equal(bits(two.estimate_maps_transforms_layout(recs, pcl, p)), bits(one.estimate_maps_transforms(maps, p)))
    T = np.stack([np.linalg.inv(truth[0]) @ t for t in truth]).astype(np.float32)
    for res in (0.05, 1e-4):
        want = one.compose_maps(maps, T, res)
        got = two.compose_maps_layout(recs, T, res, pcl, pcl)
        assert np.array_equal(got.view(np.uint32), expected_records(want, pcl)), res
    one.close(); two.close()


@pytest.mark.parametrize("env", [{"MM3D_DEVICE": "0"}, {}], ids=["device0", "default_devices"])
def test_cpp_api_on_pcl_points(tmp_path, ctx, mm, small_maps, env):
    """map_merge_3d::estimateMapsTransforms and composeMaps (host/shim.cpp) against the packed C ABI."""
    subprocess.check_call(["make", "-C", PKG, "tools"], stdout=subprocess.DEVNULL)
    maps, _ = small_maps
    maps = [maps[0], np.zeros((0, 4), np.float32), maps[1], maps[2]]
    files = []
    for i, m in enumerate(maps):
        f = tmp_path / f"map{i}.bin"
        f.write_bytes(np.ascontiguousarray(m, np.float32).tobytes())
        files.append(str(f))
    run_env = {k: v for k, v in os.environ.items() if k not in ("MM3D_DEVICE", "MM3D_DEVICES")}
    run_env.update(env)
    r = subprocess.run([os.path.join(PKG, "build", "test_shim_layout"), str(tmp_path), "FPFH", "0.05"] + files, capture_output=True, text=True,
                       env=run_env)
    assert r.returncode == 0, r.stdout + r.stderr
    T = np.fromfile(tmp_path / "transforms.bin", np.float32).reshape(-1, 4, 4).transpose(0, 2, 1)
    want_T = ctx.estimate_maps_transforms(maps, mm.default_params(descriptor_type="FPFH"))
    assert T.shape == want_T.shape and np.array_equal(bits(T), bits(want_T))
    got = np.fromfile(tmp_path / "composed.bin", np.uint32).reshape(-1, 8)
    want = ctx.compose_maps(maps, want_T, 0.05)
    assert np.array_equal(got, expected_records(want, mm.PCL_XYZRGB))
