"""Every entry point of estimateMapsTransforms and composeMaps that runs on one GPU returns the same bits: the stateless
calls from host buffers (packed and in a caller's layout), the resident maps, the one-rank `_dist` calls and the map set.
The `_dist` calls are what the multi-GPU benchmark runs, so the single-GPU tests cover its driver through them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
WORLD = dict(n_maps=6, n_points=100_000, size_x=14.0, size_y=8.0, rooms_x=2, rooms_y=1, window_frac=0.6)


@pytest.fixture(scope="module")
def worlds(synth, tiny_maps):
    six, truth = synth.make_maps(seed=31, **WORLD)
    return {"tiny": tiny_maps, "six": (six, truth)}


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(bits(a), bits(b))


def same_up_to_nan_payload(a, b):
    """bit equality, except that any two NaNs are equal (the oracle's x86 arithmetic keeps other NaN payloads)"""
    if a.shape != b.shape:
        return False
    both_nan = np.isnan(a) & np.isnan(b)
    return np.array_equal(np.where(both_nan, 0, bits(a)), np.where(both_nan, 0, bits(b)))


def to_records(pts, layout):
    """float32[n, 4] -> uint8[n, point_step] records in `layout`; the other bytes hold the layout's template"""
    if pts is None:
        return None
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
    w = np.tile(np.frombuffer(layout.template_bytes, np.uint32), (len(pts), 1))
    src = pts.view(np.uint32)
    for k, off in enumerate((layout.offset_x, layout.offset_y, layout.offset_z, layout.offset_rgba)):
        w[:, off // 4] = src[:, k]
    return np.ascontiguousarray(w).view(np.uint8)


def estimates(ctx, mm, clouds, p):
    """name -> transforms of every one-GPU estimateMapsTransforms entry point"""
    out = {"estimate_maps_transforms": ctx.estimate_maps_transforms(clouds, p),
           "estimate_maps_transforms_layout": ctx.estimate_maps_transforms_layout([to_records(c, mm.PCL_XYZRGB) for c in clouds],
                                                                                  mm.PCL_XYZRGB, p),
           "estimate_maps_transforms_dist": ctx.estimate_maps_transforms_dist(None, clouds, p)}
    maps = ctx.maps_upload(clouds)
    out["estimate_resident"] = ctx.estimate_resident(maps, p)
    out["estimate_resident(stage_times)"] = ctx.estimate_resident(maps, p, stage_times=True)[0]
    out["estimate_resident_dist"] = ctx.estimate_resident_dist(None, len(clouds), maps, p)
    maps.free()
    ms = ctx.mapset()
    ms.update({i: c for i, c in enumerate(clouds)})
    out["mapset"] = ms.estimate(p)
    ms.free()
    return out


@pytest.mark.parametrize("method", ["MATCHING", "SAC_IA"])
@pytest.mark.parametrize("world", ["tiny", "six"])
def test_estimate_entry_points_agree(ctx, mm, worlds, world, method):
    clouds, _ = worlds[world]
    p = mm.default_params(descriptor_type="FPFH", estimation_method=method)
    got = estimates(ctx, mm, list(clouds), p)
    want = got.pop("estimate_maps_transforms")
    assert want.shape == (len(clouds), 4, 4)
    for name, T in got.items():
        assert same_bits(T, want), name


def composes(ctx, mm, clouds, T, res):
    """name -> composed points of every one-GPU composeMaps entry point"""
    out = {"compose_maps": ctx.compose_maps(clouds, T, res),
           "compose_maps_layout": ctx.compose_maps_layout([to_records(c, mm.PCL_XYZRGB) for c in clouds], T, res, mm.PCL_XYZRGB,
                                                          mm.PACKED).view(np.float32).reshape(-1, 4),
           "compose_maps_dist": ctx.compose_maps_dist(None, clouds, T, res)}
    maps = ctx.maps_upload(clouds)
    out["compose_resident_dist"] = ctx.compose_resident_dist(None, maps, T, res)
    maps.free()
    ms = ctx.mapset()
    ms.update({i: c for i, c in enumerate(clouds)})
    out["mapset"] = ms.compose(T, res)
    ms.free()
    return out


def compose_case(worlds, case):
    """clouds and transforms of a composeMaps case; every map but the first stresses one of composeMaps' rules"""
    six, truth = worlds["six"]
    T = np.stack([np.linalg.inv(truth[0]) @ t for t in truth]).astype(np.float32)
    rng = np.random.default_rng(7)
    nan_some = six[4].copy()
    rows = rng.choice(len(nan_some), len(nan_some) // 50, replace=False)
    nan_some[rows[0::3], 0] = np.nan
    nan_some[rows[1::3], 2] = np.inf
    nan_some[rows[2::3], 1] = np.nan
    all_nan = np.full((5000, 4), np.nan, np.float32)
    all_nan[:, 3] = 1.0
    if case == "mixed":
        clouds = [six[0], six[1], np.zeros((0, 4), np.float32), None, nan_some, six[5], all_nan]
        T = np.concatenate([T, T[:1]])
        T[1] = 0.0  # a zero transform: the map is left out
        return clouds, T
    if case == "all_nan":  # nothing finite is left after the skip rule
        return [all_nan, None, np.zeros((0, 4), np.float32), six[2]], np.stack([T[0], T[1], T[2], np.zeros((4, 4), np.float32)])
    if case == "far":  # 4e9 voxels along x at 1e-4 m, past the guard's 3e9 cast check; dx * dy * dz stays within int64
        far = np.array([[0, 0, 0, 1], [4e5, 0, 0, 1], [0, 1, 0, 1]], np.float32)
        return [far, six[0]], np.stack([np.eye(4, dtype=np.float32), np.zeros((4, 4), np.float32)])
    raise ValueError(case)


@pytest.mark.parametrize("res", [0.05, 0.2, 1e-4, 0.0])
@pytest.mark.parametrize("case", ["mixed", "all_nan", "far"])
def test_compose_entry_points_agree(ctx, mm, oracle, worlds, case, res):
    clouds, T = compose_case(worlds, case)
    got = composes(ctx, mm, clouds, T, res)
    want = got.pop("compose_maps")
    for name, pts in got.items():
        assert same_bits(pts, want), name
    ref = oracle.compose_maps([c if c is not None else np.zeros((0, 4), np.float32) for c in clouds], T, res)
    assert same_up_to_nan_payload(want, ref)
    kept = sum(len(c) for c, t in zip(clouds, T) if c is not None and np.abs(t).max() > 1e-5)
    if res <= 1e-4 and case != "all_nan":  # pcl::VoxelGrid's overflow guard: the plain concatenation of the kept maps
        assert len(want) == kept
    if case == "all_nan":  # non-finite points have no voxel and are no reason to pass the cloud through, at any leaf size
        assert len(want) == 0


def test_one_rank_calls_launch_the_same_kernels(ctx, mm, worlds):
    """The one-rank `_dist` calls and the map set do the device work of the ordinary calls, kernel for kernel."""
    clouds, _ = worlds["tiny"]
    p = mm.default_params(descriptor_type="FPFH")
    maps = ctx.maps_upload(clouds)

    def launches(fn):
        l0 = ctx.launches
        fn()
        return ctx.launches - l0

    est = {launches(lambda: ctx.estimate_maps_transforms(clouds, p)), launches(lambda: ctx.estimate_maps_transforms_dist(None, clouds, p)),
           launches(lambda: ctx.estimate_resident(maps, p)), launches(lambda: ctx.estimate_resident_dist(None, len(clouds), maps, p))}
    assert len(est) == 1 and est.pop() > 50
    six, truth = worlds["six"]
    T = np.stack([np.linalg.inv(truth[0]) @ t for t in truth]).astype(np.float32)
    big = ctx.maps_upload(six)
    ms = ctx.mapset()
    ms.update({i: c for i, c in enumerate(six)})
    comp = {launches(lambda: ctx.compose_maps(six, T, 0.05)), launches(lambda: ctx.compose_maps_dist(None, six, T, 0.05)),
            launches(lambda: ctx.compose_resident_dist(None, big, T, 0.05)), launches(lambda: ms.compose(T, 0.05))}
    assert len(comp) == 1
    ms.free()
    big.free()
    maps.free()
