"""The map set (mm3d_mapset): after every update sequence its estimate and compose equal the stateless calls on the slots'
current clouds, bit for bit, while it recomputes only the maps and pairs that changed."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ERR_ARG = -3
WORLD = dict(n_maps=6, n_points=100_000, size_x=14.0, size_y=8.0, rooms_x=2, rooms_y=1, window_frac=0.6)


@pytest.fixture(scope="module")
def world(synth):
    """six overlapping maps, and the same six drawn from another seed (replacement clouds)"""
    maps, truth = synth.make_maps(seed=31, **WORLD)
    alt, _ = synth.make_maps(seed=32, **WORLD)
    return maps, alt, truth


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def to_records(pts, layout):
    """float32[n, 4] -> uint8[n, point_step] records in `layout`; the other bytes hold the layout's template"""
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 4)
    w = np.tile(np.frombuffer(layout.template_bytes, np.uint32), (len(pts), 1))
    src = pts.view(np.uint32)
    for k, off in enumerate((layout.offset_x, layout.offset_y, layout.offset_z, layout.offset_rgba)):
        w[:, off // 4] = src[:, k]
    return np.ascontiguousarray(w).view(np.uint8)


def pair_list(ctx, clouds, p):
    """the row-major pair list of estimateMapsTransforms: i < j, both maps with keypoints"""
    dm = ctx.maps_upload(clouds)
    f = ctx.features_compute(dm, 0, len(clouds), p)
    _, nk, _ = f.sizes()
    f.free()
    dm.free()
    return [(i, j) for i in range(len(nk)) for j in range(i + 1, len(nk)) if nk[i] > 0 and nk[j] > 0]


def estimate_equal(ctx, ms, clouds, p):
    """the map set's estimate equals the stateless one on the same clouds; returns its work counters"""
    got, work = ms.estimate(p, work=True)
    want = ctx.estimate_maps_transforms(clouds, p)
    assert got.shape == want.shape
    assert np.array_equal(bits(got), bits(want))
    return work


def touching(pairs, m):
    return sum(1 for ij in pairs if m in ij)


@pytest.mark.parametrize("desc,method", [("PFH", "MATCHING"), ("FPFH", "MATCHING"), ("FPFH", "SAC_IA")])
def test_update_sequence(ctx, mm, world, desc, method):
    maps, alt, _ = world
    p = mm.default_params(descriptor_type=desc, estimation_method=method)
    exact = method == "MATCHING"  # SAC_IA may also re-register clean pairs whose rand() offset moved
    ms = ctx.mapset()
    cur = list(maps)
    assert ms.update({i: m for i, m in enumerate(cur)}) == [True] * 6
    assert len(ms) == 6
    P = pair_list(ctx, cur, p)
    assert len(P) >= 10
    assert estimate_equal(ctx, ms, cur, p) == [6, len(P), 0]

    cur[2] = alt[2]
    assert ms.update({2: alt[2]}) == [True]
    P = pair_list(ctx, cur, p)
    w = estimate_equal(ctx, ms, cur, p)
    assert w[0] == 1 and w[1] + w[2] == len(P)
    if exact:
        assert w == [1, touching(P, 2), len(P) - touching(P, 2)]
    else:
        assert w[1] >= touching(P, 2)

    # every map again, unchanged, in another record layout: nothing to do, no kernel
    pcl = mm.PCL_XYZRGB
    assert ms.update({i: to_records(m, pcl) for i, m in enumerate(cur)}, pcl) == [False] * 6
    l0 = ctx.launches
    got, w = ms.estimate(p, work=True)
    assert ctx.launches == l0
    assert w == [0, 0, len(P)]
    assert np.array_equal(bits(got), bits(ctx.estimate_maps_transforms(cur, p)))

    # a NULL slot, then an empty cloud in its place (the same empty map)
    cur[4] = None
    assert ms.update({4: None}) == [True]
    P = pair_list(ctx, cur, p)
    w = estimate_equal(ctx, ms, cur, p)
    assert w[0] == 1 and w[1] + w[2] == len(P)
    if exact:
        assert w[1] == 0
    cur[4] = np.zeros((0, 4), np.float32)
    assert ms.update({4: cur[4]}) == [False]
    assert estimate_equal(ctx, ms, cur, p) == [0, 0, len(P)]

    # grow through a slot index two past the end: slot 6 stays empty, slot 7 gets a map
    cur += [None, maps[4]]
    assert ms.update({7: maps[4]}) == [True]
    assert len(ms) == 8
    P = pair_list(ctx, cur, p)
    w = estimate_equal(ctx, ms, cur, p)
    assert w[0] == 2 and w[1] + w[2] == len(P)
    if exact:
        assert w[1] == touching(P, 7)
    # the last slot emptied: n_out follows the highest map index that has a pair
    cur[7] = None
    assert ms.update({7: None}) == [True]
    assert len(ctx.estimate_maps_transforms(cur, p)) < len(cur)
    assert estimate_equal(ctx, ms, cur, p)[0] == 1
    ms.free()


def test_sac_ia_offsets_move_with_an_early_source_map(ctx, mm, world):
    """Replacing map 0 changes the rand() draws of its pairs, which shifts the offsets of every later pair: the map set
    registers those again although their maps did not change."""
    maps, alt, _ = world
    p = mm.default_params(descriptor_type="FPFH", estimation_method="SAC_IA")
    ms = ctx.mapset()
    cur = list(maps)
    ms.update({i: m for i, m in enumerate(cur)})
    estimate_equal(ctx, ms, cur, p)
    cur[0] = alt[0]
    assert ms.update({0: alt[0]}) == [True]
    P = pair_list(ctx, cur, p)
    w = estimate_equal(ctx, ms, cur, p)
    assert w[0] == 1 and w[1] + w[2] == len(P)
    assert w[1] > touching(P, 0)
    # the last map changed: the offsets of earlier pairs cannot move
    cur[5] = alt[5]
    ms.update({5: alt[5]})
    P = pair_list(ctx, cur, p)
    assert estimate_equal(ctx, ms, cur, p) == [1, touching(P, 5), len(P) - touching(P, 5)]
    ms.free()


def test_parameter_change_recomputes_everything(ctx, mm, world):
    maps, _, _ = world
    p = mm.default_params(descriptor_type="FPFH")
    q = mm.default_params(descriptor_type="FPFH", inlier_threshold=0.4)
    ms = ctx.mapset()
    ms.update({i: m for i, m in enumerate(maps)})
    P = pair_list(ctx, maps, p)
    assert estimate_equal(ctx, ms, maps, p) == [6, len(P), 0]
    assert estimate_equal(ctx, ms, maps, q) == [6, len(P), 0]
    assert estimate_equal(ctx, ms, maps, q) == [0, 0, len(P)]
    assert estimate_equal(ctx, ms, maps, p) == [6, len(P), 0]
    ms.free()


def test_change_detection_is_bitwise(ctx, mm, world):
    maps, _, _ = world
    p = mm.default_params(descriptor_type="FPFH")
    ms = ctx.mapset()
    cur = list(maps)
    base = maps[1].copy()
    base[20, 1] = 0.0
    base.view(np.uint32)[30, 2] = 0x7fc00001
    cur[1] = base
    ms.update({i: m for i, m in enumerate(cur)})
    estimate_equal(ctx, ms, cur, p)
    assert ms.update({1: base.copy()}) == [False]

    ulp = base.copy()
    ulp.view(np.uint32)[10, 0] += 1
    negzero = base.copy()
    negzero[20, 1] = -0.0
    payload = base.copy()
    payload.view(np.uint32)[30, 2] = 0x7fc00002
    for v in (ulp, negzero, payload, base):
        assert ms.update({1: v}) == [True]
        cur[1] = v
        w = estimate_equal(ctx, ms, cur, p)
        assert w[0] == 1
    ms.free()


def test_compose_matches_stateless(ctx, mm, world):
    maps, alt, truth = world
    pcl = mm.PCL_XYZRGB
    ms = ctx.mapset()
    cur = list(maps)
    ms.update({i: to_records(m, pcl) for i, m in enumerate(cur)}, pcl)
    T = np.stack([np.linalg.inv(truth[0]) @ t for t in truth]).astype(np.float32)
    T[3] = 0.0  # composeMaps leaves maps with a zero transform out
    for step in range(2):
        recs = [to_records(m, mm.PACKED) if m is not None else None for m in cur]
        for res in (0.05, 0.2):
            want = ctx.compose_maps_layout(recs, T, res, mm.PACKED, mm.PACKED)
            got = ms.compose(T, res)
            assert got.dtype == np.float32 and np.array_equal(bits(got), want.view(np.uint32).reshape(-1, 4))
            want = ctx.compose_maps_layout(recs, T, res, mm.PACKED, pcl)
            got = ms.compose(T, res, pcl)
            assert got.shape == want.shape and np.array_equal(got, want)
        cur[2] = alt[2]
        cur[5] = None
        ms.update({2: alt[2], 5: None})
    with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
        ms.compose(T[:5], 0.05)
    ms.free()
    empty = ctx.mapset()
    assert empty.compose(np.zeros((0, 4, 4), np.float32), 0.05) is None
    empty.free()


def test_errors_leave_the_set_unchanged(ctx, mm, world):
    maps, alt, _ = world
    p = mm.default_params(descriptor_type="FPFH")
    ms = ctx.mapset()
    ms.update({i: m for i, m in enumerate(maps)})
    P = pair_list(ctx, maps, p)
    estimate_equal(ctx, ms, maps, p)
    other = mm.Context(0)
    L = ctx.L
    l0, o0 = ctx.launches, other.launches
    bad = mm.Layout(18, 0, 4, 8, 12)
    with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
        ms.update({2: np.zeros((len(alt[2]), 18), np.uint8)}, bad)
    with pytest.raises(mm.MM3DError, match=f"error {ERR_ARG}"):
        ms.update({2: alt[2], -1: alt[3]})
    # a NULL layout and a foreign context, through the C ABI
    arrs, ptrs, ns = ctx._cloud_args([alt[2]])
    slot = (C.c_int32 * 1)(2)
    changed = (C.c_int32 * 1)(7)
    assert L.mm3d_mapset_update(ctx.h, ms.h, 1, slot, ptrs, ns, None, changed) == ERR_ARG
    assert L.mm3d_mapset_update(other.h, ms.h, 1, slot, ptrs, ns, C.byref(mm.PACKED), changed) == ERR_ARG
    out = np.zeros((6, 16), np.float32)
    no = C.c_int()
    f32p = C.POINTER(C.c_float)
    assert L.mm3d_mapset_estimate(other.h, ms.h, C.byref(p), out.ctypes.data_as(f32p), C.byref(no), None) == ERR_ARG
    res, n = C.c_void_p(), C.c_uint64()
    Tc = np.tile(np.eye(4, dtype=np.float32).reshape(1, 16), (6, 1))
    assert L.mm3d_mapset_compose(other.h, ms.h, 6, Tc.ctypes.data_as(f32p), C.c_double(0.05), C.byref(mm.PACKED), C.byref(res),
                                 C.byref(n)) == ERR_ARG
    assert ctx.launches == l0 and other.launches == o0
    assert len(ms) == 6 and changed[0] == 7
    assert estimate_equal(ctx, ms, maps, p) == [0, 0, len(P)]

    # a failed estimate commits nothing: the changed map is still pending at the next one
    cur = list(maps)
    cur[2] = alt[2]
    ms.update({2: alt[2]})
    with pytest.raises(mm.MM3DError, match="error -4"):
        ms.estimate(mm.default_params(descriptor_type=99))
    P = pair_list(ctx, cur, p)
    assert estimate_equal(ctx, ms, cur, p) == [1, touching(P, 2), len(P) - touching(P, 2)]
    ms.free()
    other.close()


def test_full_size_one_map_replaced(ctx, mm, synth):
    """Config 3 (32 x 1M points, SIFT + FPFH as in the benchmark): map 17 replaced by a map drawn from another seed."""
    cfg = dict(synth.CONFIGS["c3"])
    maps, _ = synth.make_maps(**cfg)
    new17 = synth.make_maps(**dict(cfg, seed=cfg["seed"] + 100), only=[17])[0][17]
    p = mm.default_params(descriptor_type="FPFH")
    ms = ctx.mapset()
    ms.update({i: m for i, m in enumerate(maps)})
    w0 = estimate_equal(ctx, ms, maps, p)
    assert w0[0] == 32 and w0[2] == 0
    maps[17] = new17
    assert ms.update({17: new17}) == [True]
    w = estimate_equal(ctx, ms, maps, p)
    assert w[0] == 1 and w[1] + w[2] >= 465
    if w[1] + w[2] == 496:  # every map has keypoints
        assert w == [1, 31, 465]
    ms.free()
