"""Nearest-neighbour search of ICP and scoring (tile_nearest / nearest_block27 in csrc/icp.cu) against brute force, at the
geometric edges where its float slack is tight: far from the origin, exact ties, squared distances equal to the bound,
correspondence distances below one voxel and past the reach-grid clamp, coarsened indexes, targets without a reach grid,
dense voxels, tile edges and clouds past the voxel-grid overflow guard.

The reference here is independent of the kernel and of the oracle: every transform and squared distance in float32 in the
kernel's operation order (numpy float32 arithmetic does not contract), the nearest point by (d^2, original index) among
those with (double) d^2 <= bound, and the fixed-point sums of icp_tile / score_kernel."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

f32 = np.float32
FIX1, FIX2, FIXD = 2.0 ** 32, 2.0 ** 24, 2.0 ** 36
DBL_MAX = np.finfo(np.float64).max


# ---------------------------------------------------------------- reference
def xform(T, pts):
    """em::transform_point: ((m0 x + m1 y) + m2 z) + m3, float32, T row-major 4 x 4."""
    m = np.asarray(T, f32).reshape(16)
    x, y, z = (np.asarray(pts, f32)[:, k] for k in range(3))
    return np.stack([((m[4 * r] * x + m[4 * r + 1] * y) + m[4 * r + 2] * z) + m[4 * r + 3] for r in range(3)], axis=1)


def dist2(q, p):
    """em::dist2_3 in float32: dx^2, += dy^2, += dz^2 (broadcasts)."""
    dx, dy, dz = (q[..., k] - p[..., k] for k in range(3))
    r = dx * dx
    r = r + dy * dy
    return r + dz * dz


def nearest(q, tgt, bound):
    """Per query: (original index, d^2) of the nearest target point by (d^2, index) among those with (double) d^2 <= bound;
    index -1 when there is none."""
    q = np.asarray(q, f32)[:, :3]
    t = np.asarray(tgt, f32)[:, :3]
    idx = np.full(len(q), -1, np.int64)
    d2 = np.zeros(len(q), f32)
    if len(t) == 0 or len(q) == 0:
        return idx, d2
    if len(q) * len(t) <= 20_000_000:
        step = max(1, 4_000_000 // len(t))
        for s in range(0, len(q), step):
            dd = dist2(q[s:s + step, None, :], t[None, :, :])
            dd = np.where(dd.astype(np.float64) <= bound, dd, np.inf)
            j = np.argmin(dd, axis=1)  # first minimum = lowest original index
            hit = np.isfinite(dd[np.arange(len(j)), j])
            idx[s:s + step] = np.where(hit, j, -1)
            d2[s:s + step] = np.where(hit, dd[np.arange(len(j)), j], 0)
        return idx, d2
    # candidates from a float64 k-d tree with a margin far above float32 rounding, then exact float32 distances
    tree = cKDTree(t.astype(np.float64))
    mag = float(max(np.abs(q).max(), np.abs(t).max()))
    r = np.sqrt(max(bound, 0.0)) * (1 + 1e-4) + 1e-5 * (1.0 + mag)
    for i, cand in enumerate(tree.query_ball_point(q.astype(np.float64), r)):
        if not cand:
            continue
        c = np.sort(np.asarray(cand, np.int64))
        dd = dist2(q[i][None, :], t[c])
        ok = dd.astype(np.float64) <= bound
        if ok.any():
            c, dd = c[ok], dd[ok]
            k = np.lexsort((c, dd))[0]
            idx[i], d2[i] = c[k], dd[k]
    return idx, d2


def to_fix(v, scale):
    return np.rint(np.asarray(v, np.float64) * scale).astype(np.int64)


def ref_score(src, tgt, T, max_distance):
    """TransformationValidationEuclidean: mean squared distance of the matched points, d^2 compared with the plain range."""
    idx, d2 = nearest(xform(T, src), tgt, max_distance)
    hit = idx >= 0
    if not hit.any():
        return DBL_MAX
    return (float(to_fix(d2[hit], FIXD).sum()) / FIXD) / float(hit.sum())


def ref_icp_sums(src, tgt, T0, max_dist):
    """The 17 fixed-point sums of ICP iteration 1: n, Sp[3], Sq[3], Sq_a p_b[9], Sd."""
    p = xform(T0, src)
    idx, d2 = nearest(p, tgt, max_dist * max_dist)
    hit = idx >= 0
    p = p[hit].astype(np.float64)
    q = np.asarray(tgt, f32)[idx[hit], :3].astype(np.float64)
    s = [int(hit.sum())]
    s += [int(to_fix(p[:, a], FIX1).sum()) for a in range(3)]
    s += [int(to_fix(q[:, a], FIX1).sum()) for a in range(3)]
    s += [int(to_fix(q[:, a] * p[:, b], FIX2).sum()) for a in range(3) for b in range(3)]
    s += [int(to_fix(d2[hit], FIXD).sum())]
    return np.array(s, np.int64)


# ---------------------------------------------------------------- nearest_block27 as written at the parent commit
def block27_as_written(q, tgt, leaf, bound):
    """Float32 emulation of the 27-voxel block search with the parent's slack (row pruning 1.0001 / 1e-4, certain below
    0.999 voxel^2), for a target given in cell order.  Returns (index or -1, certain)."""
    inv = f32(1.0) / f32(leaf)
    inv2 = inv * inv
    fq = np.asarray(q, f32)[:3] * inv
    fl = np.floor(fq)
    ay, az = fq[1] - fl[1], fq[2] - fl[2]
    cells = np.floor(np.asarray(tgt, f32)[:, :3] * inv)
    found, best, best_i, bestv = False, f32(0), -1, f32(3e38)
    for t in range(9):
        dz, dy = t // 3 - 1, t % 3 - 1
        zd = az if dz < 0 else (f32(1) - az if dz > 0 else f32(0))
        yd = ay if dy < 0 else (f32(1) - ay if dy > 0 else f32(0))
        if zd * zd + yd * yd > bestv:
            continue
        for k in range(len(tgt)):
            c = cells[k] - fl
            if c[2] != dz or c[1] != dy or abs(c[0]) > 1:
                continue
            d = dist2(np.asarray(q, f32)[:3], np.asarray(tgt, f32)[k, :3])
            if float(d) > bound:
                continue
            if not found or d < best:
                found, best, best_i = True, d, k
                bestv = d * inv2 * f32(1.0001) + f32(1e-4)
    return best_i, bool(found and best * inv2 < f32(0.999))


# ---------------------------------------------------------------- case classes
def _pts(a):
    a = np.asarray(a, f32).reshape(-1, 3)
    return np.concatenate([a, np.zeros((len(a), 1), f32)], axis=1)


def _bits(*words):
    return np.array(words, np.uint32).view(f32)


EYE = np.eye(4, dtype=f32)
# (q, A, B) as float32 bit patterns: B is the nearest point; the parent's row pruning skipped it and kept A as certain
PLANTED = [
    (_bits(0x43fa32c7, 0x43fa3c52, 0x43fa0884), _bits(0x43fa3710, 0x43fa3c52, 0x43fa0884), _bits(0x43fa32c7, 0x43fa3c52, 0x43fa0ccc)),
    (_bits(0x447a3507, 0x447a250f, 0x447a15cf), _bits(0x447a38d2, 0x447a250f, 0x447a15cf), _bits(0x447a3507, 0x447a250f, 0x447a1999)),
]


def _row_edge(inv, row, first):
    """The smallest (first) or largest float32 v whose cell floor(fl(v * inv)) is `row`."""
    if not first:
        return np.nextafter(_row_edge(inv, row + 1, True), f32(-np.inf))
    v = f32(float(row) / float(inv))
    while np.floor(v * inv) >= row:
        v = np.nextafter(v, f32(-np.inf))
    while np.floor(v * inv) < row:
        v = np.nextafter(v, f32(np.inf))
    return v


def _just_farther(q, d2b, axis):
    """A point that differs from q along `axis` only, with the smallest float32 d^2 above d2b."""
    a = q.copy()
    a[axis] = f32(float(q[axis]) + np.sqrt(float(d2b)))
    while dist2(q, a) > d2b:
        a[axis] = np.nextafter(a[axis], f32(-np.inf))
    while dist2(q, a) <= d2b:
        a[axis] = np.nextafter(a[axis], f32(np.inf))
    return a


def planted_configs(offset, n, seed, leaf=0.1, spacing=3.0):
    """n (q, A, B) triples around `offset`, each at its own lattice site `spacing` apart.  B lies just across a (z, y) row
    boundary (the parent's row pruning case) or, for one third, in voxel v +- 2 along z with q at the far edge of its voxel
    (the certainty case); A differs from q along x with the smallest d^2 above d^2(B)."""
    rng = np.random.default_rng(seed)
    inv = f32(1.0) / f32(leaf)
    side = int(np.ceil(n ** (1 / 3)))
    out = []
    for i in range(n):
        site = np.array([i % side, (i // side) % side, i // side // side], np.float64) * spacing
        q = (offset + site + rng.uniform(0, leaf, 3)).astype(f32)
        kind, sgn = i % 3, (1 if rng.random() < 0.5 else -1)
        if kind < 2:  # row boundary along z (kind 0) or y (kind 1)
            ax = 2 - kind
            b = q.copy()
            b[ax] = _row_edge(inv, np.floor(q[ax] * inv) + sgn, first=sgn > 0)
        else:  # q at the far edge of its z voxel, B two voxels along
            fl = np.floor(q * inv)
            q[0] = f32((float(fl[0]) + 0.2) / float(inv))
            q[2] = _row_edge(inv, fl[2], first=sgn < 0)
            b = q.copy()
            b[2] = _row_edge(inv, fl[2] + 2 * sgn, first=sgn > 0)
        a = _just_farther(q, dist2(q, b), 0)
        out.append((q, a, b))
    return out


def _planted_cloud(cfgs):
    src = _pts([q for q, _, _ in cfgs])
    tgt = _pts([p for _, a, b in cfgs for p in (a, b)])  # A before B: a tie on the index would pick A
    return src, tgt


def case_planted():
    cases = []
    for k, (q, a, b) in enumerate(PLANTED):
        cases.append(dict(name=f"planted{k}", src=_pts([q]), tgt=_pts([a, b]), leaf=0.1, dists=(1.0,)))
    for off in (0.0, 100.0, 500.0, 1000.0, 4000.0):
        for sgn in (1, -1):
            cfgs = planted_configs(np.full(3, sgn * off), 61, seed=int(off) * 2 + (sgn > 0))
            src, tgt = _planted_cloud(cfgs)
            cases.append(dict(name=f"planted@{sgn * off:+g}", src=src, tgt=tgt, leaf=0.1, dists=(1.0,)))
    return cases


def _plane(leaf, n=40, z0=0.0, seed=0, origin=(0.0, 0.0)):
    """A voxelised, jittered plane patch: one point per voxel of an n x n patch at height z0."""
    rng = np.random.default_rng(seed)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    x = origin[0] + (i.ravel() + 0.5 + rng.uniform(-0.3, 0.3, i.size)) * leaf
    y = origin[1] + (j.ravel() + 0.5 + rng.uniform(-0.3, 0.3, i.size)) * leaf
    z = z0 + rng.uniform(-0.05, 0.05, i.size) * leaf
    return _pts(np.stack([x, y, z], 1))


SWEEP = (0, 0.5, 0.999, 1, 1.001, 1.5, 2.5, 3.49, 3.5, 3.51, 5, 9.5, 9.99, 10, 10.01, 12, 14.9, 15, 16, 40)
CORR = (0.05, 0.1, 0.35, 1.0, 2.0)  # below the reach clamp of 2 voxels, the 3.5-voxel group split, default, past the 15-voxel clamp


def _sweep_queries(leaf, shift=0.0, n=40):
    qs = []
    for h in SWEEP:
        for fx, fy in ((0.5, 0.5), (0.0, 0.5), (0.0, 0.0), (0.25, 0.75)):  # voxel centre, face, corner, inside
            for cx in (3, n // 2, n - 4):
                qs.append(((cx + fx) * leaf + shift, (n // 2 + fy) * leaf + shift, h * leaf + shift))
    return _pts(qs)[:-3]  # 237 queries: not a multiple of the tile


def case_sweep(shift=0.0):
    leaf = 0.1
    tgt = _plane(leaf)
    tgt[:, :3] += f32(shift)
    return [dict(name=f"sweep@{shift:+g}", src=_sweep_queries(leaf, shift), tgt=tgt, leaf=leaf, dists=CORR)]


TIE_DIRS = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], np.float64)


def case_ties(shift=0.0, seed=3):
    """Queries exactly equidistant from 2-6 target points (leaf 0.125, offsets in 1/16 m, exact in float32): tied points
    in one row (+-x), in different rows (y, z), one inside the 27-voxel block and one outside (1.5 voxels either way from
    a voxel centre).  The target is shuffled, so the index sorts a private copy and keeps the original indices."""
    rng = np.random.default_rng(seed)
    leaf = 0.125
    src, tgt = [], []
    for i in range(150):
        c = np.array([i % 6, (i // 6) % 5, i // 30], np.float64) * 1.5 + shift
        q = c + leaf * np.array([0.5, 0.5, 0.5]) if i % 2 else c + leaf * np.array([0.25, 0.75, 0.5])
        r = leaf * (0.5, 1.0, 1.5, 0.75)[i % 4]
        k = 2 + i % 5
        dirs = TIE_DIRS[rng.permutation(6)[:k]] if i % 3 else TIE_DIRS[[0, 1, 2, 3, 4, 5][:k]]
        src.append(q)
        tgt.extend(q + r * dirs)
        tgt.append(q + (r + leaf * 0.5) * TIE_DIRS[rng.integers(6)])  # a farther decoy
    src, tgt = _pts(src), _pts(tgt)
    tgt = tgt[rng.permutation(len(tgt))]
    return [dict(name=f"ties@{shift:+g}", src=src[:-1], tgt=tgt, leaf=leaf, dists=(0.2, 1.0))]


def case_bound():
    """d^2 exactly equal to the bound is a match; one float farther is not (q = (1 + 4k, 1, 1), p = q + 0.5 x)."""
    qs, ps = [], []
    for k in range(20):
        q = np.array([1 + 4 * k, 1, 1], f32)
        p = q.copy()
        p[0] = f32(q[0] + f32(0.5))
        if k % 2:
            p[0] = np.nextafter(p[0], f32(np.inf))
        qs.append(q)
        ps.append(p)
    return [dict(name="bound", src=_pts(qs), tgt=_pts(ps), leaf=0.1, dists=(0.5,), score_bounds=(0.25,))]


def case_boundaries():
    """Leaves 0.125 and 0.25; queries and targets on voxel boundaries, straddling zero and all negative."""
    rng = np.random.default_rng(5)
    cases = []
    for leaf in (0.125, 0.25):
        for shift, name in ((0.0, "straddle"), (-7.0, "negative")):
            tgt = rng.integers(-8, 8, size=(600, 3)) * (leaf / 2) + shift
            src = rng.integers(-10, 10, size=(301, 3)) * (leaf / 4) + shift
            cases.append(dict(name=f"{name}@{leaf}", src=_pts(src), tgt=_pts(tgt), leaf=leaf, dists=(leaf * 0.5, leaf, 0.35, 1.0)))
    return cases


def case_far():
    cases = []
    for off in (100.0, 500.0, 1000.0, 4000.0):
        for sgn in (1, -1):
            cases += case_sweep(sgn * off) + case_ties(sgn * off)
    return cases


def case_irregular():
    """A hollow box with queries inside (equidistant from several walls), a concave corner, a thin line, and five isolated
    points with queries 12-15 voxels away at a 2 m correspondence distance (long or abandoned downhill walks)."""
    leaf = 0.1
    g = np.arange(0.0, 2.01, 0.1)
    a, b = np.meshgrid(g, g, indexing="ij")
    a, b = a.ravel(), b.ravel()
    walls = []
    for c in (0.0, 2.0):
        walls += [np.stack([np.full_like(a, c), a, b], 1), np.stack([a, np.full_like(a, c), b], 1), np.stack([a, b, np.full_like(a, c)], 1)]
    box = np.unique(np.concatenate(walls), axis=0)
    corner = np.concatenate([np.stack([a, b, np.zeros_like(a)], 1), np.stack([np.zeros_like(a), a, b], 1)]) + [5.0, 0, 0]
    line = np.stack([np.arange(0, 3, 0.05), np.zeros(60), np.zeros(60)], 1) + [0, 5.0, 0]
    iso = np.array([[10, 10, 10], [14, 10, 10], [10, 14, 10], [10, 10, 14], [14, 14, 14]], np.float64)
    tgt = np.concatenate([box, corner, line, iso])
    rng = np.random.default_rng(7)
    qs = [[1.0, 1.0, 1.0], [0.5, 1.0, 1.0], [1.0, 0.95, 1.05], [1.5, 1.5, 1.5]] + list(rng.uniform(0.2, 1.8, size=(60, 3)))
    qs += list(np.array([5.0, 0, 0]) + rng.uniform(0.05, 0.6, size=(40, 3)))
    qs += list(np.array([0, 5.0, 0]) + np.c_[rng.uniform(0, 3, 40), rng.uniform(-0.5, 0.5, (40, 2))])
    for p in iso:
        for r in (1.2, 1.35, 1.5):
            d = rng.normal(size=(4, 3))
            qs += list(p + r * d / np.linalg.norm(d, axis=1, keepdims=True))
    return [dict(name="irregular", src=_pts(qs), tgt=_pts(tgt), leaf=leaf, dists=(0.35, 1.0, 2.0))]


def case_coarse():
    """A 200 m x 200 m x 5 m target at leaf 0.1: one-voxel cells would exceed 2^27, so the index coarsens (shift != 0) and
    the block and the walk are off.  And a 400 m x 400 m x 10 m target, whose reach grid would exceed 2^30 cells."""
    rng = np.random.default_rng(9)
    cases = []
    for ext, name in (((200.0, 200.0, 5.0), "coarse"), ((400.0, 400.0, 10.0), "no_reach")):
        tgt = rng.uniform(0, 1, size=(60_000, 3)) * ext
        tgt[:8] = [[0, 0, 0], [ext[0], ext[1], ext[2]], [ext[0], 0, 0], [0, ext[1], 0], [0, 0, ext[2]], [ext[0], ext[1], 0], [0, 0, 0], [0, 0, 0]]
        src = tgt[rng.choice(len(tgt), 3001, replace=False)] + rng.normal(scale=0.3, size=(3001, 3))
        cases.append(dict(name=name, src=_pts(src), tgt=_pts(tgt), leaf=0.1, dists=(0.35, 1.0)))
    return cases


def case_dense():
    """A target that is not voxelised: hundreds of points per voxel, duplicated coordinates."""
    rng = np.random.default_rng(11)
    base = rng.uniform(0, 0.3, size=(1500, 3))
    tgt = np.concatenate([base, base[rng.choice(1500, 1500)]])
    tgt = np.round(tgt / 0.01) * 0.01  # more duplicates and exact ties
    tgt = tgt[rng.permutation(len(tgt))]
    src = rng.uniform(-0.2, 0.5, size=(777, 3))
    return [dict(name="dense", src=_pts(src), tgt=_pts(tgt), leaf=0.1, dists=(0.05, 0.35, 1.0))]


def case_tiles():
    """Source sizes 1, 127, 128, 129, 257: on the surface, all off it (large windows in phase 2) and mixed tiles."""
    leaf = 0.1
    tgt = _plane(leaf, n=30, seed=2)
    rng = np.random.default_rng(13)
    cases = []
    for n in (1, 127, 128, 129, 257):
        xy = rng.uniform(0.2, 2.8, size=(n, 2))
        for kind, h in (("on", rng.uniform(-0.02, 0.02, n)), ("off", rng.uniform(0.6, 0.95, n)),
                        ("mixed", np.where(rng.random(n) < 0.5, 0.01, rng.uniform(0.3, 0.95, n)))):
            cases.append(dict(name=f"tile{n}_{kind}", src=_pts(np.c_[xy, h]), tgt=tgt, leaf=leaf, dists=(1.0,)))
    return cases


def case_guard_target():
    """A target whose box exceeds 2^31 voxels at the index leaf (pcl::VoxelGrid's overflow guard): a plane patch plus two
    points 300 m x 300 m x 24 m apart."""
    tgt = np.concatenate([_plane(0.1, n=40, seed=4), _pts([[300.0, 300.0, 24.0], [-0.5, -0.5, -0.5]])])
    return [dict(name="past_guard", src=_sweep_queries(0.1), tgt=tgt, leaf=0.1, dists=(0.35, 1.0))]


CLASSES = dict(planted=case_planted, sweep=case_sweep, bound=case_bound, ties=case_ties, boundaries=case_boundaries,
               far=case_far, irregular=case_irregular, coarse=case_coarse, dense=case_dense, tiles=case_tiles,
               past_guard=case_guard_target)


def _subcases(case):
    """(ICP correspondence distance or None, score max_distance or None) pairs of one case."""
    for d in case["dists"]:
        yield d, d
    for b in case.get("score_bounds", ()):
        yield None, b


# ---------------------------------------------------------------- checks
def _first_difference(ctx, case, bound):
    """Re-run single-query scores and describe the first query whose matched d^2 differs from brute force."""
    src, tgt = case["src"], case["tgt"]
    idx, d2 = nearest(xform(EYE, src), tgt, bound)
    for i in range(min(len(src), 300)):
        got = ctx.score(src[i:i + 1], tgt, EYE, bound, index_leaf=case["leaf"])
        want = DBL_MAX if idx[i] < 0 else float(to_fix(d2[i], FIXD)) / FIXD
        if got != want:
            return f"first differing query {i} at {src[i, :3].tolist()}: d^2 {got!r} instead of {want!r} (target point {idx[i]})"
    return "no single query differs in the first 300"


def _check_case(ctx, oracle, case):
    src, tgt, leaf = case["src"], case["tgt"], case["leaf"]
    for dist, sb in _subcases(case):
        what = f"{case['name']} dist={dist} score_bound={sb}"
        if sb is not None:
            got, want = ctx.score(src, tgt, EYE, sb, index_leaf=leaf), ref_score(src, tgt, EYE, sb)
            assert got == want, f"{what}: score {got!r} vs brute force {want!r}; " + _first_difference(ctx, case, sb)
            assert oracle.score(src, tgt, EYE, sb) == want, f"{what}: oracle score"
        if dist is None:
            continue
        _, dbg = ctx.icp(src, tgt, EYE, dist, 1, 1e-6, index_leaf=leaf)
        want = ref_icp_sums(src, tgt, EYE, dist)
        assert np.array_equal(dbg["sums"][0], want), \
            f"{what}: ICP iteration 1 sums\n{dbg['sums'][0]}\nvs brute force\n{want}; " + _first_difference(ctx, case, dist * dist)
        gT, gdbg = ctx.icp(src, tgt, EYE, dist, 20, 1e-8, index_leaf=leaf)
        wT, wdbg = oracle.icp(src, tgt, EYE, dist, 20, 1e-8)
        assert (gdbg["iterations"], gdbg["converged"]) == (wdbg["iterations"], wdbg["converged"]), what
        assert np.array_equal(gdbg["sums"], wdbg["sums"]), f"{what}: per-iteration ICP sums differ from the oracle"
        assert np.array_equal(gT.view(np.uint32), wT.view(np.uint32)), f"{what}: ICP transform differs from the oracle"


def test_reference_matches_oracle_on_every_case(oracle):
    """The brute-force reference reproduces oracle.score and iteration 1 of oracle.icp on every case class (no device)."""
    for name, make in CLASSES.items():
        for case in make():
            src, tgt = case["src"], case["tgt"]
            for dist, sb in _subcases(case):
                what = f"{case['name']} dist={dist} score_bound={sb}"
                if sb is not None:
                    assert ref_score(src, tgt, EYE, sb) == oracle.score(src, tgt, EYE, sb), what
                if dist is not None:
                    _, wdbg = oracle.icp(src, tgt, EYE, dist, 1, 1e-6)
                    assert np.array_equal(ref_icp_sums(src, tgt, EYE, dist), wdbg["sums"][0]), what


def test_planted_cases_defeat_the_old_block_rule():
    """The two planted configurations, and part of the generated ones at 500 m and beyond, make the 27-voxel block as
    the parent wrote it keep a farther point and call it certain; at 0 m and 100 m none does."""
    for q, a, b in PLANTED:
        i, certain = block27_as_written(q, np.stack([a, b]), 0.1, 1.0)
        assert (i, certain) == (0, True)
        idx, _ = nearest(_pts([q]), _pts([a, b]), 1.0)
        assert idx[0] == 1
    for off, expect in ((0.0, False), (100.0, False), (1000.0, True)):
        fails = 0
        for sgn in (1, -1):
            for q, a, b in planted_configs(np.full(3, sgn * off), 61, seed=int(off) * 2 + (sgn > 0)):
                assert dist2(q, b) < dist2(q, a)
                i, certain = block27_as_written(q, np.stack([a, b]), 0.1, 1.0)
                fails += certain and i == 0
        assert (fails > 0) == expect, (off, fails)


@pytest.mark.gpu
@pytest.mark.parametrize("cls", list(CLASSES))
def test_nearest_neighbour_edges(ctx, oracle, cls):
    for case in CLASSES[cls]():
        _check_case(ctx, oracle, case)


@pytest.mark.gpu
def test_far_from_origin_tiny_stages_icp(ctx, oracle, tiny_stages, tiny_maps):
    """The tiny maps' filtered clouds translated far from the origin, through every ICP iteration from a perturbed ground
    truth, and their score, against the oracle."""
    s, t = tiny_stages
    _, truth = tiny_maps
    gt = (np.linalg.inv(truth[1]) @ truth[0]).astype(f32)
    c, sn = np.cos(0.05), np.sin(0.05)
    pert = np.array([[c, -sn, 0, 0.08], [sn, c, 0, -0.05], [0, 0, 1, 0.03], [0, 0, 0, 1]], f32)
    for off in (100.0, -500.0, 1000.0, -4000.0):
        src, tgt = s["filtered"].copy(), t["filtered"].copy()
        src[:, :3] += f32(off)
        tgt[:, :3] += f32(off)
        sh = np.eye(4, dtype=f32)
        sh[:3, 3] = off
        T0 = (sh @ pert @ gt @ np.linalg.inv(sh)).astype(f32)
        wT, wdbg = oracle.icp(src, tgt, T0, 1.0, 30, 1e-6)
        gT, gdbg = ctx.icp(src, tgt, T0, 1.0, 30, 1e-6, index_leaf=0.1)
        assert (gdbg["iterations"], gdbg["converged"]) == (wdbg["iterations"], wdbg["converged"]), off
        assert np.array_equal(gdbg["sums"], wdbg["sums"]), f"offset {off}: per-iteration sums differ"
        assert np.array_equal(gT.view(np.uint32), wT.view(np.uint32)), f"offset {off}: transform differs"
        assert np.array_equal(gdbg["sums"][0], ref_icp_sums(src, tgt, T0, 1.0)), f"offset {off}: iteration 1 vs brute force"
        assert ctx.score(src, tgt, wT, 1.0, index_leaf=0.1) == oracle.score(src, tgt, wT, 1.0) == ref_score(src, tgt, wT, 1.0), off


def _past_guard_maps(tiny_maps):
    maps, _ = tiny_maps
    out = []
    for m in maps:
        extra = np.zeros((2, 4), f32)
        extra[0, :3] = m[:, :3].min(axis=0)
        extra[1, :3] = m[:, :3].min(axis=0) + f32([300.0, 300.0, 24.0])
        extra[:, 3] = m[:2, 3]
        out.append(np.concatenate([m, extra]))
    return out


@pytest.mark.gpu
def test_maps_past_the_voxel_grid_guard(ctx, mm, oracle, tiny_maps):
    """Two tiny maps, each with two extra points 300 m x 300 m x 24 m apart: the box exceeds 2^31 voxels at resolution 0.1,
    pcl::VoxelGrid passes the cloud through, and the whole path still runs and matches the oracle pair for pair."""
    import oracle_py
    from test_full_size_gpu import _pairs_against_oracle
    maps = _past_guard_maps(tiny_maps)
    for m in maps:
        assert oracle.downsample(m, 0.1)[1]["passthrough"] == 1
    p_gpu, p_cpu = mm.default_params(descriptor_type="FPFH"), oracle_py.default_params(descriptor_type=2)
    want = oracle.estimate_maps_transforms(maps, p_cpu)
    got = ctx.estimate_maps_transforms(maps, p_gpu)
    np.testing.assert_allclose(got, want["transforms"], rtol=0, atol=1e-5)
    _pairs_against_oracle(ctx, oracle, maps, p_gpu, p_cpu, "past the voxel-grid guard")


@pytest.mark.gpu
def test_index_coordinates_out_of_int32_fail_loudly(ctx):
    """A target whose voxel coordinates do not fit in int32 at the index leaf is an error, not a silent wrong answer."""
    tgt = _pts([[0.0, 0.0, 0.0], [3.0e8, 0.0, 0.0]])
    with pytest.raises(RuntimeError, match="int32"):
        ctx.score(_pts([[0.0, 0.0, 0.0]]), tgt, EYE, 1.0, index_leaf=0.1)
    with pytest.raises(RuntimeError, match="int32"):
        ctx.icp(_pts([[0.0, 0.0, 0.0]] * 4), tgt, EYE, 1.0, 5, 1e-6, index_leaf=0.1)
