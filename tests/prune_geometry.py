"""Adversarial clouds for the pruned top-k search (csrc/search.cu section 3b): geometry that stresses its walk outwards from
a home block and its block bound (test infrastructure, shared by the CPU and GPU tests and tools/fuzz_search.py).

family(name, seed, n, s) -> (ref [n, 3], qry [s, 3]) float32, one cloud per call:
  plane / tilted_plane    zero thickness along one axis (a grid of one cell on it) or along a slanted normal
  line_axis / line_diag   a line along x (two axes of one cell) and along the diagonal (a 32^3 grid, nearly all empty)
  ground_objects          a LiDAR-like ground plane with a few dense compact objects; queries on the ground and on them
  shell                   a spherical shell, queries at and near its centre: every block has nearly the same bound
  shell_snapped           integer points of a shell band, integer queries at and around the centre: exact ties
  two_clusters            two dense clusters far apart, queries in the empty space between them (empty home cells)
  density                 a core 1000 times denser than its halo, queries in the halo
  outside                 refs in a box, queries beyond every face, edge and corner (clamped into the border cells)
  lattice                 shuffled refs on an integer lattice, queries at cell, face and edge midpoints: ties across blocks
  precision               extents of 1e-3 .. 1e-1 at offsets of 1e3 .. 3e5 (PRECISION[seed % 5]): the expanded forms'
                          rounding is as large as the point spacing
"""
import numpy as np

F = np.float32
FAMILIES = ("plane", "tilted_plane", "line_axis", "line_diag", "ground_objects", "shell", "shell_snapped", "two_clusters",
            "density", "outside", "lattice", "precision")
PRECISION = ((1e-3, 1e3), (1e-2, 3e4), (1e-1, 3e5), (3e-3, -1e5), (3e-2, -3e5))      # (extent, offset)


def _pick(rng, pts, m):
    return pts[rng.choice(len(pts), m, replace=len(pts) < m)]


def _ball(rng, m, r0, r1):
    """m points uniform in the spherical shell r0 <= |p| <= r1"""
    d = rng.normal(size=(m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return d * np.cbrt(rng.uniform(r0 ** 3, r1 ** 3, (m, 1)))


def _int_shell(R):
    """integer points with R^2 - R <= |p|^2 <= R^2 + R"""
    g = np.arange(-R - 1, R + 2)
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    n2 = (p * p).sum(1)
    return p[(n2 >= R * R - R) & (n2 <= R * R + R)]


def family(name, seed, n=3000, s=600):
    rng = np.random.default_rng([seed, FAMILIES.index(name)])
    if name == "plane":
        ref = np.c_[rng.uniform(0, 40, (n, 2)), np.full(n, 1.5)]
        qry = np.c_[rng.uniform(-2, 42, (s, 2)), 1.5 + rng.choice([0.0, 0.0, 0.3, -2.0], s) * rng.random(s)]
    elif name == "tilted_plane":
        e = np.linalg.qr(rng.normal(size=(3, 3)))[0]
        ref = rng.uniform(-20, 20, (n, 2)) @ e[:2] + [3.0, -1.0, 7.0]
        qry = rng.uniform(-21, 21, (s, 2)) @ e[:2] + [3.0, -1.0, 7.0] + np.outer(rng.normal(size=s) * (rng.random(s) < 0.3), e[2])
    elif name == "line_axis":
        ref = np.c_[rng.uniform(0, 100, n), np.full(n, 2.0), np.full(n, -3.0)]
        qry = np.c_[rng.uniform(-5, 105, s), 2.0 + rng.normal(size=s) * (rng.random(s) < 0.5), np.full(s, -3.0)]
    elif name == "line_diag":
        ref = np.outer(rng.uniform(0, 100, n), np.ones(3) / np.sqrt(3.0)) + [1.0, 2.0, 3.0]
        qry = np.outer(rng.uniform(-5, 105, s), np.ones(3) / np.sqrt(3.0)) + [1.0, 2.0, 3.0] + rng.normal(size=(s, 3)) * 0.5
    elif name == "ground_objects":
        ng = int(0.7 * n)
        centres = np.c_[rng.uniform(-25, 25, (5, 2)), np.ones(5)]
        ground = np.c_[rng.uniform(-30, 30, (ng, 2)), rng.normal(size=ng) * 0.02]
        objs = centres[rng.integers(0, 5, n - ng)] + rng.normal(size=(n - ng, 3)) * 0.3
        ref = np.concatenate([ground, objs])[rng.permutation(n)]
        qry = np.concatenate([_pick(rng, ground if ng else objs, s // 2), _pick(rng, objs if n > ng else ground, s - s // 2)])
        qry += rng.normal(size=(s, 3)) * 0.05
    elif name == "shell":
        c = np.array([3.0, -2.0, 7.0])
        ref = c + _ball(rng, n, 10.0, 10.0)
        qry = c + np.concatenate([np.zeros((s // 4, 3)), rng.normal(size=(s - s // 4, 3)) * 0.05])
    elif name == "shell_snapped":
        pts = _int_shell(14)                                      # ~2500 points
        ref = _pick(rng, pts, n) + 100
        q = rng.integers(-1, 2, (s, 3)).astype(float) * (rng.random((s, 1)) < 0.7)
        qry = q + 100
    elif name == "two_clusters":
        ref = np.where(rng.random((n, 1)) < 0.5, -50.0, 50.0) * [1, 0, 0] + rng.normal(size=(n, 3))
        qry = np.c_[rng.uniform(-45, 45, s), rng.normal(size=(s, 2)) * 2.0]
        qry[: s // 8] = 0.0                                      # the midpoint: neighbours on both sides
    elif name == "density":
        ref = np.concatenate([_ball(rng, n // 2, 0.0, 0.1), _ball(rng, n - n // 2, 0.1, 1.0)])[rng.permutation(n)]
        qry = _ball(rng, s, 0.1, 1.0)
    elif name == "outside":
        ref = rng.uniform(0, 10, (n, 3))
        dirs = np.array([d for d in np.ndindex(3, 3, 3) if d != (1, 1, 1)], float) - 1.0       # 26 faces, edges, corners
        reach = np.array([0.01, 1.0, 10.0, 1e3, 1e5])
        d = dirs[rng.integers(0, 26, s)]
        qry = 5.0 + d * (5.0 + reach[rng.integers(0, len(reach), (s, 1))]) + (d == 0) * rng.uniform(-5, 5, (s, 3))
    elif name == "lattice":
        g = np.arange(16)
        pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
        ref = _pick(rng, pts, n)[rng.permutation(n)] * 0.25 + 8.0
        half = rng.integers(0, 15, (s, 3)) + np.where(rng.random((s, 3)) < [0.9, 0.7, 0.5], 0.5, 0.0)
        qry = half * 0.25 + 8.0
    elif name == "precision":
        ext, off = PRECISION[seed % len(PRECISION)]
        ref = off + rng.random((n, 3)) * ext
        qry = off + rng.uniform(-0.2, 1.2, (s, 3)) * ext
    else:
        raise ValueError(name)
    return ref.astype(F), qry.astype(F)


def batch(names, seed, n, s):
    """one family per batch item -> (ref [B, n, 3], qry [B, s, 3])"""
    pairs = [family(nm, seed + i, n, s) for i, nm in enumerate(names)]
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])


def mixed(seed, n=3000, s=600, k=16):
    """B = 6 items of different families at scales 1e-3 .. 1e4 and offsets; item 1 holds non-finite refs, item 4 fewer
    than k finite ones (it visits every block)"""
    names = ("ground_objects", "shell", "two_clusters", "lattice", "density", "outside")
    ref, qry = batch(names, seed, n, s)
    scale = np.array([1e-3, 1e-1, 1.0, 0.25, 1e2, 1e4], F)[:, None, None]
    off = np.array([[0, 0, 0], [50, -20, 3], [-1e3, 0, 0], [0, 0, 0], [3e3, 1e3, -2e3], [0, 0, 0]], F)[:, None, :]
    ref = (ref * scale + off).astype(F)
    qry = (qry * scale + off).astype(F)
    rng = np.random.default_rng(seed)
    ref[1, rng.choice(n, 40, replace=False)] = np.nan
    ref[1, rng.choice(n, 5, replace=False), rng.integers(0, 3)] = np.inf
    ref[4, k // 2:] = np.nan                                        # k/2 finite refs
    return ref, qry
