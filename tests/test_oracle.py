"""CPU tests: pin oracle/strict.c (and the torch port that bench.py times) against

  (1) tests/golden/reference_outputs.npz -- outputs of the REAL reference executed in the build
      container by tests/golden/make_golden.py;
  (2) the real reference itself when /root/reference is present (build container only);
  (3) each other.

Index comparisons are tie-aware (SURVEY Appendix A.4): torch's topk/sort are not index-stable,
so rows containing exactly equal distances among the k+1 nearest are exempted from the
index-equality check (their distance vectors must still agree bit for bit).
"""
import hashlib
import os

import numpy as np
import pytest
import torch

from b200pc import synth
from oracle import ref_loader, ref_torch, strict

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.npz"))


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


@pytest.fixture(scope="module")
def pair100():
    return synth.batch_pairs(100, 2, 4096)


def tie_free_rows(ref, qry, k, form):
    """rows whose k+1 smallest distances are pairwise distinct (indices are then unambiguous)."""
    kk = min(k + 1, ref.shape[1])
    _, d = strict.knn(ref, qry, kk, form)
    return (np.diff(d, axis=-1) != 0).all(-1)


# ---------------------------------------------------------------- golden vectors
def test_golden_square_distance(pair100):
    a, b = pair100
    assert np.array_equal(bits(strict.square_distance(a[:, :96], b[:, :64])), bits(GOLD["sqdist_small"]))
    assert np.array_equal(sha(strict.square_distance(a, b[:, :1024])), GOLD["sqdist_4096x1024_sha"])
    assert np.array_equal(sha(strict.square_distance(a[:, :1024], b)), GOLD["sqdist_1024x4096_sha"])
    assert np.array_equal(sha(strict.square_distance(a, b[:, :256])), GOLD["sqdist_permuted_sha"])


def test_golden_fps(pair100):
    a, _ = pair100
    g = GOLD["fps_4096_512"]
    assert np.array_equal(strict.farthest_point_sample(a, 512, g[:, 0]), g)
    a16, _ = synth.batch_pairs(101, 1, 16384)
    g = GOLD["fps_16384_1024"]
    assert np.array_equal(strict.farthest_point_sample(a16, 1024, g[:, 0]), g)
    dup = np.concatenate([a[:, :1500], a[:, :548]], 1)
    g = GOLD["fps_dup_2048_700"]
    assert np.array_equal(strict.farthest_point_sample(dup, 700, g[:, 0]), g)


def test_golden_fps_start_comes_from_torch_cpu_rng():
    # the reference draws torch.randint(0, N, (B,)) after manual_seed (Pointnet2Utils.py:76)
    torch.manual_seed(3000)
    assert np.array_equal(torch.randint(0, 4096, (2,), dtype=torch.long).numpy(), GOLD["fps_4096_512"][:, 0])


@pytest.mark.parametrize("r,ns,nq", [(1.0, 32, 512), (0.5, 16, 512), (0.1, 16, 256), (4.0, 8, 64)])
def test_golden_ball_query(pair100, r, ns, nq):
    a, b = pair100
    g = GOLD["ball_r%g_ns%d_q%d" % (r, ns, nq)]
    assert np.array_equal(strict.query_ball_point(r, ns, a, b[:, :nq]), g)


def test_golden_ball_query_self(pair100):
    a, _ = pair100
    assert np.array_equal(strict.query_ball_point(0.5, 16, a, a[:, ::8]), GOLD["ball_self_r0.5_ns16"])


def test_golden_index_points():
    rng = np.random.default_rng(5)
    feats = rng.normal(size=(2, 4096, 24)).astype(np.float32)
    idx = GOLD["gather_idx"].astype(np.int64)
    assert np.array_equal(sha(strict.index_points(feats, idx)), GOLD["gather_out_sha"])


@pytest.mark.parametrize("k,nq,nr", [(16, 512, 4096), (8, 256, 64), (64, 256, 256)])
def test_golden_knn_group(pair100, k, nq, nr):
    a, b = pair100
    ref, qry = a[:, :nr].copy(), b[:, :nq].copy()
    g = GOLD["knn_k%d_q%d_r%d" % (k, nq, nr)].astype(np.int64)
    mine = strict.knn_point(k, ref, qry)
    clean = tie_free_rows(ref, qry, k, strict.FORM_KNN)
    assert clean.mean() > 0.9
    assert np.array_equal(mine[clean], g[clean])
    # rows with ties: same multiset of distances, bit for bit
    full = strict.square_distance(ref, qry)                      # [B,N,S], refs are `src`
    for bi, si in np.argwhere(~clean):
        dg = np.sort(full[bi, g[bi, si], si]); dm = np.sort(full[bi, mine[bi, si], si])
        assert np.array_equal(bits(dg), bits(dm))


def test_golden_three_nn_variant_a(pair100):
    a, _ = pair100
    S, N = 64, 1024
    dense = a[:, :N].copy(); sparse = a[:, :N:N // S][:, :S].copy()
    d, idx = strict.three_nn(dense, sparse)
    w = strict.three_weights(d, 0)
    rows = GOLD["fp_a_weight_rows"]                              # [B,N,S] three non-zeros per row
    mine = np.zeros_like(rows)
    np.put_along_axis(mine, idx, w, axis=-1)
    clean = tie_free_rows(sparse, dense, 3, strict.FORM_QFIRST)
    assert clean.mean() > 0.95
    assert np.array_equal((rows != 0)[clean], (mine != 0)[clean])            # same three neighbours
    np.testing.assert_allclose(mine[clean], rows[clean], rtol=1e-5, atol=1e-7)
    feat = GOLD["fp_a_feat"].transpose(0, 2, 1).copy()            # [B,S,C]
    out = strict.three_interpolate(feat, idx, w).transpose(0, 2, 1)
    np.testing.assert_allclose(out[:, :, clean[0] & clean[1]], GOLD["fp_a_out"][:, :, clean[0] & clean[1]], rtol=1e-5, atol=1e-6)


def test_golden_three_nn_variant_b(pair100):
    a, _ = pair100
    S, N = 64, 1024
    dense = a[:, :N].copy(); sparse = a[:, :N:N // S][:, :S].copy()
    d, idx = strict.three_nn(dense, sparse)
    w = strict.three_weights(d, 1)
    feat = GOLD["fp_a_feat"].transpose(0, 2, 1).copy()
    out = strict.three_interpolate(feat, idx, w).transpose(0, 2, 1)
    clean = tie_free_rows(sparse, dense, 3, strict.FORM_QFIRST)
    m = clean[0] & clean[1]
    np.testing.assert_allclose(out[:, :, m], GOLD["fp_b_out"][:, :, m], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------- torch port == strict oracle
def test_torch_port_matches_strict(pair100):
    a, b = pair100
    A, B_ = torch.from_numpy(a[:, :2048]), torch.from_numpy(b[:, :512])
    assert np.array_equal(bits(ref_torch.dense_sqdist(A, B_).numpy()), bits(strict.square_distance(a[:, :2048], b[:, :512])))
    start = torch.tensor([3, 99])
    assert np.array_equal(ref_torch.fps(A, 128, start).numpy(), strict.farthest_point_sample(a[:, :2048], 128, start.numpy()))
    assert np.array_equal(ref_torch.ball(1.0, 32, A, B_).numpy(), strict.query_ball_point(1.0, 32, a[:, :2048], b[:, :512]))
    clean = tie_free_rows(a[:, :2048], b[:, :512], 16, strict.FORM_KNN)
    assert np.array_equal(ref_torch.knn_topk(16, A, B_).numpy()[clean], strict.knn_point(16, a[:, :2048], b[:, :512])[clean])
    feat = torch.randn(2, 512, 16, generator=torch.Generator().manual_seed(1))
    out, d, idx, w = ref_torch.three_nn_interp(A, B_, feat, variant=0)
    sd, si = strict.three_nn(a[:, :2048], b[:, :512])
    c3 = tie_free_rows(b[:, :512], a[:, :2048], 3, strict.FORM_QFIRST)
    assert np.array_equal(idx.numpy()[c3], si[c3])
    np.testing.assert_allclose(out.numpy()[c3], strict.three_interpolate(feat.numpy(), si, strict.three_weights(sd, 0))[c3], rtol=1e-5, atol=1e-6)


def test_strict_knn_direct_and_chamfer_against_dense_float64():
    a, b = synth.batch_pairs(7, 2, 600)
    d64 = ((a[:, :, None, :].astype(np.float64) - b[:, None, :, :].astype(np.float64)) ** 2).sum(-1)
    dist, idx = strict.knn_points(a, b, 4)
    ref_sorted = np.sort(d64, axis=-1)[:, :, :4]
    np.testing.assert_allclose(dist, ref_sorted, rtol=1e-5, atol=1e-6)
    loss = strict.chamfer(a, b)[0]
    ref_loss = (d64.min(2).mean(1) + d64.min(1).mean(1)).mean()
    assert abs(loss - ref_loss) <= 1e-5 * ref_loss
    tl = ref_torch.chamfer_dense(torch.from_numpy(a), torch.from_numpy(b)).item()
    assert abs(tl - ref_loss) <= 1e-5 * ref_loss


def test_strict_tie_rule_lowest_index():
    pts = synth.grid_snapped(1, 1, 400, span=3)
    q = synth.grid_snapped(2, 1, 50, span=3)
    idx, d = strict.knn(pts, q, 8, strict.FORM_KNN)
    full = strict.square_distance(pts, q)[0]                      # [N,S]
    for s in range(50):
        order = np.lexsort((np.arange(400), full[:, s]))[:8]      # by (distance, index)
        assert np.array_equal(idx[0, s], order)


def test_strict_edge_cases():
    pts = np.random.default_rng(0).normal(size=(1, 5, 3)).astype(np.float32)
    idx, _ = strict.knn(pts, pts, 5, 0)                           # k == N
    assert sorted(idx[0, 0].tolist()) == [0, 1, 2, 3, 4]
    out = strict.query_ball_point(0.01, 4, pts, pts + 100.0)      # all balls empty -> sentinel N
    assert (out == 5).all()
    with pytest.raises(IndexError):
        strict.index_points(pts, np.array([[5]]))
    assert strict.farthest_point_sample(pts, 5, np.array([2]))[0, 0] == 2


# ---------------------------------------------------------------- real reference (container only)
needs_ref = pytest.mark.skipif(not ref_loader.available(), reason="reference checkout not present (GPU box)")


@needs_ref
def test_real_reference_agrees_with_oracle_live():
    R = ref_loader.pointnet2_utils()
    a, b = synth.batch_pairs(200, 2, 1500)
    A, B_ = torch.from_numpy(a), torch.from_numpy(b[:, :300])
    assert np.array_equal(bits(R.square_distance(A, B_).numpy()), bits(strict.square_distance(a, b[:, :300])))
    assert np.array_equal(R.query_ball_point(0.8, 16, A, B_).numpy(), strict.query_ball_point(0.8, 16, a, b[:, :300]))
    torch.manual_seed(5)
    f = R.farthest_point_sample(A, 200).numpy()
    assert np.array_equal(f, strict.farthest_point_sample(a, 200, f[:, 0]))
    idx = torch.from_numpy(f)
    assert np.array_equal(R.index_points(A, idx).numpy(), strict.index_points(a, f))


@needs_ref
def test_real_reference_layers_import_with_stubs():
    L = ref_loader.layers()
    assert hasattr(L, "Group") and hasattr(L, "FeaturePropagation") and hasattr(L, "PointsFusion")


# ---------------------------------------------------------------- fused grouping (SURVEY 8f rank 1)
def _group_inputs(pair100):
    a, b = pair100
    seed, D = (int(v) for v in GOLD["group_feat_seed6"])
    feat = np.random.default_rng(seed).normal(size=(2, D, 4096)).astype(np.float32).transpose(0, 2, 1).copy()   # [B,N,D]
    return a, b, feat


def test_golden_group_forward_ball(pair100):
    # the WHOLE output of the real Group.forward (ball query, centres taken from the refs), as a digest
    a, _, feat = _group_inputs(pair100)
    centres = np.ascontiguousarray(a[:, ::8])
    idx = strict.query_ball_point(1.0, 32, a, centres)
    assert np.array_equal(sha(strict.group_points(a, centres, feat, idx)), GOLD["group_ball_self_r1_ns32_sha"])


def test_golden_group_forward_knn(pair100):
    a, b, feat = _group_inputs(pair100)
    qry = np.ascontiguousarray(b[:, :48])
    clean = tie_free_rows(a, qry, 16, strict.FORM_KNN)           # topk's order among exact ties is unspecified
    assert clean.mean() > 0.9
    mine = strict.group_points(a, qry, feat, strict.knn_point(16, a, qry))        # [B,8,16,S]
    gold = GOLD["group_knn16_q48"]
    assert mine.shape == gold.shape == (2, 8, 16, 48)
    for bi in range(2):
        assert np.array_equal(bits(mine[bi][:, :, clean[bi]]), bits(gold[bi][:, :, clean[bi]]))


def test_group_points_feature_first_order_and_no_features(pair100):
    a, b, feat = _group_inputs(pair100)
    qry = np.ascontiguousarray(b[:, :64]); idx = strict.knn_point(4, a, qry)
    x = strict.group_points(a, qry, feat, idx, xyz_first=True); f = strict.group_points(a, qry, feat, idx, xyz_first=False)
    assert x.shape == f.shape == (2, 8, 4, 64)
    assert np.array_equal(x[:, :3], f[:, 5:]) and np.array_equal(x[:, 3:], f[:, :5])      # SA-MSG puts the features first
    assert np.array_equal(strict.group_points(a, qry, None, idx), x[:, :3])


# ---------------------------------------------------------------- PolyPCI polynomial fit (SURVEY 8f rank 4)
def _polyfit_case(tag):
    T = GOLD["polyfit_%s_T" % tag]; tq, deg = GOLD["polyfit_%s_t" % tag]
    return T, float(tq), int(deg)


def test_golden_polyfit_restatement_and_linear_weights():
    from oracle import ref_polyfit
    from b200pc import polypci
    prng = np.random.default_rng(9)                                        # same draws, same order as make_golden.py
    for tag in ("f5_d3", "f7_d2"):
        T, tq, deg = _polyfit_case(tag)
        frames = (prng.normal(size=(len(T), 96)) * 30).astype(np.float32)
        gold = GOLD["polyfit_%s" % tag]
        mine = ref_polyfit.fitting_and_predict(T, frames, tq, deg).astype(np.float32)
        # same numpy calls as the real function: identical up to the LAPACK build of the machine running the test
        np.testing.assert_allclose(mine, gold, rtol=2e-6, atol=1e-6)
        # the product's formulation: ONE weight vector per batch item (least squares is linear in the data)
        w = polypci.poly_weights(T, tq, deg)
        assert w.shape == (len(T),) and w.dtype == np.float64
        np.testing.assert_allclose((w @ frames.astype(np.float64)).astype(np.float32)[None], gold, rtol=2e-6, atol=1e-6)
        assert abs(w.sum() - 1.0) < 1e-12                                 # a polynomial fit reproduces constants


# ---------------------------------------------------------------- the search kernel's conservative prefilter, emulated
def _fma32(a, b, c):
    # one rounding: the product of two fp32 is exact in fp64; the sum is rounded to fp32 once for all but ~2^-29 of the cases
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


@pytest.mark.parametrize("scale,offset", [(30.0, 0.0), (1.0, 0.0), (30.0, 2000.0), (1e-3, 0.0), (5.0, 3e5)])
def test_filter_threshold_is_conservative_for_all_three_forms(scale, offset):
    """search.cu: u = fma(z,-2qz, fma(y,-2qy, fma(x,-2qx, w'))) with w' = |r|^2 (1 - 20 eps) must satisfy
    dist_ref <= tau  =>  u < (tau - |q|^2) + 4.5e-7 |tau| + 1.1e-6 |q|^2 + 1e-35   for every reference rounding.
    Checked with tau = the pair's own distance (the tightest threshold that must still let the pair through)."""
    f32 = np.float32
    rng = np.random.default_rng(int(scale * 7 + offset) % 1000)
    n = 200000
    r = (rng.normal(size=(n, 3)) * scale + offset).astype(f32)
    q = (r + rng.normal(size=(n, 3)) * scale * rng.choice([1e-3, 1e-2, 0.1, 1.0], size=(n, 1))).astype(f32)
    sqn = lambda p: ((p[:, 0] * p[:, 0]).astype(f32) + (p[:, 1] * p[:, 1]).astype(f32)).astype(f32) + (p[:, 2] * p[:, 2]).astype(f32)
    w, nq = sqn(r).astype(f32), sqn(q).astype(f32)
    a = (f32(-2.0) * q).astype(f32)
    T = _fma32(r[:, 2], a[:, 2], _fma32(r[:, 1], a[:, 1], (r[:, 0] * a[:, 0]).astype(f32)))
    d = {0: ((T + w).astype(f32) + nq).astype(f32), 1: ((T + nq).astype(f32) + w).astype(f32)}
    dx, dy, dz = (q[:, 0] - r[:, 0]).astype(f32), (q[:, 1] - r[:, 1]).astype(f32), (q[:, 2] - r[:, 2]).astype(f32)
    d[2] = _fma32(dz, dz, _fma32(dy, dy, (dx * dx).astype(f32)))
    wp = (w * f32(1.0 - 20.0 * 5.9604645e-8)).astype(f32)
    u = _fma32(r[:, 2], a[:, 2], _fma32(r[:, 1], a[:, 1], _fma32(r[:, 0], a[:, 0], wp)))
    for form, tau in d.items():
        margin = ((f32(4.5e-7) * np.abs(tau)).astype(f32) + ((f32(1.1e-6) * nq).astype(f32) + f32(1e-35)).astype(f32)).astype(f32)
        thr = ((tau - nq).astype(f32) + margin).astype(f32)
        assert (u < thr).all(), "form %d: %d of %d pairs would be filtered out" % (form, int((~(u < thr)).sum()), n)


# ---------------------------------------------------------------- the occupancy grid of the top-k searches, emulated
def _sorted_slot(p, n_tiles, tps, TILE=512):
    """search.cu sorted_slot(): tile slot of the ref at position p of the cell order"""
    span = tps * TILE
    s = p // span
    r = p - s * span
    t = np.minimum(tps, n_tiles - s * tps)
    q = r // t
    return s * span + (r - q * t) * TILE + q


@pytest.mark.parametrize("n_tiles,tps", [(32, 32), (32, 8), (33, 8), (7, 3), (1, 1), (5, 5), (9, 2)])
def test_sorted_slot_is_a_bijection_and_every_tile_a_strided_sample(n_tiles, tps):
    n = n_tiles * 512
    p = np.arange(n, dtype=np.int64)
    sl = _sorted_slot(p, n_tiles, tps)
    assert np.array_equal(np.sort(sl), p)                                   # every slot exactly once
    for s0 in range(0, n_tiles, tps):                                       # a split's refs stay inside the split's tiles
        t = min(tps, n_tiles - s0)
        inside = (p >= s0 * 512) & (p < (s0 + t) * 512)
        assert sl[inside].min() == s0 * 512 and sl[inside].max() == (s0 + t) * 512 - 1
        for tile in range(s0, s0 + t):                                      # tile = every t-th position of the range, in order
            pos = np.sort(p[(sl // 512) == tile])
            assert np.array_equal(pos, s0 * 512 + (tile - s0) + t * np.arange(512))


def _corner_seed(ref, q, k):
    """search.cu grid_bbox_kernel + grid_corner_seed() in float64 (the kernel's fp32 slack is part of the formula)"""
    eps16 = 9.6e-7
    lo, hi = ref.min(0), ref.max(0)
    ext = hi - lo
    h = ext.max() / 128
    while True:
        dim = np.clip(np.ceil(ext / h), 1, 128).astype(np.int64)
        if dim.prod() <= 131072:
            break
        h *= 2
    cell = lambda pts, l: (np.clip(((pts - lo) / h).astype(np.int64), 0, dim - 1) >> l)
    counts = []
    for l in range(5):
        d = (dim + (1 << l) - 1) >> l
        c = cell(ref, l)
        counts.append((np.bincount((c[:, 2] * d[1] + c[:, 1]) * d[0] + c[:, 0], minlength=int(d.prod())).reshape(d[2], d[1], d[0]), d))
    max_w = float((np.maximum(np.abs(lo), np.abs(hi)) ** 2).sum()) * 1.000001
    out = np.empty(len(q))
    for i, qq in enumerate(q):
        c0 = cell(qq[None], 0)[0]
        lev, rho = -1, 1
        if counts[0][0][c0[2], c0[1], c0[0]] >= k:
            lev, rho = 0, 0
        else:
            for l in range(5):
                cn, d = counts[l]
                c = c0 >> l
                z0, z1 = max(c[2] - 1, 0), min(c[2] + 1, d[2] - 1)
                y0, y1 = max(c[1] - 1, 0), min(c[1] + 1, d[1] - 1)
                x0, x1 = max(c[0] - 1, 0), min(c[0] + 1, d[0] - 1)
                if cn[z0:z1 + 1, y0:y1 + 1, x0:x1 + 1].sum() >= k:
                    lev = l
                    break
        bound = 0.0
        for a in range(3):
            L, H = lo[a], hi[a]
            if lev >= 0:
                gl = counts[lev][1][a]
                cl = c0[a] >> lev
                a0, a1 = max(cl - rho, 0), min(cl + rho, gl - 1)
                hl = h * (1 << lev)
                L = lo[a] + a0 * hl
                Hn = lo[a] + (a1 + 1) * hl
                H = max(Hn, hi[a]) if a1 == gl - 1 else Hn
            delta = 1e-3 * h + 1e-6 * max(abs(lo[a]), abs(hi[a]))
            bound += max(abs(qq[a] - (L - delta)), abs((H + delta) - qq[a])) ** 2
        out[i] = bound * 1.00001 + eps16 * (float((qq ** 2).sum()) + max_w) + 1e-37
    return out


@pytest.mark.parametrize("k", [1, 3, 16, 64])
def test_grid_corner_threshold_bounds_the_kth_reference_distance(k):
    """the starting threshold of the gridded top-k searches must never be below the k-th smallest distance IN THE
    REFERENCE'S ROUNDING (all three forms) -- otherwise a true neighbour would be filtered out"""
    a, b = synth.batch_pairs(40, 1, 6000)
    ref, qry = a[0], b[0][:400]
    far = (qry[:40] * 3.0 + 25.0).astype(np.float32)                        # some queries outside the refs' bounding box
    rng = np.random.default_rng(k)
    cl = (rng.normal(size=(3000, 3)) * 0.02 + rng.choice([-40.0, 0.0, 55.0], size=(3000, 1))).astype(np.float32)   # three tight clusters
    for refs, qs in ((ref, qry), (ref, far), (cl, cl[::10].copy()), (ref + np.float32(2000.0), qry + np.float32(2000.0))):
        tau0 = _corner_seed(refs.astype(np.float64), qs.astype(np.float64), k)
        for form in (0, 1, 2):
            _, od = strict.knn(refs[None], qs[None], k, form)
            assert (od[0, :, k - 1].astype(np.float64) <= tau0).all(), "form %d: threshold below the k-th distance" % form


def test_fps_oracle_is_unfused_on_the_near_tie_clouds():
    """the adversarial FPS clouds: the oracle follows the unfused arithmetic (the reference's), which differs
    from the fused one on every such cloud -- so the GPU test on the same data detects a contracted kernel"""
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from adversarial import fps_rot90_cloud, first_round_pick
    for N in (301, 4097, 16385):
        c = fps_rot90_cloud(900, N // 2)
        a, b = first_round_pick(c, False), first_round_pick(c, True)
        assert a != b
        got = strict.farthest_point_sample(c[None], 2, np.array([0]))[0, 1]
        assert got == a


def test_read_bin_shapes(tmp_path):
    """b200pc.io.read_bin: the reference's np.fromfile(...).reshape(-1, 5 | 4) (Dataset/InterpolationData.py:142,
    PointINet20230424/data/interpolation_data.py:34)"""
    from b200pc import io as bio
    a = np.arange(35, dtype=np.float32); p = tmp_path / "n.bin"; a.tofile(p)
    assert bio.read_bin(str(p)).shape == (7, 5) and bio.read_bin(str(p), 5).shape == (7, 5)
    b = np.arange(24, dtype=np.float32); q = tmp_path / "k.bin"; b.tofile(q)
    assert bio.read_bin(str(q)).shape == (6, 4)
    with pytest.raises(ValueError):
        bio.read_bin(str(q), 5)
    if ref_loader.available():
        kitti, nusc = ref_loader.demo_bins()
        if nusc:
            assert bio.read_bin(nusc[0], 5).shape[1] == 5
        if kitti:
            assert bio.read_bin(kitti[0], 4).shape[0] > 100000


def test_knn_points_and_chamfer_against_an_independent_kd_tree():
    """a8 / a9 are "parity unpinned" (pytorch3d is neither vendored nor pinned by the reference).  Beside the dense float64
    formula, an INDEPENDENT implementation of the same semantics: scipy's cKDTree in float64.  On every query whose k+1
    nearest float64 distances are separated by more than fp32 rounding the oracle's indices must equal the tree's, and the
    squared distances agree to 1e-5 relative; Chamfer (point-mean + batch-mean of nearest squared distances) likewise."""
    from scipy.spatial import cKDTree
    a, b = synth.batch_pairs(77, 2, 4096)
    k = 16
    od, oi = strict.knn_points(b, a, k)
    sep_total = 0
    for bi in range(2):
        tree = cKDTree(a[bi].astype(np.float64))
        dd, ii = tree.query(b[bi].astype(np.float64), k=k + 1)
        d2 = dd ** 2
        gaps = np.diff(d2, axis=1)                                       # [S, k]
        clear = (gaps > 1e-5 * d2[:, 1:] + 1e-9).all(axis=1)            # no near-tie among the first k+1
        sep_total += int(clear.sum())
        assert np.array_equal(oi[bi][clear], ii[clear, :k])
        np.testing.assert_allclose(od[bi][clear], d2[clear, :k], rtol=1e-5, atol=1e-7)
    assert sep_total > 0.95 * 2 * 4096                                   # the comparison covers nearly every query
    loss, dx, ix, dy, iy = strict.chamfer(a, b)
    want = 0.0
    for bi in range(2):
        ta, tb = cKDTree(a[bi].astype(np.float64)), cKDTree(b[bi].astype(np.float64))
        want += (tb.query(a[bi].astype(np.float64))[0] ** 2).mean() + (ta.query(b[bi].astype(np.float64))[0] ** 2).mean()
    assert abs(loss - want / 2) <= 1e-5 * abs(want / 2)


# ---------------------------------------------------------------- non-finite coordinates (include/b200pc.h, "Non-finite")
# The rule every search follows: a (query, ref) pair is a candidate only if its distance is finite.  A row holds its
# candidates in ascending (distance, index) order, then -1 with distance +inf.  The restatements below compute the same
# distances as the oracle's forms with numpy and apply that rule with a plain lexsort.
def _dense_form(ref, qry, form):
    """[B,S,N] distances in the oracle's rounding: forms 0 / 1 from square_distance, form 2 emulated (direct, FMA)"""
    if form == 0:
        return strict.square_distance(ref, qry).transpose(0, 2, 1)
    if form == 1:
        return strict.square_distance(qry, ref)
    f32 = np.float32
    with np.errstate(invalid="ignore", over="ignore"):
        d = (qry[:, :, None, :] - ref[:, None, :, :]).astype(f32)          # q - r: squared, so the sign is irrelevant
        acc = (d[..., 0] * d[..., 0]).astype(f32)
        acc = _fma32(d[..., 1], d[..., 1], acc)
        return _fma32(d[..., 2], d[..., 2], acc)


def _topk_finite(dist, k):
    """the k smallest finite entries of every row of dist [..., N] by (value, index), padded with (-1, +inf)"""
    flat = dist.reshape(-1, dist.shape[-1])
    idx = np.full((flat.shape[0], k), -1, np.int64)
    val = np.full((flat.shape[0], k), np.inf, np.float32)
    for r, row in enumerate(flat):
        cand = np.flatnonzero(np.isfinite(row))
        order = cand[np.lexsort((cand, row[cand]))][:k]
        idx[r, :len(order)] = order
        val[r, :len(order)] = row[order]
    return idx.reshape(dist.shape[:-1] + (k,)), val.reshape(dist.shape[:-1] + (k,))


def _non_finite_cloud(seed, B, N, S):
    """refs and queries with NaN, +inf and -inf in one or all three coordinates, mixed-sign finite coordinates, a
    (+inf, 0, 0) query, and -- for B > 1 -- a last batch item whose refs are all non-finite"""
    rng = np.random.default_rng(seed)
    ref = rng.normal(size=(B, N, 3)).astype(np.float32) * 4
    qry = rng.normal(size=(B, S, 3)).astype(np.float32) * 4
    bad = [np.nan, np.inf, -np.inf]
    for b in range(B):
        for j, n in enumerate(rng.choice(N, size=N // 5, replace=False)):
            if j % 3 == 0:
                ref[b, n] = bad[j % 9 // 3]
            else:
                ref[b, n, j % 3] = bad[j % 2]
    qry[:, 0] = [np.inf, 0.0, 0.0]
    qry[:, 1] = [np.nan, 1.0, 1.0]
    qry[:, 2] = -np.inf
    qry[:, 3] = [0.5, np.inf, -np.inf]
    if B > 1:
        ref[-1, :, rng.integers(0, 3)] = np.nan
        ref[-1, ::2] = np.inf
    return ref, qry


def test_non_finite_knn_keeps_only_finite_candidates_in_the_issue_case():
    # 40 refs: refs 3 and 20..25 are NaN and ref 10 has y = +inf, so 32 refs are finite; the queries are finite
    rng = np.random.default_rng(1)
    ref = rng.normal(size=(1, 40, 3)).astype(np.float32)
    ref[0, [3, 20, 21, 22, 23, 24, 25]] = np.nan
    ref[0, 10, 1] = np.inf
    qry = rng.normal(size=(1, 6, 3)).astype(np.float32)
    finite = np.setdiff1d(np.arange(40), [3, 10, 20, 21, 22, 23, 24, 25])
    for form in (0, 1, 2):
        full = _dense_form(ref, qry, form)
        for k in (4, 32, 33, 40):
            idx, dist = strict.knn(ref, qry, k, form)
            want_i, want_d = _topk_finite(full, k)
            np.testing.assert_array_equal(idx, want_i)
            np.testing.assert_array_equal(bits(dist), bits(want_d))
            n = min(k, 32)
            assert np.isin(idx[..., :n], finite).all() and (idx[..., n:] == -1).all() and np.isinf(dist[..., n:]).all()
            assert (np.diff(dist[..., :n], axis=-1) >= 0).all()


@pytest.mark.parametrize("form", [0, 1, 2])
@pytest.mark.parametrize("k", [1, 8, 30, 50])             # below, at and above the 40 finite refs of the first item
def test_non_finite_knn_matches_restatement(form, k):
    ref, qry = _non_finite_cloud(2, 3, 50, 12)
    idx, dist = strict.knn(ref, qry, k, form)
    want_i, want_d = _topk_finite(_dense_form(ref, qry, form), k)
    np.testing.assert_array_equal(idx, want_i)
    np.testing.assert_array_equal(bits(dist), bits(want_d))
    assert (idx[-1] == -1).all()                           # the item without a finite ref ranks nothing
    assert (idx[:, 0:4] == -1).all()                       # nor do the non-finite queries
    assert (idx[:2, 4:, :min(k, 40)] >= 0).all()           # a finite query ranks every finite ref


def test_non_finite_knn_ties_by_index():
    # grid-snapped points: exact arithmetic and many equal distances, with NaN refs between them
    ref = synth.grid_snapped(3, 1, 300, span=3).copy()
    ref[0, 7::11] = np.nan
    qry = synth.grid_snapped(4, 1, 40, span=3)
    for form in (0, 1, 2):
        full = _dense_form(ref, qry, form)
        idx, dist = strict.knn(ref, qry, 16, form)
        want_i, want_d = _topk_finite(full, 16)
        assert (np.diff(want_d, axis=-1) == 0).any(-1).mean() > 0.5
        np.testing.assert_array_equal(idx, want_i)
        np.testing.assert_array_equal(bits(dist), bits(want_d))


def test_non_finite_nearest_and_chamfer():
    x, y = _non_finite_cloud(5, 2, 60, 30)
    for a, b in ((x, y), (y, x)):
        mn, arg = strict.nearest(a, b)
        want_i, want_d = _topk_finite(_dense_form(b, a, 2), 1)
        np.testing.assert_array_equal(arg, want_i[..., 0])
        np.testing.assert_array_equal(bits(mn), bits(want_d[..., 0]))
    loss, dx, ix, dy, iy = strict.chamfer(x, y)
    assert loss == np.inf and (ix[1] == -1).all() and (dy[1] == np.inf).all()
    # finite clouds: the loss stays finite and matches the float64 formula
    xf, yf = x[:1, 4:].copy(), y[:1].copy()
    xf[~np.isfinite(xf).all(-1)] = 0.25
    yf[~np.isfinite(yf).all(-1)] = -0.5
    loss = strict.chamfer(xf, yf)[0]
    d64 = ((xf[:, :, None].astype(np.float64) - yf[:, None].astype(np.float64)) ** 2).sum(-1)
    want = (d64.min(2).mean(1) + d64.min(1).mean(1)).mean()
    assert abs(loss - want) <= 1e-5 * want


def test_non_finite_ball_query_never_hits():
    ref, qry = _non_finite_cloud(6, 2, 80, 20)
    for radius, ns in ((1.0, 8), (3.0, 32), (1e3, 80)):
        got = strict.query_ball_point(radius, ns, ref, qry)
        d = _dense_form(ref, qry, 1)
        hit = d <= strict.radius_sq(radius)                # NaN compares false: never a hit
        want = np.full(got.shape, 80, np.int64)
        for b, s in np.ndindex(2, 20):
            h = np.flatnonzero(hit[b, s])[:ns]
            if len(h):
                want[b, s] = h[0]
                want[b, s, :len(h)] = h
        np.testing.assert_array_equal(got, want)
        assert (got[1] == 80).all() and (got[:, :4] == 80).all()


def test_three_interpolate_applies_the_kernels_index_rule():
    # -1 (an unfilled three-NN slot) wraps once to the last row, like Python indexing; anything still out of range reads
    # row 0 with weight 0 -- the kernels' clean_neighbour
    rng = np.random.default_rng(7)
    feat = rng.normal(size=(2, 5, 4)).astype(np.float32)
    feat[1, 0, 2] = np.inf
    idx = np.array([[[0, 1, -1], [-5, 4, 2], [6, -6, 3], [-1, -1, -1]]] * 2, np.int64)
    w = rng.uniform(0.1, 1, size=(2, 4, 3)).astype(np.float32)
    got = strict.three_interpolate(feat, idx, w)
    want = np.empty_like(got)
    for b, n in np.ndindex(2, 4):
        terms = []
        for j in range(3):
            i, ww = idx[b, n, j], w[b, n, j]
            i = i + 5 if i < 0 else i
            if not 0 <= i < 5:
                i, ww = 0, np.float32(0)
            with np.errstate(invalid="ignore"):
                terms.append((feat[b, i] * ww).astype(np.float32))
        want[b, n] = ((terms[0] + terms[1]).astype(np.float32) + terms[2]).astype(np.float32)
    np.testing.assert_array_equal(bits(got), bits(want))
    assert np.isnan(got[1, 2, 2])                          # 0 * inf of a dropped neighbour, as on the device


@pytest.mark.parametrize("start", [0, 3, 5, 9])
def test_non_finite_fps_matches_the_reference_loop(start):
    # NaN and +inf distances never lower a running minimum (the reference's `dist < distance` mask); 1e30 points square to
    # +inf; a non-finite start leaves every minimum at 1e10
    a, _ = synth.batch_pairs(8, 2, 300)
    a = a.copy()
    a[:, 3] = np.nan; a[:, 5, 1] = np.inf; a[:, 9, 0] = -np.inf; a[:, 40] = 1e30; a[:, 41, 2] = -1e30; a[1, 100:110, 2] = np.nan
    st = np.array([start, start])
    want = ref_torch.fps(torch.from_numpy(a), 64, torch.from_numpy(st)).numpy()
    np.testing.assert_array_equal(strict.farthest_point_sample(a, 64, st), want)
