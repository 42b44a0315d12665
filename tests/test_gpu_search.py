"""GPU parity of the neighbour searches (kNN, three-NN, knn_points, ball query) against the strict
oracle.  Bar: indices and distances BIT-EXACT on every row, ties included (the oracle and the
kernels both realise the total order (distance, index); SURVEY Appendix A.4 rule 3)."""
import numpy as np
import pytest
import torch

from b200pc import ops, pointnet2_utils as P, pytorch3d_shim as S3, synth
from oracle import strict
from test_gpu_plans import Knobs, expect     # sets knobs and reads back the plan that ran (B200PC_DEBUG_PLAN)

pytestmark = pytest.mark.gpu


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


CASES = [
    # (B, N refs, S queries, k)   -- shapes from SURVEY section 8a plus ragged/edge sizes
    (2, 4096, 2048, 16),
    (1, 256, 256, 64),      # FlowEmbedding, Models.py:33
    (2, 16, 64, 8),         # SetUpConv 64x16
    (1, 64, 256, 8),
    (1, 1000, 777, 1),      # ragged: N, S not multiples of anything
    (3, 513, 31, 3),        # one ref past a tile boundary
    (1, 5, 9, 5),           # k == N
    (1, 2048, 100, 32),
    (2, 1024, 256, 8),      # SetUpConv 1024 x 256 (refs = 256 in the model; both orientations are small-path shapes)
    (1, 700, 5000, 16),     # small refs, many queries: the planner keeps the streaming kernel
    (1, 1024, 64, 100),     # large k on the warp-per-query path
    (1, 4096, 300, 128),    # large k on the streaming kernel (SA-MSG style nsample 128)
]


@pytest.mark.parametrize("small_path", ["1", "0"])     # N <= 1024: warp-per-query kernel vs the streaming kernel
@pytest.mark.parametrize("B,N,S,k", CASES)
@pytest.mark.parametrize("form", [0, 1, 2])
def test_knn_matches_strict_oracle(cuda_dev, monkeypatch, B, N, S, k, form, small_path):
    if small_path == "0":
        if N > 1024:
            pytest.skip("streaming kernel is the only path for N > 1024")
        monkeypatch.setenv("B200PC_SMALL_PATH", "0"); ops.reload_tuning()
    a, b = synth.batch_pairs(10, B, max(N, S))
    ref, qry = a[:, :N].copy(), b[:, :S].copy()
    idx, dist = ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), k, form, want_dist=True)
    oi, od = strict.knn(ref, qry, k, form)
    assert idx.dtype == torch.int64 and idx.shape == (B, S, k)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))


@pytest.mark.parametrize("form", [0, 1, 2])
def test_knn_tie_stress_lowest_index_wins(cuda_dev, form):
    # grid-snapped coordinates: all arithmetic exact, many exactly equal distances and duplicates
    ref = synth.grid_snapped(7, 2, 3000, span=6)
    qry = synth.grid_snapped(8, 2, 500, span=6)
    idx, dist = ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), 16, form, want_dist=True)
    oi, od = strict.knn(ref, qry, 16, form)
    ties = (od[:, :, 1:] == od[:, :, :-1]).any(-1).mean()
    assert ties > 0.5, "the stress set is supposed to be full of ties"
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))


def test_knn_split_path_small_query_count(cuda_dev, monkeypatch, capfd):
    # few queries against many refs -> the ref range is split over gridDim.z and merged
    knobs = Knobs(monkeypatch, capfd)
    knobs.set()
    a, b = synth.batch_pairs(3, 1, 16384)
    ref, qry = a, b[:, :1024].copy()
    for k, form in ((8, 0), (16, 2), (3, 1)):
        (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), k, form, want_dist=True))
        assert len(plans) == 1 and int(plans[0]["split"]) > 1, plans      # the planner still serves the split path here
        oi, od = strict.knn(ref, qry, k, form)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)
        np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))


def test_knn_sorted_input_order_worst_case(cuda_dev):
    # refs sorted by decreasing distance from the queries' region: every ref is a candidate
    rng = np.random.default_rng(0)
    ref = np.sort(rng.uniform(1.0, 50.0, size=(1, 3000, 1)).astype(np.float32), axis=1)[:, ::-1]
    ref = np.concatenate([ref, np.zeros_like(ref), np.zeros_like(ref)], -1).copy()
    qry = rng.normal(0, 0.1, size=(1, 200, 3)).astype(np.float32)
    idx = P.knn_point(16, _t(ref, cuda_dev), _t(qry, cuda_dev))
    np.testing.assert_array_equal(idx.cpu().numpy(), strict.knn_point(16, ref, qry))


def test_knn_k_larger_than_n_raises(cuda_dev):
    ref = torch.zeros(1, 4, 3, device=cuda_dev); qry = torch.zeros(1, 2, 3, device=cuda_dev)
    with pytest.raises(RuntimeError):
        P.knn_point(5, ref, qry)


def test_cpu_tensor_is_rejected_no_fallback():
    with pytest.raises(RuntimeError):
        P.knn_point(2, torch.zeros(1, 4, 3), torch.zeros(1, 2, 3))


BALL_CASES = [
    # (B, N, S, radius, nsample)  -- FlowNet3D SetConv shapes (Models.py:31-35) and C2's
    (1, 16384, 1024, 0.5, 16),
    (2, 1024, 256, 1.0, 16),
    (1, 256, 64, 2.0, 8),
    (2, 64, 16, 4.0, 8),
    (2, 4096, 4096, 1.0, 32),
    (1, 999, 333, 0.3, 16),
    (1, 3000, 500, 0.1, 32),   # ISAPCI SA-MSG radius: mostly tiny / empty balls
    (1, 8192, 700, 3.0, 128),  # nsample 128, dense balls
]


@pytest.mark.parametrize("small_path", ["1", "0"])
@pytest.mark.parametrize("B,N,S,radius,nsample", BALL_CASES)
def test_ball_query_matches_strict_oracle(cuda_dev, monkeypatch, B, N, S, radius, nsample, small_path):
    if small_path == "0":
        if N > 1024:
            pytest.skip("streaming kernel is the only path for N > 1024")
        monkeypatch.setenv("B200PC_SMALL_PATH", "0"); ops.reload_tuning()
    a, b = synth.batch_pairs(20, B, max(N, S))
    xyz, new_xyz = a[:, :N].copy(), b[:, :S].copy()
    out = P.query_ball_point(radius, nsample, _t(xyz, cuda_dev), _t(new_xyz, cuda_dev))
    exp = strict.query_ball_point(radius, nsample, xyz, new_xyz)
    assert out.dtype == torch.int64 and out.shape == (B, S, nsample)
    np.testing.assert_array_equal(out.cpu().numpy(), exp)


def test_ball_query_empty_ball_sentinel_is_n(cuda_dev):
    xyz = np.zeros((1, 100, 3), np.float32); xyz[0, :, 0] = np.arange(100)
    q = np.array([[[1000.0, 0, 0], [5.2, 0, 0]]], np.float32)
    out = P.query_ball_point(0.5, 4, _t(xyz, cuda_dev), _t(q, cuda_dev)).cpu().numpy()
    assert (out[0, 0] == 100).all()          # the reference's out-of-range sentinel, not clamped
    np.testing.assert_array_equal(out[0, 1], [5, 5, 5, 5])


def test_ball_query_subset_queries_self_included(cuda_dev):
    # queries are a subset of the refs (the SetConv situation): d(self) is ~0 but may be slightly negative
    a, _ = synth.batch_pairs(30, 2, 4096)
    q = a[:, ::4].copy()
    out = P.query_ball_point(0.5, 16, _t(a, cuda_dev), _t(q, cuda_dev))
    np.testing.assert_array_equal(out.cpu().numpy(), strict.query_ball_point(0.5, 16, a, q))


def test_three_nn_and_weights(cuda_dev):
    a, _ = synth.batch_pairs(40, 2, 4096)
    known = a[:, ::16].copy()   # 256 sparse points
    for variant in (0, 1):
        dist, idx, w = P.three_nn_weights(_t(a, cuda_dev), _t(known, cuda_dev), variant=variant)
        od, oi = strict.three_nn(a, known)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)
        np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
        ow = strict.three_weights(od, variant)
        # tolerance stated by north_star: 1e-5 relative on fp32 values
        np.testing.assert_allclose(w.cpu().numpy(), ow, rtol=1e-5, atol=1e-12)


def test_knn_points_shim_contract(cuda_dev):
    a, b = synth.batch_pairs(50, 2, 2048)
    p1, p2 = _t(b, cuda_dev), _t(a, cuda_dev)
    r = S3.knn_points(p1, p2, K=16, return_nn=True)
    od, oi = strict.knn_points(b, a, 16)
    np.testing.assert_array_equal(r.idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(r.dists.cpu().numpy()), _bits(od))
    np.testing.assert_array_equal(r.knn.cpu().numpy(), strict.index_points(a, oi))
    g = S3.knn_gather(p2, r.idx)
    assert torch.equal(g, r.knn)
    # K=1 (PolyPCI.rebuild, Models_V1.py:113)
    r1 = S3.knn_points(p1, p2, K=1, return_nn=True)
    assert torch.equal(r1.idx, r.idx[:, :, :1])


def test_c2_full_size_properties(cuda_dev):
    """BASELINE config 2 at full size (B=8, 16384 x 16384, k=16): sortedness, self-consistency
    of distances, and a sampled exact check against the oracle."""
    a, b = synth.batch_pairs(0, 8, 16384)
    ref, qry = _t(a, cuda_dev), _t(b, cuda_dev)
    idx, dist = ops.knn_search(ref, qry, 16, 0, want_dist=True)
    d = dist.cpu().numpy(); i = idx.cpu().numpy()
    assert (np.diff(d, axis=-1) >= 0).all()
    assert i.min() >= 0 and i.max() < 16384
    assert all(len(set(r)) == 16 for r in i[0, :64])
    sel = np.arange(0, 16384, 97)
    oi, od = strict.knn(a[:2], b[:2, sel], 16, 0)
    np.testing.assert_array_equal(i[:2, sel], oi)
    np.testing.assert_array_equal(_bits(d[:2, sel]), _bits(od))
    ball = P.query_ball_point(1.0, 32, ref, qry).cpu().numpy()
    np.testing.assert_array_equal(ball[:1, sel], strict.query_ball_point(1.0, 32, a[:1], b[:1, sel]))


# ---- the conservative prefilter (search.cu filter_threshold): exactness must not depend on magnitudes ----
@pytest.mark.parametrize("form", [0, 1, 2])
@pytest.mark.parametrize("offset,scale", [((1000.0, -2500.0, 300.0), 1.0),     # far from the origin: the filter margin is large
                                          ((0.0, 0.0, 0.0), 1e-12),            # tiny magnitudes
                                          ((3.0e5, 1.0e5, -2.0e5), 50.0)])     # expanded form cancels catastrophically
def test_knn_exact_far_from_origin_and_tiny(cuda_dev, form, offset, scale):
    # Known limit, not covered here: when the dot products themselves are SUBNORMAL (coordinates below ~1e-19) folding
    # the reference's "-2 *" into the query, s.(-2d) instead of -2(s.d), rounds at a different bit and the expanded
    # forms differ from the oracle by 1-3 denormal ulps (measured at scale 1e-20; the direct form stays exact).
    a, b = synth.batch_pairs(21, 2, 3000)
    off = np.asarray(offset, np.float32)
    ref = (a[:, :3000] * np.float32(scale) + off).astype(np.float32)
    qry = (b[:, :700] * np.float32(scale) + off).astype(np.float32)
    idx, dist = ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), 16, form, want_dist=True)
    oi, od = strict.knn(ref, qry, 16, form)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)


def test_ball_query_exact_far_from_origin(cuda_dev):
    a, b = synth.batch_pairs(22, 2, 4096)
    off = np.asarray((800.0, 1200.0, -50.0), np.float32)
    ref, qry = (a + off).astype(np.float32), (b[:, :512] + off).astype(np.float32)
    for r, ns in ((0.7, 16), (2.0, 32)):
        out = P.query_ball_point(r, ns, _t(ref, cuda_dev), _t(qry, cuda_dev))
        np.testing.assert_array_equal(out.cpu().numpy(), strict.query_ball_point(r, ns, ref, qry))


@pytest.mark.parametrize("form", [0, 1, 2])
def test_broadcast_filter_fallback_matches(cuda_dev, monkeypatch, capfd, form):
    # B200PC_FILTER=0 keeps the queries in registers and broadcasts the refs (the warm-up filter, used for the whole
    # tile): same results by construction, kept under test because it is the A/B baseline of the lane filter
    knobs = Knobs(monkeypatch, capfd)
    knobs.set()
    a, b = synth.batch_pairs(23, 1, 5000)
    ref, qry = a[:, :5000].copy(), b[:, :1500].copy()
    want, plans, _ = knobs.run(lambda: ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), 16, form, want_dist=True))
    expect(plans, filter="lane")
    knobs.set(FILTER=0)
    got, plans, _ = knobs.run(lambda: ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), 16, form, want_dist=True))
    expect(plans, filter="broadcast")
    assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])
    oi, od = strict.knn(ref, qry, 16, form)
    np.testing.assert_array_equal(got[0].cpu().numpy(), oi)


def test_randomised_shapes_scales_and_ties_fuzz(cuda_dev):
    # 60 random (B, N, S, k, form, scale, offset, duplicates, small-path) draws, kNN and ball query, bit-exact against the
    # oracle; tools/fuzz_search.py is the same loop for longer runs (1 700 cases clean at the time of writing)
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("fuzz_search", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "fuzz_search.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    assert mod.run(60, 11, cuda_dev) == 0


@pytest.mark.parametrize("form", [0, 2])
def test_knn_spatially_sorted_clouds_exact_and_not_pathological(cuda_dev, monkeypatch, capfd, form):
    # a scan-ordered / spatially sorted cloud is the adversarial arrival order for a streaming k-best; the strided
    # tiles (search.cu slot_to_ref) make it behave like a shuffled one.  Results are identical either way.
    knobs = Knobs(monkeypatch, capfd)
    knobs.set()
    a, b = synth.batch_pairs(31, 2, 16384)
    order = lambda x: np.stack([c[np.lexsort((c[:, 2], c[:, 1], np.round(c[:, 0])))] for c in x])     # sorted along x, then y
    ref, qry = order(a), order(b)[:, ::8].copy()
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, 16, form, want_dist=True))
    expect(plans, order="strided")
    oi, od = strict.knn(ref, qry, 16, form)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    knobs.set(NATURAL_ORDER=1)                                            # refs visited in index order: same answer
    (idx2, dist2), plans, _ = knobs.run(lambda: ops.knn_search(r, q, 16, form, want_dist=True))
    expect(plans, order="natural")
    assert torch.equal(idx, idx2) and torch.equal(dist, dist2)


@pytest.mark.parametrize("small_path", ["1", "0"])
def test_ball_query_non_finite_inputs_same_on_both_paths(cuda_dev, monkeypatch, small_path):
    """a NaN / inf coordinate makes NaN distances: never a hit, whichever kernel path serves the call (the streaming and the
    warp-per-query kernels use the same predicate d <= r2); rows with finite inputs are unaffected"""
    if small_path == "0":
        monkeypatch.setenv("B200PC_SMALL_PATH", "0"); ops.reload_tuning()
    a, b = synth.batch_pairs(12, 1, 900)
    ref, qry = a.copy(), b[:, :200].copy()
    ref[0, 5] = [np.nan, 0.0, 0.0]; ref[0, 17] = [np.inf, 1.0, 2.0]
    qry[0, 3] = [np.nan, np.nan, np.nan]
    got = P.query_ball_point(1.5, 16, _t(ref, cuda_dev), _t(qry, cuda_dev)).cpu().numpy()
    clean = ref.copy(); clean[0, 5] = 1e6; clean[0, 17] = -1e6                   # the same cloud with the bad points moved far away
    want = strict.query_ball_point(1.5, 16, clean, np.nan_to_num(qry, nan=1e7))
    assert not np.isin(got, [5, 17]).any()
    np.testing.assert_array_equal(np.delete(got, 3, axis=1), np.delete(want, 3, axis=1))
    assert (got[0, 3] == 900).all()                                              # the NaN query: empty ball -> N
