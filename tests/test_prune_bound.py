"""The block bound of the pruned search (csrc/search.cu section 3b, prune_lb), emulated on the host in fp32.

Claim: for every (query, block) pair, LB <= the smallest of the reference's rounded distances from the query to the block's
refs, in every form -- so a block that holds a ref with distance <= tau is never pruned.  The distances are oracle/strict's
(the reference's arithmetic); LB is prune_lb's sequence of fp32 operations (numpy float32 rounds every operation to
nearest; an FMA is emulated in float64, exact for the product, which can differ from a true FMA by double rounding in rare
ties -- far inside the bound's slack of two to three times its worst case).  Blocks are compact clusters of 64 refs, at
extents from 1e-3 to 1e4 and offsets up to 3e5, with queries inside, next to and far from them: ~1.05 M pairs."""
import numpy as np
import pytest

from oracle import strict

F = np.float32
NB, BLOCK, S = 64, 64, 1024


def _fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F)


def _sq_norm(p):
    return (p[..., 0] * p[..., 0] + p[..., 1] * p[..., 1]) + p[..., 2] * p[..., 2]


def prune_lb(lo, hi, w, q, nq):
    """prune_lb of search.cu: lo, hi [NB, 3], w [NB] (largest fl|r|^2), q [S, 3], nq [S] -> [S, NB]"""
    lo, hi, q = lo[None], hi[None], q[:, None]
    g = np.maximum(np.maximum(lo - q, q - hi), F(0))
    G = _fma(g[..., 2], g[..., 2], _fma(g[..., 1], g[..., 1], g[..., 0] * g[..., 0]))
    sub = _fma(np.full(G.shape, F(1.2e-6)), (nq[:, None] + w[None]).astype(F), np.full(G.shape, F(1e-37)))
    with np.errstate(invalid="ignore", over="ignore"):
        lb = G * F(1.0 - 2.0 ** -19) - sub
    return np.where(G < F(2.0 ** 126), lb, F(-np.inf))


def _case(seed, extent, offset):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(-1.0, 1.0, (NB, 3)) * extent
    spread = extent * rng.uniform(0.005, 0.1, (NB, 1, 1))
    ref = (centres[:, None, :] + rng.normal(size=(NB, BLOCK, 3)) * spread + offset).astype(F).reshape(-1, 3)
    near = ref[rng.integers(0, NB * BLOCK, S // 2)] + rng.normal(size=(S // 2, 3)) * extent * 0.02
    far = rng.uniform(-1.5, 1.5, (S - S // 2, 3)) * extent + offset
    qry = np.concatenate([near, far]).astype(F)
    return ref, qry


@pytest.mark.parametrize("offset", [0.0, 1e3, 3e5, -3e5])
@pytest.mark.parametrize("extent", [1e-3, 1.0, 100.0, 1e4])
def test_block_bound_never_exceeds_the_reference_distance(extent, offset):
    ref, qry = _case(int(extent * 7 + offset) & 0xffff, extent, offset)
    blocks = ref.reshape(NB, BLOCK, 3)
    lo, hi = blocks.min(1), blocks.max(1)
    w = _sq_norm(blocks).max(1)
    nq = _sq_norm(qry)
    lb = prune_lb(lo, hi, w, qry, nq)
    scale = nq[:, None] + w[None]                       # the expanded forms' rounding error is ~1e-6 of this
    tight = []
    for form in (0, 1, 2):
        idx, dist = strict.knn(ref[None], qry[None], NB * BLOCK, form)
        D = np.empty((S, NB * BLOCK), F)
        np.put_along_axis(D, idx[0], dist[0], 1)
        dmin = D.reshape(S, NB, BLOCK).min(2)           # the smallest rounded distance of every (query, block) pair
        bad = lb > dmin
        assert not bad.any(), (form, np.argwhere(bad)[:5], lb[bad][:5], dmin[bad][:5])
        clear = dmin > 1e-3 * scale
        if clear.sum() > 1000:
            tight.append(np.median(lb[clear] / dmin[clear]))
    # not a vacuous bound: where the distance stands clear of the rounding error, LB is close to it
    assert all(t > 0.9 for t in tight), tight


def test_overflowing_and_non_finite_bounds_visit():
    lo = np.array([[3e19, 0, 0]], F); hi = lo.copy()
    q = np.array([[-3e19, 0, 0], [0, 0, 0]], F)
    with np.errstate(over="ignore"):
        lb = prune_lb(lo, hi, _sq_norm(lo), q, _sq_norm(q))
    assert np.isneginf(lb).all()                        # G >= 2^126 (or |r|^2 = inf): the block is always visited
