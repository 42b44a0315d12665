"""Oracles of the ragged-batch entries (b200pc_knn_ragged, b200pc_chamfer_ragged_*, the pytorch3d shim with lengths).

* kNN: oracle.strict.knn per item on ref[b, :n_b] / qry[b, :s_b] (n_b, s_b = the lengths clamped to [0, N] / [0, S]), padded
  with -1 / +inf -- the project's convention for slots without a candidate.
* Chamfer: a float64 torch restatement of pytorch3d.loss.chamfer_distance with x_lengths / y_lengths (its knn_points pads
  the slots beyond lengths2 with distance 0, its masks zero the points beyond lengths1), both reductions, differentiable.
"""
import numpy as np
import torch

from oracle import strict


def clamp_lengths(lengths, full, B):
    if lengths is None:
        return np.full(B, full, np.int64)
    return np.clip(np.asarray(lengths, np.int64), 0, full)


def knn(ref, qry, ref_len, qry_len, k, form):
    """-> (idx int64 [B,S,k], dist fp32 [B,S,k]) of the ragged search"""
    ref = np.asarray(ref, np.float32); qry = np.asarray(qry, np.float32)
    B, N, _ = ref.shape; S = qry.shape[1]
    n = clamp_lengths(ref_len, N, B); s = clamp_lengths(qry_len, S, B)
    idx = np.full((B, S, k), -1, np.int64)
    dist = np.full((B, S, k), np.inf, np.float32)
    for b in range(B):
        if n[b] == 0 or s[b] == 0:
            continue
        kk = min(k, int(n[b]))
        oi, od = strict.knn(ref[b:b + 1, :n[b]].copy(), qry[b:b + 1, :s[b]].copy(), kk, form)
        idx[b, :s[b], :kk] = oi[0]
        dist[b, :s[b], :kk] = od[0]
    return idx, dist


def chamfer_terms(x, y, x_len, y_len):
    """per-point terms of the ragged Chamfer entry: (sums [B,2] float64, dx [B,N] fp32, ix, dy [B,M] fp32, iy) with -1 / +inf for
    padded points and for points whose other cloud is empty"""
    x = np.asarray(x, np.float32); y = np.asarray(y, np.float32)
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    ix, dx = knn(y, x, y_len, x_len, 1, strict.FORM_DIRECT)
    iy, dy = knn(x, y, x_len, y_len, 1, strict.FORM_DIRECT)
    nx = clamp_lengths(x_len, N, B); ny = clamp_lengths(y_len, M, B)
    sums = np.zeros((B, 2), np.float64)
    for b in range(B):
        sums[b, 0] = dx[b, :nx[b], 0].astype(np.float64).sum()
        sums[b, 1] = dy[b, :ny[b], 0].astype(np.float64).sum()
    return sums, dx[..., 0], ix[..., 0], dy[..., 0], iy[..., 0]


def chamfer_distance64(x, y, x_len=None, y_len=None, point_reduction="mean", batch_reduction="mean"):
    """pytorch3d.loss.chamfer_distance (norm 2, no weights / normals) restated in float64 torch; x, y may require grad."""
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    nx = torch.as_tensor(clamp_lengths(None if x_len is None else np.asarray(x_len), N, B))
    ny = torch.as_tensor(clamp_lengths(None if y_len is None else np.asarray(y_len), M, B))

    def one_direction(a, bpts, na, nb):
        terms = []
        for i in range(B):
            if na[i] == 0:
                terms.append(a.new_zeros(()))
                continue
            if nb[i] == 0:                     # every slot of the knn is padding: distance 0
                terms.append(a.new_zeros(()))
                continue
            d = ((a[i, :na[i], None, :] - bpts[i, None, :nb[i], :]) ** 2).sum(-1)
            terms.append(d.min(dim=1).values.sum())
        c = torch.stack(terms)
        if point_reduction == "mean":
            c = c / na.clamp(min=1).to(c.dtype)
        if batch_reduction is not None:
            c = c.sum()
            if batch_reduction == "mean":
                c = c / max(B, 1)
        return c

    return one_direction(x, y, nx, ny) + one_direction(y, x, ny, nx)
