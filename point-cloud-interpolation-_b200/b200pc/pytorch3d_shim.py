"""pytorch3d-shaped entry points backed by libb200pc.so.

The reference imports `knn_points`, `knn_gather` (Utils/Layers.py:10, PolyPCI/Models/Models_V1.py:12,
PointINet20230424/models/layers.py:16) and `chamfer_distance` (Utils/Utils.py:9) from pytorch3d,
which it neither vendors nor pins.  These functions reproduce the call signatures and the
documented semantics the reference relies on: squared L2 in direct form, K results ascending,
ties to the lower index, int64 indices; chamfer with point_reduction = batch_reduction = "mean".
Ragged batches (`lengths1` / `lengths2`, `lengths`, `x_lengths` / `y_lengths`) and the other Chamfer reductions follow
pytorch3d's documentation: the ops keep the project's -1 / +inf for empty slots, and this module turns only the slots that
are empty BECAUSE OF the lengths into pytorch3d's zero padding.
PARITY UNPINNED: no golden vector for this arithmetic exists in the reference, and pytorch3d is not installed here.
"""
from collections import namedtuple

import torch

from . import ops

_KNN = namedtuple("KNN", "dists idx knn")


def knn_gather(x, idx, lengths=None):
    """x [B,M,C], idx [B,N,K] -> [B,N,K,C].  lengths [B] (valid points of each cloud of x): slots k >= lengths[b] are
    zero-filled, as pytorch3d's knn_gather does."""
    out = ops.gather(x, idx)
    if lengths is not None:
        K = idx.shape[-1]
        lengths = ops._lengths(lengths, x.shape[0], out.device, "lengths")
        pad = lengths[:, None] <= torch.arange(K, device=out.device)[None]               # [B,K]
        out = torch.where(pad[:, None, :, None], out.new_zeros(()), out)
    return out


def knn_points(p1, p2, lengths1=None, lengths2=None, norm=2, K=1, version=-1, return_nn=False, return_sorted=True):
    """for every point of p1 [B,P1,3] its K nearest points of p2 [B,P2,3].
    -> KNN(dists [B,P1,K] squared, idx [B,P1,K] int64, knn [B,P1,K,3] or None).

    lengths1 / lengths2 (int [B], None = full): the valid points of each cloud, clamped to [0, P1] / [0, P2].  Slots that are
    empty because of them -- rows i >= lengths1[b], and slots k >= lengths2[b] -- hold idx 0 and dists 0 (pytorch3d's
    documented padding) and, with return_nn, zero rows.  A slot inside the lengths that is empty because of a non-finite
    coordinate keeps -1 / +inf (INTEGRATION.md section 4).  Padded slots give p1 and p2 no gradient.
    pytorch3d versions differ in what they return for rows beyond lengths1 with return_nn (its knn_gather masks only
    k >= lengths2, so such rows may hold p2[b, 0] there); this shim returns zeros."""
    if norm != 2:
        raise NotImplementedError("b200pc.knn_points: only norm=2 (the reference's only use)")
    if p1.shape[-1] != 3 or p2.shape[-1] != 3:
        raise ValueError("b200pc.knn_points: points must be [B,P,3]")
    K = min(int(K), p2.shape[1])
    if K <= 0 or p1.shape[1] == 0:
        B, P1 = p1.shape[0], p1.shape[1]
        z = p1.new_zeros(B, P1, 0)
        return _KNN(z, z.long(), p1.new_zeros(B, P1, 0, 3) if return_nn else None)
    grad = torch.is_grad_enabled() and (p1.requires_grad or p2.requires_grad)
    if lengths1 is None and lengths2 is None:
        idx, dists = ops.knn_search(p2.detach(), p1.detach(), K, ops.FORM_DIRECT, want_dist=True)
        nn = None
        if return_nn or grad:
            nn = ops.gather(p2, idx)
        if grad:  # differentiable distances recomputed from the gathered neighbours
            diff = p1.unsqueeze(2) - nn
            dists = (diff * diff).sum(-1)
        return _KNN(dists, idx, nn if return_nn else None)
    return _knn_points_ragged(p1, p2, lengths1, lengths2, K, return_nn, grad)


def _knn_points_ragged(p1, p2, lengths1, lengths2, K, return_nn, grad):
    B, P1, P2 = p1.shape[0], p1.shape[1], p2.shape[1]
    dev = p1.device
    l1 = ops._lengths(lengths1, B, dev, "lengths1")
    l2 = ops._lengths(lengths2, B, dev, "lengths2")
    idx, dists = ops.knn_ragged(p2.detach(), p1.detach(), K, ops.FORM_DIRECT, l2, l1, want_dist=True)
    n1 = torch.full((B,), P1, dtype=torch.int64, device=dev) if l1 is None else l1.clamp(0, P1)
    n2 = torch.full((B,), P2, dtype=torch.int64, device=dev) if l2 is None else l2.clamp(0, P2)
    pad = (torch.arange(P1, device=dev)[None, :, None] >= n1[:, None, None]) | \
          (torch.arange(K, device=dev)[None, None, :] >= n2[:, None, None])                # [B,P1,K]
    idx = torch.where(pad, torch.zeros((), dtype=idx.dtype, device=dev), idx)
    dists = torch.where(pad, dists.new_zeros(()), dists)
    nn = None
    if return_nn or grad:
        nn = torch.where(pad[..., None], dists.new_zeros(()), ops.gather(p2, idx))
    if grad:
        # padded rows of p1 may hold anything (NaN included): they are replaced before the arithmetic, so that no NaN
        # reaches the backward pass of a masked slot
        q = torch.where((torch.arange(P1, device=dev)[None, :] >= n1[:, None])[..., None], p1.new_zeros(()), p1)
        diff = q.unsqueeze(2) - nn
        dists = torch.where(pad, dists.new_zeros(()), (diff * diff).sum(-1))
    return _KNN(dists, idx, nn if return_nn else None)


def chamfer_distance(x, y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None, weights=None,
                     batch_reduction="mean", point_reduction="mean", norm=2, **_ignored):
    """x [B,N,3], y [B,M,3] -> (loss, None).  x_lengths / y_lengths (int [B], None = full): the valid points of each cloud,
    clamped to [0, N] / [0, M].  point_reduction "mean" (each direction's sum divided by max(length, 1)) or "sum";
    batch_reduction "mean", "sum" or None (per-item losses [B]).  Weights, normals and norm=1 are not implemented.
    The defaults without lengths are the reference's only use (Utils/Utils.py:47) and run the dense op."""
    if any(v is not None for v in (x_normals, y_normals, weights)):
        raise NotImplementedError("b200pc.chamfer_distance: normals / weights are not used by the reference")
    if norm != 2:
        raise NotImplementedError("b200pc.chamfer_distance: only norm=2 is implemented")
    if point_reduction in ("max", None):
        raise NotImplementedError("b200pc.chamfer_distance: point_reduction=%r is not implemented" % (point_reduction,))
    if x_lengths is None and y_lengths is None and batch_reduction == "mean" and point_reduction == "mean":
        return ops.chamfer(x, y)[0], None
    sums = ops.chamfer_ragged(x, y, x_lengths, y_lengths)[0]
    B, N, M = sums.shape[0], x.shape[1], y.shape[1]
    xl = ops._lengths(x_lengths, B, sums.device, "x_lengths")
    yl = ops._lengths(y_lengths, B, sums.device, "y_lengths")
    # against an EMPTY other cloud every nearest-neighbour slot is empty because of the lengths: pytorch3d's knn pads it with
    # distance 0, where the op has +inf
    if xl is not None or yl is not None:
        nx = torch.full_like(sums[:, 0], float(N)) if xl is None else xl.clamp(0, N).to(sums.dtype)
        ny = torch.full_like(sums[:, 0], float(M)) if yl is None else yl.clamp(0, M).to(sums.dtype)
        sums = torch.stack([torch.where(ny == 0, sums.new_zeros(()), sums[:, 0]),
                            torch.where(nx == 0, sums.new_zeros(()), sums[:, 1])], 1)
    return ops.chamfer_reduce(sums, xl, yl, N, M, point_reduction, batch_reduction), None
