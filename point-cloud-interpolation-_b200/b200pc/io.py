"""Data-loader side of the hot path (SURVEY 8f rank 3): raw LiDAR sweeps -> fixed-size clouds by farthest point sampling
ON THE DEVICE.

The reference's loaders read a sweep with `np.fromfile(fn, np.float32).reshape(-1, 5)` (nuScenes: x y z intensity ring;
Dataset/InterpolationData.py:141-147, PolyPCI/Dataset/Dataset.py:165-172) or `.reshape([-1, 4])` (KITTI,
PointINet20230424/data/interpolation_data.py:34) and down-sample every frame to `npoints` with open3d's
`farthest_point_down_sample` on the host -- 2*field+3 frames per training sample, ~34 700 -> 16 000 points each, the input
pipeline's bottleneck.  Here the sweep is uploaded once and the a3 kernel (one thread-block cluster per cloud, up to
262 144 points: a full HDL-64 sweep of 133 312 returns, or a 128-beam x 2 048-column one) picks the samples; a batch of sweeps runs as one launch, one cluster per sweep.

Arithmetic: the kernel computes what the reference's own `farthest_point_sample` computes (fp32,
(dx*dx + dy*dy) + dz*dz, first arg-max) -- bit-exact against the strict CPU checker used by the tests.  open3d's implementation starts at point 0
and works in float64 on points converted to double; open3d is neither vendored nor pinned by the reference, so the
"open3d" variant here (start index 0, fp32 arithmetic) is PARITY UNPINNED: same algorithm, picks may differ where two
candidates tie to within fp32 rounding.
"""
import numpy as np
import torch

from . import ops


def read_bin(path, columns=None):
    """a raw little-endian float32 sweep -> [N, columns]; columns: 5 (nuScenes), 4 (KITTI) or None = infer
    (5 if the file length allows it and not 4, else 4)."""
    raw = np.fromfile(path, dtype=np.float32)
    if columns is None:
        columns = 5 if (raw.size % 5 == 0 and raw.size % 4 != 0) else 4 if raw.size % 4 == 0 else 5
    if raw.size % columns:
        raise ValueError("%s: %d floats do not form rows of %d columns" % (path, raw.size, columns))
    return raw.reshape(-1, columns)


def _upload(clouds, device):
    """list of [Ni,3] float32 arrays -> ([B,Nmax,3] device tensor, [B] point counts).  Short clouds are padded with copies of
    their point 0: a duplicate of the start point has min-distance 0 and a higher index than the original, so the
    first-arg-max rule never picks it before every real point is taken."""
    n = [int(c.shape[0]) for c in clouds]
    nmax = max(n)
    host = torch.empty(len(clouds), nmax, 3, dtype=torch.float32).pin_memory() if torch.cuda.is_available() else torch.empty(len(clouds), nmax, 3)
    for i, c in enumerate(clouds):
        t = torch.from_numpy(np.ascontiguousarray(c[:, :3], dtype=np.float32))
        host[i, :n[i]] = t
        if n[i] < nmax:
            host[i, n[i]:] = t[0]
    return host.to(device, non_blocking=True), n


def sample_clouds(clouds, npoints, device="cuda", start="open3d", return_index=False):
    """Farthest point sampling of a batch of sweeps in ONE launch.  clouds: list of [Ni,>=3] float32 arrays (xyz first).
    start: "open3d" (index 0, like open3d's farthest_point_down_sample -- parity unpinned, see the module docstring),
    "reference" (torch.randint on the CPU generator, like Utils/Pointnet2Utils.py:76) or a list of B start indices.
    -> [B,npoints,3] device tensor (, [B,npoints] int64 indices).  npoints may not exceed the smallest sweep."""
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("b200pc.io: sampling runs on the device; there is no CPU path")
    xyz, n = _upload(clouds, device)
    if npoints > min(n):
        raise ValueError("npoints=%d exceeds the smallest sweep (%d points)" % (npoints, min(n)))
    B = len(clouds)
    if isinstance(start, str):
        if start == "open3d":
            first = torch.zeros(B, dtype=torch.long)
        elif start == "reference":
            first = torch.stack([torch.randint(0, ni, (1,), dtype=torch.long)[0] for ni in n])
        else:
            raise ValueError("start must be 'open3d', 'reference' or a list of indices")
    else:
        first = torch.as_tensor(list(start), dtype=torch.long)
    idx, pts = ops.fps(xyz, int(npoints), first.to(device, non_blocking=True), want_xyz=True)
    return (pts, idx) if return_index else pts


def load_and_sample(path, npoints, columns=5, device="cuda", start="open3d", return_index=False):
    """`NuscenesDataset.get_lidar` (Dataset/InterpolationData.py:141-147) with the down-sampling on the device:
    read the sweep, keep xyz, FPS to `npoints` -> [npoints,3] device tensor (the reference returns the same rows as a
    numpy array and transposes them afterwards)."""
    scan = read_bin(path, columns)
    out = sample_clouds([scan], npoints, device=device, start=start, return_index=return_index)
    return (out[0][0], out[1][0]) if return_index else out[0]


def load_and_sample_many(paths, npoints, columns=5, device="cuda", start="open3d", return_index=False):
    """all frames of a training sample (2*field+3 sweeps, Dataset/InterpolationData.py:148-176) in one FPS launch."""
    return sample_clouds([read_bin(p, columns) for p in paths], npoints, device=device, start=start, return_index=return_index)
