"""Spherical mini-batch k-means, step by step: the test reference of `sis_kmeans_steps` (csrc/kmeans.cu).

The host loop of MiniBatchSphericalKMeans.fit (scf/segmentation/gan_local_edit/spherical_kmeans.py:159-312, i.e. sklearn
0.24.2's MiniBatchKMeans._mini_batch_step on unit rows with the centres renormalised after every step), restated in torch
so it runs on any device and dtype (fp64 in the tests), with the library's counter-based draws instead of numpy's
RandomState:
  h(t, j, s) = splitmix64(splitmix64(splitmix64(seed) ^ t) ^ (j << 1 | s))
  batch row j of step t = h(t, j, 0) mod n; rows that replace starved centres = the n_re smallest h(t, j, 1).
The starvation test `count < ratio * max count` is evaluated in fp32 whatever the working dtype, as the library does:
counts are integers, so that test is exact in both, and a fp64 threshold could fall on the other side of a count.
"""
from typing import Callable, Optional

import numpy
import torch

_M64 = (1 << 64) - 1


def splitmix64(x: numpy.ndarray) -> numpy.ndarray:
    x = numpy.asarray(x, dtype=numpy.uint64)
    with numpy.errstate(over='ignore'):
        x = x + numpy.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> numpy.uint64(30))) * numpy.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> numpy.uint64(27))) * numpy.uint64(0x94D049BB133111EB)
    return x ^ (x >> numpy.uint64(31))


def draw(seed: int, t: int, n_rows: int, stream: int) -> numpy.ndarray:
    """h(t, j, stream) for j = 0 .. n_rows-1, uint64."""
    h = splitmix64(splitmix64(numpy.uint64(seed & _M64)) ^ numpy.uint64(t))
    j = numpy.arange(n_rows, dtype=numpy.uint64)
    return splitmix64(h ^ ((j << numpy.uint64(1)) | numpy.uint64(stream)))


def batch_rows(seed: int, t: int, batch_size: int, n: int) -> torch.Tensor:
    return torch.from_numpy((draw(seed, t, batch_size, 0) % numpy.uint64(n)).astype(numpy.int64))


def normalize_rows(x: torch.Tensor) -> torch.Tensor:
    return x / x.norm(dim=1, keepdim=True).clamp_min(1e-12)


def assign(xb: torch.Tensor, centers: torch.Tensor):
    """(labels, squared distances) of the rows of `xb` to their nearest centre, ties to the lower index."""
    d = ((xb[:, None, :] - centers[None, :, :]) ** 2).sum(2)
    dist, labels = d.min(1)
    return labels, dist


def step(xb: torch.Tensor, centers: torch.Tensor, counts: torch.Tensor, reassign: bool, ratio: float,
         keys: Optional[numpy.ndarray]):
    """`_mini_batch_step` (dense), centres and counts modified in place; returns (labels, squared distances)."""
    labels, dist = assign(xb, centers)
    k, bs = centers.shape[0], xb.shape[0]
    if reassign and ratio > 0:
        c32 = counts.float()
        starved = c32 < torch.tensor(ratio, dtype=torch.float32) * c32.max()
        if int(starved.sum()) > 0.5 * bs:
            keep = torch.argsort(counts, stable=True)[int(0.5 * bs):]
            starved[keep] = False
        n_re = int(starved.sum())
        if n_re:
            order = numpy.lexsort((numpy.arange(bs), keys))          # ascending key, ties to the lower row
            pick = torch.from_numpy(order[:n_re].astype(numpy.int64)).to(xb.device)
            centers[starved] = xb[pick]
            counts[starved] = counts[~starved].min() if bool((~starved).any()) else 0
    sums = torch.zeros_like(centers).index_add_(0, labels, xb)
    n_in = torch.bincount(labels, minlength=k).to(centers.dtype)
    hit = n_in > 0
    centers[hit] = centers[hit] * counts[hit, None] + sums[hit]
    counts += n_in
    centers[hit] = centers[hit] / counts[hit, None]
    return labels, dist


def explicit_step(x: torch.Tensor, centers: torch.Tensor, counts: torch.Tensor, idx: torch.Tensor):
    """The validation step of an n_init trial: one step on the rows `idx`, no reassignment; returns the new centres."""
    centers = normalize_rows(centers)
    step(x[idx], centers, counts, False, 0.0, None)
    return normalize_rows(centers)


def fit_steps(x: torch.Tensor, centers: torch.Tensor, counts: torch.Tensor, seed: int, batch_size: int, max_steps: int,
              max_no_improvement: Optional[int], ratio: float, batch_inertia: Optional[Callable[[int, float], float]] = None,
              on_step: Optional[Callable] = None):
    """The step loop of `fit` from the given centres and counts.  Returns (centres, counts, n_iter).
    `batch_inertia(t, own)` may replace the step's batch inertia (the tests replay the device's values so that the
    early-stopping decision, which compares EWAs, sees the same numbers); `on_step(t, idx, labels, centers, counts)` is
    called after every step."""
    n = x.shape[0]
    alpha = min(1.0, batch_size * 2.0 / (n + 1))
    ewa = ewa_min = None
    no_improvement = 0
    t = 0
    for t in range(max_steps):
        idx = batch_rows(seed, t, batch_size, n).to(x.device)
        centers = normalize_rows(centers)
        reassign = (t + 1) % (10 + int(counts.min())) == 0
        keys = draw(seed, t, batch_size, 1) if reassign else None
        labels, dist = step(x[idx], centers, counts, reassign, ratio, keys)
        centers = normalize_rows(centers)
        bi = float(numpy.float32(float(dist.sum()) / batch_size))
        if batch_inertia is not None:
            bi = batch_inertia(t, bi)
        ewa = bi if ewa is None else ewa * (1 - alpha) + bi * alpha
        if ewa_min is None or ewa < ewa_min:
            ewa_min, no_improvement = ewa, 0
        else:
            no_improvement += 1
        if on_step is not None:
            on_step(t, idx, labels, centers, counts)
        if max_no_improvement is not None and no_improvement >= max_no_improvement:
            break
    return centers, counts, t + 1
