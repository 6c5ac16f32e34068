"""Catalog creation (SURVEY.md §8(f) row 4): spherical mini-batch k-means over captured activations, on the device.

Mirrors the surface of
  scf/segmentation/gan_local_edit/spherical_kmeans.py:159-312   MiniBatchSphericalKMeans.fit
  scf/segmentation/gan_local_edit/factor_catalog.py:14-68       FactorCatalog(k).fit_predict(X, raw=True)
  scf/create_semantic_segmentation.py:114-137                   find_and_render_clusters, save_catalogs
The reference's `fit` is sklearn 0.24.2's MiniBatchKMeans loop (k-means++ init on a random subset, per-centre learning
rate 1 / count, random reassignment of starved centres, EWA-inertia early stopping) run on unit-normalised rows with the
centres re-normalised after every step.  Here every step of every fit runs in `sis_kmeans_steps` (csrc/kmeans.cu): one
launch advances all fits -- every k of every layer -- by up to KMEANS_CHUNK_STEPS steps, and the host reads the fits'
`done` words once per launch.  The k-means++ seeding stays in PyTorch (one-off, on at most `init_size` rows); each
n_init trial's validation step is one `sis_kmeans_steps` call on an explicit index list, and the final labelling of all
points is `sis_label_assign` (the hot path's labelling kernel: centres are unit vectors, so the nearest centre by squared
distance is the spherical assignment).

Draws come from the library's counter-based hash (see include/sis_b200.h), not from numpy's RandomState: the reference's
exact result is not reproduced (PARITY UNPINNED: it depends on sklearn 0.24.2 internals), and a fit's result does not
depend on which other fits share its launches.  oracle/kmeans_oracle.py restates the steps for the tests.  The `.npz`
this writes is what `labelling.load_catalog_file` reads.
"""
from pathlib import Path
from typing import Dict, Iterable, List, Optional

import numpy
import torch

from . import _lib
from .labelling import label_assign

# Steps per sis_kmeans_steps launch.  A fit stops at a step the host cannot predict (early stopping), so every launch
# is followed by one read of the `done` words.  One step of a 100-row batch is tens of microseconds per CTA, so 32
# steps keep that read well under a tenth of the launch while a finished fit wastes at most 31 empty steps (a done fit
# returns at once).
KMEANS_CHUNK_STEPS = 32
_DONE_WORD, _STEPS_WORD = 3, 1          # int64 words of sis_kmeans_state


def _normalize_rows(x: torch.Tensor) -> torch.Tensor:
    return x / x.norm(dim=1, keepdim=True).clamp_min(1e-12)


def _channel_major(x: torch.Tensor) -> torch.Tensor:
    """Rows [n, C] -> [1, C, n', 1] as the labelling kernel reads NCHW, n' = n padded to a multiple of 4 by repeating
    the first rows (their labels are dropped)."""
    xt = x.t()
    pad = (-x.shape[0]) % 4
    if pad:
        xt = torch.cat([xt, xt[:, :pad]], dim=1)
    return xt.contiguous().reshape(1, x.shape[1], -1, 1)


def _labels(x_cm: torch.Tensor, n: int, centers: torch.Tensor) -> torch.Tensor:
    ids, _ = label_assign(x_cm, centers, want_ids_i64=True, want_margin=False)
    return ids.reshape(-1)[:n]


def _sq_dist(x: torch.Tensor, centers: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """Squared distance of each row of `x` to centre `labels[i]`."""
    d = (x * x).sum(1) - 2.0 * (x * centers[labels]).sum(1) + (centers * centers).sum(1)[labels]
    return d.clamp_min(0)


def _kmeans_pp(x: torch.Tensor, k: int, gen: torch.Generator) -> torch.Tensor:
    """k-means++ seeding on the rows of `x` (unit vectors): D^2 sampling with the usual 2 + log k local trials."""
    n = x.shape[0]
    trials = 2 + int(numpy.log(k))
    first = int(torch.randint(n, (1,), generator=gen, device=x.device))
    centers = [x[first]]
    closest = ((x - centers[0]) ** 2).sum(1)
    for _ in range(1, k):
        cand = torch.multinomial(closest.clamp_min(1e-30), trials, replacement=True, generator=gen)
        d_cand = ((x[None, :, :] - x[cand][:, None, :]) ** 2).sum(2)          # [trials, n]
        pot = torch.minimum(closest[None], d_cand).sum(1)
        best = int(pot.argmin())
        centers.append(x[cand[best]])
        closest = torch.minimum(closest, d_cand[best])
    return torch.stack(centers)


class KMeansFit:
    """Device buffers of one fit of `sis_kmeans_steps`: unit rows `points` [n, C], `centers` [k, C] and `counts` [k]
    (both updated in place) and the fit's state (int64 words of `sis_kmeans_state`, or None for explicit steps only)."""

    def __init__(self, points: torch.Tensor, centers: torch.Tensor, counts: Optional[torch.Tensor] = None,
                 state: Optional[torch.Tensor] = None):
        self.points, self.centers = points, centers
        self.counts = torch.zeros(centers.shape[0], device=centers.device) if counts is None else counts
        self.state = state

    def descriptor(self) -> _lib.KmeansFit:
        for t in (self.points, self.centers, self.counts):
            _lib.require_cuda(t, 'k-means buffer')
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise RuntimeError('k-means points, centers and counts must be contiguous float32 tensors')
        return _lib.KmeansFit(self.points.data_ptr(), self.points.shape[0], self.points.shape[1], self.centers.shape[0],
                              self.centers.data_ptr(), self.counts.data_ptr(),
                              self.state.data_ptr() if self.state is not None else None)

    @property
    def done(self) -> bool:
        return bool(self.state[_DONE_WORD])

    @property
    def steps_done(self) -> int:
        return int(self.state[_STEPS_WORD])


def new_states(n_fits: int, device) -> torch.Tensor:
    """Uninitialised states of `n_fits` fits, [n_fits, words] int64; row i is fit i's state."""
    words = _lib.load().sis_kmeans_state_bytes() // 8
    return torch.empty(n_fits, words, dtype=torch.int64, device=device)


def init_state(fit: KMeansFit, seed: int, batch_size: int, max_steps: int, max_no_improvement: Optional[int],
               reassignment_ratio: float):
    with torch.cuda.device(fit.state.device):
        _lib.check(_lib.load().sis_kmeans_init_state(
            _lib.ptr(fit.state), int(seed) & ((1 << 64) - 1), int(batch_size), int(max_steps),
            -1 if max_no_improvement is None else int(max_no_improvement), float(reassignment_ratio),
            _lib.current_stream_ptr(fit.state.device)))


def kmeans_steps(fits: List[KMeansFit], steps: int, indices: Optional[torch.Tensor] = None,
                 batch_inertia: Optional[torch.Tensor] = None):
    """One `sis_kmeans_steps` launch over `fits` (all on one device): up to `steps` drawn steps each, or, with `indices`
    (int32 row indices), one step of every fit on those rows.  `batch_inertia` [len(fits), steps] fp32 receives the
    batch inertia of each step run."""
    arr = (_lib.KmeansFit * len(fits))(*[f.descriptor() for f in fits])
    dev = fits[0].centers.device
    if indices is not None:
        _lib.require_cuda(indices, 'indices')
        if indices.dtype != torch.int32 or not indices.is_contiguous():
            raise RuntimeError('indices must be a contiguous int32 tensor')
    if batch_inertia is not None:
        _lib.require_cuda(batch_inertia, 'batch_inertia')
        if batch_inertia.dtype != torch.float32 or batch_inertia.shape != (len(fits), steps) or not batch_inertia.is_contiguous():
            raise RuntimeError(f'batch_inertia must be a contiguous float32 [{len(fits)}, {steps}] tensor')
    with torch.cuda.device(dev):
        _lib.check(_lib.load().sis_kmeans_steps(arr, len(fits), int(steps), _lib.ptr(indices),
                                                0 if indices is None else indices.numel(), _lib.ptr(batch_inertia),
                                                _lib.current_stream_ptr(dev)))


class _Result:
    def __init__(self, centers, labels, init_inertia, n_iter):
        self.centers, self.labels, self.init_inertia, self.n_iter = centers, labels, init_inertia, n_iter


def _fit_all(points_by_layer: Dict, ks: Iterable[int], random_state: Optional[int] = 0, batch_size: int = 100,
             max_iter: int = 100, n_init: int = 3, init_size: Optional[int] = None, reassignment_ratio: float = 0.01,
             max_no_improvement: Optional[int] = 10, compute_labels: bool = True, stats: Optional[dict] = None,
             **_unused) -> Dict:
    """{layer: (unit rows [n, C], {k: _Result})}: every k on every layer, driven together."""
    ks = [int(k) for k in ks]
    seed = int(random_state or 0)
    layers, fits, meta = {}, [], []
    for layer, pts in points_by_layer.items():
        _lib.require_cuda(pts, f'points of layer {layer}')
        rows = pts.permute(0, 2, 3, 1).reshape(-1, pts.shape[1]) if pts.dim() == 4 else pts      # ptutils.partial_flat
        x = _normalize_rows(rows.float()).contiguous()
        n = x.shape[0]
        for k in ks:
            if n < k:
                raise ValueError(f'n_samples={n} should be >= n_clusters={k}')
        size = min(n, init_size or 3 * batch_size)
        # each fit seeds as the single fit would: its own generator, validation rows first, then one subset per trial
        gens = [torch.Generator(device=x.device) for _ in ks]
        for g in gens:
            g.manual_seed(seed)
        valid_idx = [torch.randint(n, (size,), generator=g, device=x.device) for g in gens][0]
        valid = x[valid_idx]
        trials = []                                     # [trial][k index] -> KMeansFit
        for _ in range(n_init):
            trial = [KMeansFit(x, _normalize_rows(_kmeans_pp(x[torch.randint(n, (size,), generator=g, device=x.device)], k, g)).contiguous())
                     for g, k in zip(gens, ks)]
            kmeans_steps(trial, 1, indices=valid_idx.to(torch.int32))
            trials.append(trial)
        valid_cm = _channel_major(valid)
        inertia = torch.stack([torch.stack([_sq_dist(valid, f.centers, _labels(valid_cm, size, f.centers)).sum()
                                            for f in trial]) for trial in trials]).cpu()       # [n_init, len(ks)]
        best = inertia.argmin(0).tolist()
        layers[layer] = (x, pts.shape[0:1] + pts.shape[2:] if pts.dim() == 4 else (n,))
        for i, k in enumerate(ks):
            f = trials[best[i]][i]
            fits.append(f)
            meta.append((layer, k, float(inertia[best[i], i]), n))
    states = new_states(len(fits), fits[0].centers.device)
    for f, s, (_, _, _, n) in zip(fits, states, meta):
        f.state = s
        init_state(f, seed, batch_size, max_iter * ((n + batch_size - 1) // batch_size), max_no_improvement, reassignment_ratio)
    active = list(range(len(fits)))
    launches = 0
    while active:
        kmeans_steps([fits[i] for i in active], KMEANS_CHUNK_STEPS)
        launches += 1
        done = states[active, _DONE_WORD].cpu().tolist()          # the one host synchronisation of the chunk
        active = [i for i, d in zip(active, done) if not d]
    steps = states[:, _STEPS_WORD].cpu().tolist()
    if stats is not None:
        stats.update(fits=len(fits), step_launches=launches, host_syncs=launches, steps=int(sum(steps)), max_steps=int(max(steps)))
    out = {layer: (x, {}) for layer, (x, _) in layers.items()}
    cm = {}
    for f, n_iter, (layer, k, init_inertia, n) in zip(fits, steps, meta):
        labels = None
        if compute_labels:
            x, shape = layers[layer]
            if layer not in cm:
                cm[layer] = _channel_major(x)
            labels = _labels(cm[layer], n, f.centers).reshape(shape)
        out[layer][1][k] = _Result(f.centers, labels, init_inertia, int(n_iter))
    return out


def fit_catalogs(points_by_layer: Dict, ks: Iterable[int], random_state: Optional[int] = 0, stats: Optional[dict] = None,
                 **kmeans_args) -> Dict:
    """Fit every k of `ks` on every layer in one batched run: {layer: {k: (centres float32 [k, C], labels)}}.
    Points are activation maps [N, C, H, W] (labels int64 [N, H, W] on the device) or rows [n, C] (labels [n]).
    `kmeans_args` are MiniBatchSphericalKMeans' options; `stats`, when given, receives the number of fits, step
    launches, host synchronisations of the step loop and steps run."""
    res = _fit_all(points_by_layer, ks, random_state, stats=stats, **kmeans_args)
    return {layer: {k: (r.centers.cpu().numpy(), r.labels) for k, r in by_k.items()} for layer, (_, by_k) in res.items()}


class MiniBatchSphericalKMeans:
    """sklearn-style estimator with the reference's attributes (`cluster_centers_`, `labels_`, `inertia_`, `n_iter_`)."""

    def __init__(self, n_clusters: int = 8, random_state: Optional[int] = 0, batch_size: int = 100, max_iter: int = 100, n_init: int = 3,
                 init_size: Optional[int] = None, reassignment_ratio: float = 0.01, max_no_improvement: int = 10, compute_labels: bool = True,
                 **_unused):
        self.n_clusters, self.random_state, self.batch_size, self.max_iter, self.n_init = n_clusters, random_state, batch_size, max_iter, n_init
        self.init_size, self.reassignment_ratio, self.max_no_improvement = init_size, reassignment_ratio, max_no_improvement
        self.compute_labels = compute_labels
        self.cluster_centers_ = None
        self.labels_ = None

    def fit(self, X, y=None, sample_weight=None):
        if sample_weight is not None:
            raise NotImplementedError('sample weights are not used by the catalog creation path')
        _lib.require_cuda(X, 'X')
        x, by_k = _fit_all({0: X}, [self.n_clusters], self.random_state, batch_size=self.batch_size, max_iter=self.max_iter,
                           n_init=self.n_init, init_size=self.init_size, reassignment_ratio=self.reassignment_ratio,
                           max_no_improvement=self.max_no_improvement, compute_labels=self.compute_labels)[0]
        r = by_k[self.n_clusters]
        self.init_inertia_, self.n_iter_ = r.init_inertia, r.n_iter
        self._centers_device = r.centers
        self.cluster_centers_ = r.centers.cpu().numpy()
        if self.compute_labels:
            self.labels_ = r.labels.cpu().numpy()
            self.inertia_ = float(_sq_dist(x, r.centers, r.labels).sum())
        return self

    def predict(self, X) -> numpy.ndarray:
        x = _normalize_rows(X.float().contiguous())
        return _labels(_channel_major(x), x.shape[0], self._centers_device.to(x.device)).cpu().numpy()


def find_clusters(all_activations: Dict[int, torch.Tensor], num_clusters: int, min_size: int = 0, **kmeans_args):
    """create_semantic_segmentation.py:96-137 without the rendering: ({layer: heat maps}, {str(layer): centres} plus
    'id_to_size_map').  Layers whose maps are not larger than `min_size` are skipped (`strip_activations`, :93-94).
    Every layer's fit is one FactorCatalog(k).fit_predict(X, raw=True): [N, k, H, W] one-hot heat maps."""
    kept = {key: act for key, act in all_activations.items()
            if not min_size or (act.shape[-2] > min_size and act.shape[-1] > min_size)}
    fitted = fit_catalogs(kept, [num_clusters], **kmeans_args)
    heat, catalogs, sizes = {}, {}, {}
    for key, act in kept.items():
        centers, labels = fitted[key][num_clusters]
        heat[key] = torch.nn.functional.one_hot(labels, num_clusters).permute(0, 3, 1, 2).float()
        catalogs[str(key)] = centers
        sizes[key] = f'{act.shape[-2]}x{act.shape[-1]}'
    return heat, catalogs, sizes


def save_catalogs(catalogs: Dict[str, numpy.ndarray], num_clusters: int, dest_dir) -> Path:
    """`<dest_dir>/<k>.npz` ({layer: float32 [k, C]}): the catalog format `ClusterSegmenter.load_catalog` prefers (the
    reference pickles sklearn-backed FactorCatalog objects, create_semantic_segmentation.py:131-137)."""
    dest_dir = Path(dest_dir)
    dest_dir.mkdir(parents=True, exist_ok=True)
    path = dest_dir / f'{num_clusters}.npz'
    numpy.savez(path, **{k: numpy.asarray(v, dtype=numpy.float32) for k, v in catalogs.items()})
    return path
