"""Activation -> semantic-class labelling on the device, with the reference's segmenter surface.

Mirrors the GPU part of
  scf/segmentation/gan_local_edit/factor_catalog.py:47-75         FactorCatalog.predict
  scf/segmentation/base_dataset_segmenter.py:15-50                BaseDatasetSegmenter
  scf/segmentation/base_cluster_based_dataset_segmenter.py:18-146 BaseClusterBasedDatasetSegmenter
  scf/segmentation/black_white_handwritten_printed_text_segmenter.py:11-40
`PredictedClusters` keeps the reference's shape: {layer_str: {class_name: bool Tensor[B, S, S]}}.
The reference's per-layer chain (device->host copy, [N,k,C] temporary, argmin, host->device copy, k compare
kernels per class, uint8 nearest interpolate) is one `sis_label_assign` launch per layer here.
The CPU contour post-processing that follows in the reference (`create_segmentation_image`) is a SURVEY §8f
"next" row and is not part of this package yet.
"""
import json
import pickle
from collections import defaultdict
from pathlib import Path
from typing import Dict, List, Optional, Set

import numpy
import torch

from . import _lib

PredictedClusters = Dict[str, Dict[str, torch.Tensor]]


class FactorCatalog:
    """Inference half of the reference's FactorCatalog: k centroids [k, C] and `predict`."""

    def __init__(self, k: int, centroids=None):
        self.k = k
        self.cluster_centers = None
        self._centroids_host = None
        self.annotations = {}
        if centroids is not None:
            self.set_centroids(centroids)

    def set_centroids(self, centroids):
        c = torch.as_tensor(numpy.asarray(centroids.detach().cpu() if isinstance(centroids, torch.Tensor) else centroids),
                            dtype=torch.float32).contiguous()
        if c.dim() != 2:
            raise ValueError('centroids must be [k, C]')
        self._centroids_host = c
        self.k = c.shape[0]
        self.cluster_centers = None

    def centroids_on(self, device) -> torch.Tensor:
        if self._centroids_host is None:
            raise RuntimeError('FactorCatalog has no centroids')
        if self.cluster_centers is None or self.cluster_centers.device != torch.device(device):
            self.cluster_centers = self._centroids_host.to(device)
        return self.cluster_centers

    def predict(self, X: torch.Tensor) -> torch.Tensor:
        """[B, C, H, W] fp32 CUDA -> int64 [B, H, W] cluster ids (ties -> lowest id), all on the device."""
        ids, _ = label_assign(X, self.centroids_on(X.device), want_ids_i64=True)
        return ids

    def __repr__(self):
        return f'FactorCatalog(k={self.k})'


def label_assign(act: torch.Tensor, centroids: torch.Tensor, class_bits: Optional[torch.Tensor] = None, n_class: int = 0,
                 image_size: int = 0, mode: int = 0, want_ids_i64: bool = False, want_ids_u8: bool = False,
                 want_margin: bool = False, hist: Optional[torch.Tensor] = None):
    """One `sis_label_assign` launch.  Returns (ids or None, dict(masks=uint8 [n_class,B,S,S], margin=..., ids_u8=...))."""
    _lib.require_cuda(act, 'activations')
    _lib.require_cuda(centroids, 'centroids')
    if act.dim() != 4:
        raise RuntimeError('activations must be [B, C, H, W]')
    x = act.contiguous().float()
    c = centroids.contiguous().float()
    b, ch, h, w = x.shape
    if c.shape[1] != ch:
        raise RuntimeError(f'centroids have {c.shape[1]} channels, activations {ch}')
    dev = x.device
    out_hw = (image_size, image_size) if mode == 1 else (h, w)
    want_masks = class_bits is not None and n_class > 0
    need_u8 = want_ids_u8 or (want_masks and mode == 0 and (image_size % h or image_size % w or h != w))
    ids64 = torch.empty((b,) + out_hw, dtype=torch.int64, device=dev) if want_ids_i64 else None
    ids8 = torch.empty((b,) + out_hw, dtype=torch.uint8, device=dev) if need_u8 else None
    margin = torch.empty((b,) + out_hw, dtype=torch.float32, device=dev) if want_margin else None
    masks = torch.empty((n_class, b, image_size, image_size), dtype=torch.uint8, device=dev) if want_masks else None
    if hist is not None:
        _lib.require_cuda(hist, 'hist')
        if hist.dtype != torch.int64 or hist.numel() < c.shape[0] or not hist.is_contiguous():
            raise RuntimeError('hist must be a contiguous int64 tensor with >= k entries')
    with torch.cuda.device(dev):
        _lib.check(_lib.load().sis_label_assign(
            _lib.ptr(x), b, ch, h, w, _lib.ptr(c), c.shape[0], _lib.ptr(class_bits), n_class, image_size, mode,
            _lib.ptr(ids8), _lib.ptr(ids64), _lib.ptr(masks), _lib.ptr(margin), _lib.ptr(hist),
            _lib.current_stream_ptr(dev)))
    return ids64, {'masks': masks, 'margin': margin, 'ids_u8': ids8}


class LabelJobSpec:
    """One labelling job to run INSIDE `Generator.forward` (see `sis_label_job`): the activation is labelled right after
    it is produced, and shares its single HBM read with the ToRGB of the same tensor where shapes allow."""

    def __init__(self, activation_idx: int, centroids: torch.Tensor, class_bits: Optional[torch.Tensor] = None, n_class: int = 0,
                 image_size: int = 0, masks: Optional[torch.Tensor] = None, ids_u8: Optional[torch.Tensor] = None,
                 ids_i64: Optional[torch.Tensor] = None, margin: Optional[torch.Tensor] = None, hist: Optional[torch.Tensor] = None,
                 names: Optional[List[str]] = None):
        self.activation_idx, self.centroids, self.class_bits, self.n_class = activation_idx, centroids, class_bits, n_class
        self.image_size, self.masks, self.ids_u8, self.ids_i64, self.margin, self.hist = image_size, masks, ids_u8, ids_i64, margin, hist
        self.names = names

    def fill(self, c_job):
        c_job.activation_idx = int(self.activation_idx)
        c_job.d_centroids = self.centroids.data_ptr()
        c_job.k = int(self.centroids.shape[0])
        c_job.d_cluster_class_bits = self.class_bits.data_ptr() if self.class_bits is not None else None
        c_job.n_class = int(self.n_class)
        c_job.image_size = int(self.image_size)
        for name in ('ids_u8', 'ids_i64', 'masks', 'margin', 'hist'):
            t = getattr(self, name)
            setattr(c_job, 'd_' + name, t.data_ptr() if t is not None else None)


def extract_centroids_from_pickle(path) -> Dict[str, numpy.ndarray]:
    """Read a reference catalog pickle (`catalogs/{k}.pkl`: {str(layer): FactorCatalog, 'id_to_size_map': ...},
    scf/create_semantic_segmentation.py:123-137) WITHOUT importing sklearn or the reference: every unknown class is
    replaced by a plain attribute bag, and `_factorization.cluster_centers_` is pulled out.  Only an explicit whitelist of
    constructors is resolved, so a crafted catalog cannot reach `builtins.eval` and friends (the reference's plain
    `pickle.load` can); prefer the `.npz` catalog format where you control the files."""

    class _Bag:
        def __init__(self, *a, **k):
            pass

        def __setstate__(self, state):
            if isinstance(state, dict):
                self.__dict__.update(state)
            elif isinstance(state, tuple) and len(state) == 2 and isinstance(state[1], dict):
                self.__dict__.update(state[1] or {})
                if isinstance(state[0], dict):
                    self.__dict__.update(state[0])

    # exact (module, name) pairs the container structure and numpy arrays need; everything else -- including the rest of
    # `builtins` (eval, exec, getattr, __import__ ...) -- resolves to an inert attribute bag
    allowed = {('collections', 'OrderedDict'), ('collections', 'defaultdict'), ('copyreg', '_reconstructor'), ('_codecs', 'encode'),
               ('builtins', 'object'), ('builtins', 'dict'), ('builtins', 'list'), ('builtins', 'tuple'), ('builtins', 'set'),
               ('builtins', 'frozenset'), ('builtins', 'bytearray'), ('builtins', 'complex'), ('builtins', 'slice'),
               ('numpy', 'ndarray'), ('numpy', 'dtype'), ('numpy.core.multiarray', '_reconstruct'), ('numpy.core.multiarray', 'scalar'),
               ('numpy._core.multiarray', '_reconstruct'), ('numpy._core.multiarray', 'scalar'),
               ('numpy.core.numeric', '_frombuffer'), ('numpy._core.numeric', '_frombuffer'),
               ('numpy.random._pickle', '__randomstate_ctor'), ('numpy.random._pickle', '__bit_generator_ctor'),
               ('numpy.random._pickle', '__generator_ctor')}

    class _Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            if (module, name) in allowed:
                return super().find_class(module, name)
            return type(name, (_Bag,), {})

    with open(path, 'rb') as f:
        obj = _Unpickler(f).load()
    out = {}
    for key, val in obj.items():
        fact = getattr(val, '_factorization', None)
        centers = getattr(fact, 'cluster_centers_', None) if fact is not None else None
        if centers is not None:
            out[str(key)] = numpy.asarray(centers, dtype=numpy.float32)
    return out


def load_catalog_file(path) -> Dict[str, FactorCatalog]:
    """`.npz` ({layer: float32 [k, C]}) or a reference `.pkl`."""
    path = Path(path)
    if path.suffix == '.npz':
        with numpy.load(path) as z:
            cents = {k: z[k] for k in z.files}
    else:
        cents = extract_centroids_from_pickle(path)
    return {k: FactorCatalog(v.shape[0], v) for k, v in cents.items()}


class BaseDatasetSegmenter:
    """scf/segmentation/base_dataset_segmenter.py:15-50 (device part)."""

    def __init__(self, base_dir, image_size: int, class_to_color_map: Dict):
        self.base_dir = Path(base_dir) if base_dir is not None else None
        self.image_size = image_size
        self.debug = False
        self.debug_images = {}
        self.class_to_color_map = self.load_class_to_color_map(class_to_color_map)
        self.class_id_map = self.build_class_id_map(self.class_to_color_map)

    @staticmethod
    def load_class_to_color_map(class_to_color_map: dict) -> dict:
        def rgb(color):
            if isinstance(color, str) and color.startswith('#') and len(color) == 7:
                return tuple(int(color[i:i + 2], 16) for i in (1, 3, 5))
            from PIL import ImageColor
            return ImageColor.getrgb(color)
        return {name: rgb(color) for name, color in class_to_color_map.items()}

    @staticmethod
    def build_class_id_map(class_to_color_map: dict) -> dict:
        return {name: i for i, name in enumerate(class_to_color_map)}

    def resize_to_image_size(self, tensors: PredictedClusters) -> PredictedClusters:
        """Nearest resize of every class mask to image_size (base_dataset_segmenter.py:32-42)."""
        lib = _lib.load()
        resized = {}
        for key, class_tensors in tensors.items():
            out = {}
            for class_name, t in class_tensors.items():
                if t.shape[-1] < self.image_size:
                    _lib.require_cuda(t, 'mask')
                    src = t.contiguous().view(torch.uint8) if t.dtype == torch.bool else t.contiguous().to(torch.uint8)
                    dst = torch.empty(t.shape[0], self.image_size, self.image_size, dtype=torch.uint8, device=t.device)
                    with torch.cuda.device(t.device):
                        _lib.check(lib.sis_nearest_resize_u8(_lib.ptr(src), t.shape[0], t.shape[-2], t.shape[-1],
                                                             self.image_size, self.image_size, _lib.ptr(dst),
                                                             _lib.current_stream_ptr(t.device)))
                    t = dst.view(torch.bool) if t.dtype == torch.bool else dst.to(t.dtype)
                out[class_name] = t
            resized[key] = out
        return resized

    @staticmethod
    def dilate_image(image, kernel=None, kernel_size: int = 3):
        from . import contours
        return contours.dilate_image(image, kernel, kernel_size)

    def create_segmentation_image(self, activations):
        raise NotImplementedError


class ClusterSegmenter(BaseDatasetSegmenter):
    """BaseClusterBasedDatasetSegmenter + BlackWhiteHandwrittenPrintedTextDatasetSegmenter, device part
    (base_cluster_based_dataset_segmenter.py:18-146, black_white_handwritten_printed_text_segmenter.py:11-40)."""

    def __init__(self, base_dir, image_size: int, class_to_color_map: Dict, keys_for_class_determination: List[str],
                 keys_for_finegrained_segmentation: List[str], num_clusters: int, min_class_contour_area: int = 0,
                 only_keep_overlapping: bool = True, keys_to_merge: Optional[Dict[str, List[str]]] = None,
                 catalog: Optional[Dict[str, FactorCatalog]] = None, class_label_map: Optional[Dict] = None):
        super().__init__(base_dir, image_size, class_to_color_map)
        self.keys_for_class_determination = list(keys_for_class_determination)
        self.keys_for_finegrained_segmentation = list(keys_for_finegrained_segmentation)
        self.keys_for_generation = self.keys_for_class_determination + self.keys_for_finegrained_segmentation
        self.num_clusters = num_clusters
        self.min_class_contour_area = min_class_contour_area
        self.only_keep_overlapping = only_keep_overlapping
        self.handwriting_overlap_threshold = 0.5
        self.catalog = self.adjust_catalog(catalog) if catalog is not None else self.load_catalog()
        self.class_label_map = self.invert_class_label_map(class_label_map) if class_label_map is not None \
            else self.load_class_label_map()
        self.keys_to_merge = keys_to_merge or {}
        merged_sources = [k for ks in self.keys_to_merge.values() for k in ks]
        relevant = set(self.keys_for_generation + merged_sources)
        self.keys_for_generation = set(self.keys_for_generation + merged_sources)
        unlabelled = self.check_sanity_of_class_label_map(relevant)
        assert not unlabelled, f'Some of the activation maps were not labelled completely (map_id: cluster_id):\n{unlabelled}'
        self._bits_cache = {}
        self.cluster_pixel_counts: Dict[str, torch.Tensor] = {}

    # -- inputs on disk -------------------------------------------------------------------------------------
    def adjust_catalog(self, catalog: dict) -> dict:
        return {k: v for k, v in catalog.items() if k in self.keys_for_generation}

    def load_catalog(self) -> dict:
        base = self.base_dir / 'catalogs'
        for suffix in ('.npz', '.pkl'):
            f = base / f'{self.num_clusters}{suffix}'
            if f.exists():
                return self.adjust_catalog(load_catalog_file(f))
        raise FileNotFoundError(f'no catalog {base}/{self.num_clusters}.npz|.pkl')

    @staticmethod
    def invert_class_label_map(class_label_map: Dict[str, Dict[str, str]]) -> Dict[str, Dict[str, List[int]]]:
        """{layer: {cluster_id: class_name}} -> {layer: {class_name: [cluster ids]}} (…segmenter.py:56-67)."""
        inverted = {}
        for key, sub in class_label_map.items():
            inv = defaultdict(list)
            for sub_key, label_name in sub.items():
                inv[label_name].append(int(sub_key))
            inverted[key] = inv
        return inverted

    def load_class_label_map(self):
        with (self.base_dir / f'merged_classes_{self.num_clusters}.json').open() as f:
            return self.invert_class_label_map(json.load(f))

    def check_sanity_of_class_label_map(self, relevant_keys: Set) -> Dict:
        color_keys = list(self.class_to_color_map.keys())
        unlabelled = {}
        for key in relevant_keys:
            for class_label in self.class_label_map[key]:
                if class_label not in color_keys:
                    unlabelled.setdefault(key, []).append(class_label)
        return unlabelled

    # -- device path ------------------------------------------------------------------------------------------
    def _class_bits(self, layer_id: str, class_label_map, device):
        """uint32 [k]: bit j set <=> cluster belongs to the j-th class of class_label_map[layer_id]."""
        names = list(class_label_map[layer_id].keys())
        key = (layer_id, tuple((n, tuple(class_label_map[layer_id][n])) for n in names), str(device))
        if key not in self._bits_cache:
            k = self.catalog[layer_id].k
            bits = numpy.zeros(k, dtype=numpy.uint32)
            if len(names) > 32:
                raise RuntimeError('at most 32 classes per layer')
            for j, n in enumerate(names):
                for cid in class_label_map[layer_id][n]:
                    if 0 <= cid < k:
                        bits[cid] |= numpy.uint32(1 << j)
            self._bits_cache[key] = (names, torch.from_numpy(bits.view(numpy.int32)).to(device))
        return self._bits_cache[key]

    def _label_layer(self, layer_id, act, class_label_map, image_size, ids_out=None):
        cat = self.catalog[layer_id]
        names, bits = self._class_bits(layer_id, class_label_map, act.device)
        hist = self.cluster_pixel_counts.get(layer_id)
        if hist is None or hist.device != act.device:
            hist = torch.zeros(cat.k, dtype=torch.int64, device=act.device)
            self.cluster_pixel_counts[layer_id] = hist
        _, out = label_assign(act, cat.centroids_on(act.device), class_bits=bits, n_class=len(names),
                              image_size=image_size, want_ids_u8=ids_out is not None, hist=hist)
        if ids_out is not None:
            ids_out[layer_id] = out['ids_u8']
        return names, out['masks']

    def label_layers_stacked(self, activations, class_label_map=None, native: bool = False, ids_out: Optional[Dict] = None):
        """{layer: (class names, uint8 [n_class, B, S, S])}: the kernel's own output layout, one tensor per layer
        (what `LabelledPairGenerator.iter_host` copies to pinned memory in one transfer).  `ids_out` (a dict) receives
        the uint8 [B, H, H] cluster-id map of every layer."""
        class_label_map = class_label_map if class_label_map is not None else self.class_label_map
        acts = {str(k): v for k, v in activations.items()}
        out = {}
        for layer_id in self.catalog:
            a = acts[layer_id]
            size = a.shape[-1] if (native or a.shape[-1] >= self.image_size) else self.image_size
            out[layer_id] = self._label_layer(layer_id, a, class_label_map, size, ids_out)
        return out

    def make_label_jobs(self, generator, batch: int, class_label_map=None, want_margin: bool = False) -> List[LabelJobSpec]:
        """Jobs for `Generator.forward(..., label_jobs=...)`: one per catalog layer; every job writes the cluster-id map at
        the layer's native resolution (uint8 [B, H, H]: SURVEY.md §8(d) counts it as part of a labelled pair) and the class
        masks at image size; `want_margin` adds the fp32 nearest-centroid margin d2 - d1 (parity checks).
        Read the results with `jobs_to_stacked(jobs)` / `jobs_to_ids(jobs)` / `_as_predicted(...)` after the forward."""
        class_label_map = class_label_map if class_label_map is not None else self.class_label_map
        device = generator.input.input.device
        jobs = []
        for layer_id in self.catalog:
            cat = self.catalog[layer_id]
            c, res = generator.activation_shape(int(layer_id))
            names, bits = self._class_bits(layer_id, class_label_map, device)
            size = self.image_size if res < self.image_size else res
            hist = self.cluster_pixel_counts.get(layer_id)
            if hist is None or hist.device != device:
                hist = torch.zeros(cat.k, dtype=torch.int64, device=device)
                self.cluster_pixel_counts[layer_id] = hist
            masks = torch.empty((len(names), batch, size, size), dtype=torch.uint8, device=device)
            ids8 = torch.empty((batch, res, res), dtype=torch.uint8, device=device)
            margin = torch.empty((batch, res, res), dtype=torch.float32, device=device) if want_margin else None
            jobs.append(LabelJobSpec(int(layer_id), cat.centroids_on(device), bits, len(names), size, masks=masks, ids_u8=ids8,
                                     margin=margin, hist=hist, names=names))
        return jobs

    @staticmethod
    def jobs_to_ids(jobs: List[LabelJobSpec]) -> Dict[str, torch.Tensor]:
        """{layer: uint8 [B, H, H] cluster ids at the layer's native resolution}."""
        return {str(j.activation_idx): j.ids_u8 for j in jobs}

    @staticmethod
    def jobs_to_stacked(jobs: List[LabelJobSpec]):
        return {str(j.activation_idx): (j.names, j.masks) for j in jobs}

    @staticmethod
    def _as_predicted(stacked) -> PredictedClusters:
        return {layer: {n: masks.view(torch.bool)[j] for j, n in enumerate(names)} for layer, (names, masks) in stacked.items()}

    def predict_clusters(self, activations: Dict[int, torch.Tensor], class_label_map) -> PredictedClusters:
        """Per layer: cluster ids -> per-class bool masks at the layer's native resolution (…segmenter.py:119-138)."""
        return self._as_predicted(self.label_layers_stacked(activations, class_label_map, native=True))

    def prepare_image_segmentation(self, activations, class_label_map=None) -> PredictedClusters:
        """predict_clusters + resize_to_image_size fused: one launch per layer writes the S x S masks directly."""
        return self._as_predicted(self.label_layers_stacked(activations, class_label_map))

    @staticmethod
    def _or_masks(masks: List[torch.Tensor]) -> torch.Tensor:
        """A new tensor: the byte-wise OR of same-shape uint8 / bool device masks (`sis_or_u8`)."""
        acc = masks[0].contiguous().clone()
        lib = _lib.load()
        for m in masks[1:]:
            m = m.contiguous()
            with torch.cuda.device(acc.device):
                _lib.check(lib.sis_or_u8(_lib.ptr(acc), _lib.ptr(m), acc.numel(), _lib.current_stream_ptr(acc.device)))
        return acc

    def merge_sub_images(self, predicted_clusters: PredictedClusters) -> PredictedClusters:
        """OR the class masks of several layers into a destination key (black_white…segmenter.py:31-40)."""
        for dst_key, keys in self.keys_to_merge.items():
            predicted_clusters[dst_key] = {class_name: self._or_masks([predicted_clusters[k][class_name] for k in keys])
                                           for class_name in self.class_to_color_map}
        return predicted_clusters

    def merge_stacked(self, stacked):
        """`merge_sub_images` on the kernel's stacked layout: adds {dst_key: (class names, uint8 [n_class, B, S, S])} for
        every `keys_to_merge` entry (class planes in `class_to_color_map` order, OR over the source layers)."""
        names = list(self.class_to_color_map)
        for dst_key, keys in self.keys_to_merge.items():
            per_class = [dict(zip(*stacked[k])) for k in keys]        # {class name: uint8 [B, S, S] plane} per source layer
            stacked[dst_key] = (names, torch.stack([self._or_masks([p[class_name] for p in per_class]) for class_name in names]))
        return stacked

    # -- host-side contour stage (contours.py; base_cluster_based…:148-450, black_white…:42-99) ------------------
    def contour_config(self):
        from . import contours
        return contours.ContourConfig(self.image_size, self.class_to_color_map, self.keys_for_class_determination,
                                      self.keys_for_finegrained_segmentation, self.only_keep_overlapping,
                                      self.min_class_contour_area)

    def cluster_image_to_contours(self, cluster_arrays):
        from . import contours
        return contours.cluster_image_to_contours(cluster_arrays)

    def contour_overlap(self, contour1, contour2) -> int:
        from . import contours
        return contours.contour_overlap(contour1, contour2)

    def merge_two_contours_if_overlapping(self, contour1, contour2):
        from . import contours
        return contours.merge_two_contours_if_overlapping(contour1, contour2)

    def merge_contours(self, contours_, only_keep_overlapping: bool = False):
        from . import contours
        return contours.merge_contours(contours_, only_keep_overlapping)

    def merge_contours_of_same_class_from_different_images(self, class_contours_for_sub_images, batch_size: int,
                                                           only_keep_overlapping: bool = False, class_names_to_merge=(),
                                                           drop_if_size_of_contours_zero: bool = False):
        from . import contours
        return contours.merge_contours_of_same_class_from_different_images(
            class_contours_for_sub_images, batch_size, only_keep_overlapping, class_names_to_merge, drop_if_size_of_contours_zero)

    def merge_contours_of_same_class_from_same_image(self, class_contours):
        from . import contours
        return contours.merge_contours_of_same_class_from_same_image(class_contours)

    def extract_contours(self, predicted_clusters: PredictedClusters, image_ids_to_extract: List[str]):
        from . import contours
        return contours.extract_contours(predicted_clusters, image_ids_to_extract)

    def extract_text_regions(self, predicted_clusters: PredictedClusters, batch_size: int):
        """black_white…:42-59."""
        merged = self.merge_contours_of_same_class_from_different_images(
            self.extract_contours(predicted_clusters, self.keys_for_class_determination), batch_size,
            only_keep_overlapping=self.only_keep_overlapping, drop_if_size_of_contours_zero=True)
        return self.drop_too_small_contours(merged)

    def merge_finegrained_segmentation(self, predicted_clusters: PredictedClusters, batch_size: int):
        """base_cluster_based…:334-349."""
        return self.merge_contours_of_same_class_from_different_images(
            self.extract_contours(predicted_clusters, self.keys_for_finegrained_segmentation), batch_size,
            only_keep_overlapping=True, drop_if_size_of_contours_zero=True)

    def classify_fine_grained_contours(self, text_regions_per_class, fine_grained_contours_per_class,
                                       fine_grained_class_name: str = 'printed_text'):
        from . import contours
        return contours.classify_fine_grained_contours(text_regions_per_class, fine_grained_contours_per_class,
                                                       self.class_id_map, fine_grained_class_name)

    def drop_too_small_contours(self, class_contours):
        from . import contours
        return contours.drop_too_small_contours(class_contours, self.min_class_contour_area)

    def determine_images_to_drop(self, fine_grained_contours_per_image) -> List[int]:
        from . import contours
        return contours.determine_images_to_drop(fine_grained_contours_per_image, self.image_size)

    def render_segmentation_image(self, fine_grained_prediction, classified_contours, batch_size: int,
                                  cluster_class_name: str = 'printed_text'):
        from . import contours
        return contours.render_segmentation_image(fine_grained_prediction, classified_contours, batch_size, self.image_size,
                                                  self.class_to_color_map, cluster_class_name)

    def segment_predicted_clusters(self, predicted_clusters: PredictedClusters, batch_size: int, pool=None):
        """The host half of create_segmentation_image on masks that are already merged and resized (device tensors or
        host arrays); `pool` = a concurrent.futures executor to fan the images out over."""
        from . import contours
        return contours.segment_masks_parallel(predicted_clusters, batch_size, self.contour_config(), pool)

    def create_segmentation_image(self, activations: Dict[int, torch.Tensor], pool=None):
        """black_white…:77-99: (uint8 [B,S,S,3] colour label images, ids of images to drop).  The batch size is read
        from the constant-input capture `activations[0]`, as the reference does (:79)."""
        predicted_clusters = self.merge_sub_images(self.prepare_image_segmentation(activations, self.class_label_map))
        return self.segment_predicted_clusters(predicted_clusters, len(activations[0]), pool)


def make_image(images: torch.Tensor) -> torch.Tensor:
    """`pytorch_training.images.make_image` on the device: [B,3,S,S] fp32 -> uint8 [B,S,S,3]
    (clamp(-1,1), (x+1)/2*255, truncation).  The caller moves it to the host (`.cpu().numpy()`) when needed."""
    _lib.require_cuda(images, 'images')
    squeeze = images.dim() == 3
    x = (images[None] if squeeze else images).contiguous().float()
    out = torch.empty(x.shape[0], x.shape[2], x.shape[3], 3, dtype=torch.uint8, device=x.device)
    if x.shape[2] != x.shape[3] or x.shape[1] != 3:
        raise RuntimeError('make_image expects [B, 3, S, S]')
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().sis_make_image_u8(_lib.ptr(x), x.shape[0], x.shape[2], _lib.ptr(out),
                                                 _lib.current_stream_ptr(x.device)))
    return out[0] if squeeze else out
