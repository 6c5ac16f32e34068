"""Latent / noise stream, batched generation and the seed-sharded labelled-pair pipeline.

Mirrors
  scf/latent_projecting/__init__.py:15-28      Latents
  scf/utils/dataset_creation.py:32-58          build_latent_and_noise_generator, generate_images
  scf/create_dataset_for_segmentation.py:109-148  the per-batch hot loop (GPU part)
and adds the multi-GPU partitioning of SURVEY.md §8e: one process per GPU, batch index b is owned by rank
b mod world_size, every rank replays the single reference RNG stream (CPU latents, device noise) and keeps only
its own batches, so the union over ranks equals the reference's single-process run on the same seed.  The only
collective is one all-reduce of an int64 statistics vector (NCCL on GPUs, gloo in the CPU tests).
"""
import contextlib
from dataclasses import dataclass
from typing import Dict, Iterable, Iterator, List, Optional, Tuple

import torch

from .labelling import ClusterSegmenter, make_image
from .model import Generator


@dataclass
class Latents:
    latent: torch.Tensor
    noise: List[torch.Tensor]

    def to(self, device) -> 'Latents':
        self.latent = self.latent.to(device)
        self.noise = [n.to(device) for n in self.noise]
        return self

    def __getitem__(self, key: int) -> 'Latents':
        return Latents(self.latent[key].unsqueeze(0), [n[key].unsqueeze(0) for n in self.noise])

    def detach(self):
        self.latent = self.latent.detach()
        self.noise = [n.detach() for n in self.noise]

    def numpy(self) -> 'Latents':
        return Latents(self.latent.cpu().numpy(), [n.cpu().numpy() for n in self.noise])


def _decoder_of(model):
    """The reference passes a StyleganAutoencoder whose `.decoder` is the Generator (networks/encoder/autoencoder.py);
    a bare Generator is accepted as well."""
    return getattr(model, 'decoder', model)


def build_latent_and_noise_generator(autoencoder, config: Dict, seed=1) -> Iterable[Latents]:
    """Seeded, infinite (latent, noise) stream: z = randn(B, latent_size) on the CPU generator, noise maps from
    `decoder.make_noise()` on the decoder's device; the seed is applied lazily at the first `next()`
    (utils/dataset_creation.py:32-37)."""
    decoder = _decoder_of(autoencoder)
    torch.random.manual_seed(seed)
    while True:
        latent_code = torch.randn(config['batch_size'], config['latent_size'])
        noise = decoder.make_noise()
        yield Latents(latent_code, noise)


def generate_images(batch: Latents, autoencoder, device: str = 'cuda', mean_latent: Optional[torch.Tensor] = None,
                    capture_layers=None, label_jobs=None, mix_inject_index: Optional[int] = None
                    ) -> Tuple[Dict[int, torch.Tensor], torch.Tensor]:
    """(activations, image) exactly as utils/dataset_creation.py:40-58: truncation 0.7 iff mean_latent is given.
    `capture_layers` / `label_jobs` are forwarded to the generator (extensions, see Generator.forward).
    `mix_inject_index` (extension; the reference script never passes two styles, BASELINE config 4 asks for it): style
    mixing through the generator's own two-style path (model.py:521-528) with an explicit crossover index; the second
    style of sample i is the latent of sample i-1 of the same batch (no extra draw: the stream stays the reference's)."""
    if not isinstance(batch, Latents):
        raise NotImplementedError('the encoder path (dict batches) is outside the hot path (SURVEY.md §2 row 16)')
    latents = batch.to(device)
    decoder = _decoder_of(autoencoder)
    kwargs = {}
    if capture_layers is not None:
        kwargs['capture_layers'] = capture_layers
    if label_jobs is not None:
        kwargs['label_jobs'] = label_jobs
    styles = [latents.latent]
    if mix_inject_index is not None:
        styles.append(mixing_partner(latents.latent))
        kwargs['inject_index'] = int(mix_inject_index)
    with torch.no_grad():
        image, activations = decoder(
            styles, input_is_latent=False, noise=latents.noise, return_intermediate_activations=True,
            truncation=0.7 if mean_latent is not None else 1, truncation_latent=mean_latent, **kwargs)
    return activations, image


def mixing_partner(latent: torch.Tensor) -> torch.Tensor:
    """Second style of the style-mixing extension: sample i is paired with sample i-1 of its batch."""
    return torch.roll(latent, shifts=1, dims=0)


# ------------------------------------------------------------------------------------------- sharding
def owned_batches(rank: int, world_size: int, num_batches: int) -> List[int]:
    """Batch indices owned by `rank` (round-robin; the unit is a batch because noise is drawn per batch)."""
    return list(range(rank, num_batches, world_size))


def sharded_latent_stream(generator: Generator, config: Dict, seed: int, rank: int, world_size: int,
                          replay: bool = False) -> Iterator[Tuple[int, Latents]]:
    """This rank's batches (index b = rank mod world_size) of the reference's single (latent, noise) stream.

    `replay=True` (and every CPU-device run): every rank draws every batch and yields only its own -- O(world_size) draws
    per kept batch.  Default on CUDA: the streams are addressed by POSITION instead.  CPU latents: one
    `randn(world_size * B, latent_size)` per round equals the concatenation of the reference's per-batch draws (the CPU
    normal fill works on 16-element blocks; checked by `tests/test_host_logic.py`), and the rank keeps its rows.  Device
    noise: the default CUDA generator is counter based (Philox), one `make_noise()` advances its offset by a constant
    measured on the first batch, so batch b starts at offset0 + b * delta: `set_offset` jumps there and the rank draws
    only its own maps.  Both give bit-identical batches to the replay (tests/test_pipeline_gpu.py)."""
    device = generator.input.input.device
    B, L = config['batch_size'], config['latent_size']
    positional = (not replay) and world_size > 1 and device.type == 'cuda' and (B * L) % 16 == 0
    if not positional:
        stream = iter(build_latent_and_noise_generator(generator, config, seed=seed))
        idx = 0
        while True:
            batch = next(stream)
            if idx % world_size == rank:
                yield idx, batch
            idx += 1
    torch.random.manual_seed(seed)
    gen = torch.cuda.default_generators[device.index if device.index is not None else torch.cuda.current_device()]
    offset0 = gen.get_offset()
    first_noise = generator.make_noise()
    delta = gen.get_offset() - offset0
    rnd = 0
    while True:
        z = torch.randn(world_size * B, L)
        idx = rnd * world_size + rank
        if idx == 0:
            noise = first_noise
        else:
            gen.set_offset(offset0 + idx * delta)
            noise = generator.make_noise()
        yield idx, Latents(z[rank * B:(rank + 1) * B].clone(), noise)
        rnd += 1


@dataclass
class LabelledBatch:
    batch_index: int
    image: torch.Tensor                      # [B, 3, S, S] fp32, unclamped (what the reference hands to make_image)
    masks: Dict[str, Dict[str, torch.Tensor]]  # PredictedClusters at S x S (bool)
    activations: Dict[int, torch.Tensor]
    ids: Optional[Dict[str, torch.Tensor]] = None      # {layer: uint8 [B, H, H]} cluster ids at native resolution


@dataclass
class HostBatch:
    batch_index: int
    image: torch.Tensor                      # pinned host [B, 3, S, S] fp32, or uint8 [B, S, S, 3] (image_u8=True)
    masks: Dict[str, torch.Tensor]           # pinned host {layer: uint8 [n_class, B, S, S]}
    class_names: Dict[str, List[str]]        # {layer: class name of each mask plane}
    ids: Optional[Dict[str, torch.Tensor]] = None   # pinned host {layer: uint8 [B, H, H]} cluster ids at native resolution


@dataclass
class SegmentedBatch:
    """One batch after the host-side contour stage (create_dataset_for_segmentation.py:132-140)."""
    batch_index: int
    images: 'numpy.ndarray'                  # uint8 [B, S, S, 3]   make_image(generated_images)
    label_images: 'numpy.ndarray'            # uint8 [B, S, S, 3]   colour label images
    image_ids_to_drop: List[int]

    def kept(self):
        """(images, label_images) with the dropped rows removed (numpy.delete, as the reference does)."""
        import numpy
        return numpy.delete(self.images, self.image_ids_to_drop, axis=0), numpy.delete(self.label_images, self.image_ids_to_drop, axis=0)


@dataclass
class _Step:
    """The device results of one generate -> label step (`LabelledPairGenerator._step`)."""
    batch_index: int
    latents: Latents                         # on the device
    activations: Dict[int, torch.Tensor]
    image: torch.Tensor                      # [B, 3, S, S] fp32, or uint8 [B, S, S, 3] (image_u8=True)
    stacked: Dict[str, Tuple[List[str], torch.Tensor]]  # {layer: (class names, uint8 [n_class, B, S, S])}, merged keys included
    ids: Dict[str, torch.Tensor]             # {layer: uint8 [B, H, H]}
    lane: int
    event: torch.cuda.Event                  # recorded on the lane's stream behind the step's last kernel


class LabelledPairGenerator:
    """GPU part of `build_dataset`'s loop: generate -> label, per batch, for this rank's shard."""

    def __init__(self, generator: Generator, segmenter: ClusterSegmenter, config: Dict, seed: int = 1,
                 mean_latent: Optional[torch.Tensor] = None, rank: int = 0, world_size: int = 1,
                 capture_only_labelled: bool = False, in_flight: int = 1, mix_inject_index: Optional[int] = None):
        """`in_flight` > 1 keeps that many batches in flight on as many CUDA streams, each with its own generator
        workspace (a replica of `generator`: same weights, separate native plan).  Batches are independent, so the
        latency-bound head of one step (mapping network, 4^2..16^2 layers) overlaps the tensor-bound body of the other;
        the results are the same as with one stream (same RNG draw order), yielded in order."""
        self.generator, self.segmenter = generator, segmenter
        self.in_flight = max(1, int(in_flight))
        self._replicas, self._streams = None, None
        self.mix_inject_index = mix_inject_index
        self.replay_stream = False          # True: every rank replays every draw instead of addressing the streams by position
        self.config, self.seed, self.mean_latent = config, seed, mean_latent
        self.rank, self.world_size = rank, world_size
        # key 0 must always be present: the reference reads the batch size from activations[0]
        # (black_white_handwritten_printed_text_segmenter.py:79)
        self.capture_layers = sorted({0} | {int(k) for k in segmenter.catalog}) if capture_only_labelled else None
        self.stats = {'pairs': 0, 'batches': 0}

    def _lanes(self, device):
        """(generator replica, stream) per in-flight lane; lane 0 is the user's generator on the current stream when
        in_flight == 1."""
        if self.in_flight == 1:
            return [(self.generator, None)]
        if self._replicas is None:
            import copy
            self._replicas = [self.generator] + [copy.deepcopy(self.generator).eval() for _ in range(self.in_flight - 1)]
            self._streams = [torch.cuda.Stream(device=device) for _ in range(self.in_flight)]
            # device-side caches (centroids, class-bit tables) are filled on the current stream before the lanes fork
            self.segmenter.make_label_jobs(self.generator, self.config['batch_size'])
        current = torch.cuda.current_stream(device)
        for st in self._streams:
            st.wait_stream(current)
        return list(zip(self._replicas, self._streams))

    @staticmethod
    def _hand_over(tensors, event, device):
        """Make tensors produced on a lane stream safe to use on the caller's current stream."""
        current = torch.cuda.current_stream(device)
        current.wait_event(event)
        for t in tensors:
            if t is not None and t.is_cuda:
                t.record_stream(current)

    def _step(self, lanes, lane: int, latent_stream, z: Optional[torch.Tensor] = None, image_u8: bool = False) -> _Step:
        """Generate and label this rank's next batch on lane `lane`.  Everything is enqueued on the lane's stream: the
        noise draw (in the reference's order), the generator pass with its in-forward label jobs and the merge of the
        `keys_to_merge` layers; `event` marks its end.  `z` (pinned [B, latent_size]) stages the latents for an
        asynchronous copy in; it must not be rewritten before that copy has run."""
        device = self.generator.input.input.device
        seg = self.segmenter
        g, st = lanes[lane]
        with (torch.cuda.stream(st) if st is not None else contextlib.nullcontext()):
            idx, latents = next(latent_stream)
            if z is not None:
                z.copy_(latents.latent)
                latents = Latents(z.to(device, non_blocking=True), latents.noise)
            # labelling runs inside the generator's native call (one pass over each labelled activation)
            jobs = seg.make_label_jobs(g, latents.latent.shape[0])
            acts, image = generate_images(latents, g, device=device, mean_latent=self.mean_latent, capture_layers=self.capture_layers,
                                          label_jobs=jobs, mix_inject_index=self.mix_inject_index)
            stacked = seg.merge_stacked(seg.jobs_to_stacked(jobs))   # merged destination keys (black_white...segmenter.py:31-40)
            if image_u8:
                image = make_image(image)              # uint8 NHWC on the device: a quarter of the fp32 copy
            event = torch.cuda.Event()
            event.record(torch.cuda.current_stream(device))
        self.stats['pairs'] += image.shape[0]
        self.stats['batches'] += 1
        return _Step(idx, latents, acts, image, stacked, seg.jobs_to_ids(jobs), lane, event)

    def __iter__(self) -> Iterator[LabelledBatch]:
        import collections
        device = self.generator.input.input.device
        lanes = self._lanes(device)
        pending = collections.deque()
        stream = sharded_latent_stream(self.generator, self.config, self.seed, self.rank, self.world_size, self.replay_stream)
        n = 0
        while True:
            s = self._step(lanes, n % len(lanes), stream)
            pending.append((LabelledBatch(s.batch_index, s.image, self.segmenter._as_predicted(s.stacked), s.activations, s.ids),
                            s.event))
            n += 1
            if len(pending) >= len(lanes):
                batch, done = pending.popleft()
                if len(lanes) > 1:                   # the lanes run on streams of their own
                    self._hand_over([batch.image] + list(batch.activations.values()) + list(batch.ids.values())
                                    + [m for per_class in batch.masks.values() for m in per_class.values()], done, device)
                yield batch

    def iter_host(self, depth: int = 2, image_u8: bool = False) -> Iterator['HostBatch']:
        """The same loop with HOST buffers on both sides, as `build_dataset` needs them (its next steps are CPU code):
        latents are staged in pinned memory and copied in, the fp32 image and the per-layer uint8 mask stacks are
        copied out to pinned memory on a side stream, with `depth` batches in flight so the copies overlap the next
        batch's kernels.  A yielded HostBatch stays valid until the next one is requested."""
        device = self.generator.input.input.device
        lanes = self._lanes(device)
        depth = max(depth, len(lanes))
        B, S = self.config['batch_size'], self.generator.size
        copy_stream = torch.cuda.Stream(device=device)
        slots = [{'z': torch.empty(B, self.config['latent_size']).pin_memory(),
                  'image': (torch.empty(B, S, S, 3, dtype=torch.uint8) if image_u8 else torch.empty(B, 3, S, S)).pin_memory(),
                  'masks': {}, 'ids': {}} for _ in range(depth + 1)]
        in_flight = []

        def finish(slot):
            slot['done'].synchronize()
            slot['keep'] = None
            return HostBatch(slot['index'], slot['image'], dict(slot['masks']), slot['names'], dict(slot['ids']))

        n = 0
        latent_stream = sharded_latent_stream(self.generator, self.config, self.seed, self.rank, self.world_size, self.replay_stream)
        while True:
            slot = slots[n % (depth + 1)]
            s = self._step(lanes, n % len(lanes), latent_stream, slot['z'], image_u8)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(s.event)
                slot['image'].copy_(s.image, non_blocking=True)
                for layer, (names, m) in s.stacked.items():
                    if layer not in slot['masks']:
                        slot['masks'][layer] = torch.empty(m.shape, dtype=torch.uint8).pin_memory()
                    slot['masks'][layer].copy_(m, non_blocking=True)
                for layer, t in s.ids.items():
                    if layer not in slot['ids']:
                        slot['ids'][layer] = torch.empty(t.shape, dtype=torch.uint8).pin_memory()
                    slot['ids'][layer].copy_(t, non_blocking=True)
                slot['done'] = torch.cuda.Event()
                slot['done'].record(copy_stream)
            # the device tensors must outlive the asynchronous copies; the activations are not copied, so not held here
            slot['keep'], slot['index'] = (s.image, s.stacked, s.ids, s.latents), s.batch_index
            slot['names'] = {layer: names for layer, (names, _) in s.stacked.items()}
            in_flight.append(slot)
            n += 1
            if len(in_flight) >= depth:
                yield finish(in_flight.pop(0))

    def iter_segmented(self, depth: int = 2, pool=None, lag: int = 1, device_contours: Optional[bool] = None) -> Iterator[SegmentedBatch]:
        """generate -> label -> contour post-processing, pipelined.  Yields what the reference's loop has after
        create_segmentation_image + make_image (create_dataset_for_segmentation.py:132-140).

        `device_contours` True: the contour stage runs on the GPU right behind the labelling kernels
        (`contours_device.DeviceContourStage`); only the uint8 image, the uint8 label image and one flag per image
        leave the device, and the few images whose drop decision depends on contour order go through the host path.
        False: the masks are copied out and the per-image host tasks (`contours.segment_masks`) run on `pool` (a
        concurrent.futures executor; None = inline) while the GPU produces the next `lag` batches.
        None (default): the device when the configuration is one it handles."""
        cfg = self.segmenter.contour_config()
        if device_contours is None:
            device_contours = self.device_contours_supported()
        if device_contours:
            yield from self._iter_segmented_device(depth, pool, lag, cfg)
        else:
            yield from self._iter_segmented_host(depth, pool, lag, cfg)

    def device_contours_supported(self) -> bool:
        """Whether `iter_segmented` takes the device contour stage by default: every class is present under every key the
        stage reads, and the image size is at most 1024 (a window row of the hole fill is 32 word columns)."""
        from . import contours_device
        names = {layer: list(self.segmenter.class_label_map[layer].keys()) for layer in self.segmenter.catalog}
        for dst in self.segmenter.keys_to_merge:
            names[dst] = list(self.segmenter.class_to_color_map)
        try:
            stage = contours_device.DeviceContourStage(self.segmenter.contour_config())
        except KeyError:
            return False
        return stage.supports(names) and self.generator.size <= 1024

    def _iter_segmented_device(self, depth, pool, lag, cfg) -> Iterator[SegmentedBatch]:
        import collections

        import numpy

        from . import contours_device
        device = self.generator.input.input.device
        lanes = self._lanes(device)
        stages = [contours_device.DeviceContourStage(cfg) for _ in lanes]      # one workspace per lane
        B, S = self.config['batch_size'], self.generator.size
        copy_stream = torch.cuda.Stream(device=device)
        n_slots = max(depth, len(lanes)) + lag + 3
        slots = [{'z': torch.empty(B, self.config['latent_size']).pin_memory(),
                  'image': torch.empty(B, S, S, 3, dtype=torch.uint8).pin_memory(),
                  'label': torch.empty(B, S, S, 3, dtype=torch.uint8).pin_memory(),
                  'flags': torch.empty(B, dtype=torch.int32).pin_memory()} for _ in range(n_slots)]
        keys = set(cfg.keys_for_class_determination) | set(cfg.keys_for_finegrained_segmentation)
        pending = collections.deque()
        self.contour_stats = {'images': 0, 'host_fallback': 0, 'wait_copy_s': 0.0, 'wait_fallback_s': 0.0,
                              'enqueue_generator_s': 0.0, 'enqueue_stage_s': 0.0, 'host_copies_s': 0.0}
        fallback_lag = 8                    # batches a fall-back task may take before the loop waits for it (host copies of 8 batches)
        if pool is not None and hasattr(pool, '_max_workers'):
            # start the workers now (a spawned process imports numpy / OpenCV / this package: seconds, once), not at the
            # first fall-back in the middle of the run
            warm = [pool.submit(contours_device.warm_worker) for _ in range(pool._max_workers)]
            for w in warm:
                w.result()

        import time
        resolved = collections.deque()      # batches whose flags are known; their host fall-backs (if any) are running

        def resolve(slot):
            """Copies done: read the flags, start the host path for the undecided images (asynchronously on `pool`)."""
            t0 = time.perf_counter()
            slot['done'].synchronize()
            self.contour_stats['wait_copy_s'] += time.perf_counter() - t0
            flags = slot['flags'].numpy()
            t1 = time.perf_counter()
            images, labels = slot['image'].numpy().copy(), slot['label'].numpy().copy()
            self.contour_stats['host_copies_s'] += time.perf_counter() - t1
            drop = [int(b) for b in numpy.flatnonzero(flags == contours_device.FLAG_DROP)]
            undecided = [int(b) for b in numpy.flatnonzero(flags == contours_device.FLAG_HOST)]
            self.contour_stats['images'] += len(flags)
            self.contour_stats['host_fallback'] += len(undecided)
            tasks = []
            if undecided:
                idx = torch.as_tensor(undecided, device=device)
                host = {k: (n, m.index_select(1, idx).cpu().numpy()) for k, (n, m) in slot['stacked'].items() if k in keys}
                for j in range(len(undecided)):
                    one = {k: (n, m[:, j:j + 1]) for k, (n, m) in host.items()}
                    tasks.append(pool.submit(contours_device.host_fallback, one, [0], cfg) if pool is not None
                                 else contours_device.host_fallback(one, [0], cfg))
            slot['stacked'] = slot['keep'] = None
            resolved.append((slot['index'], images, labels, drop, undecided, tasks))

        def collect():
            index, images, labels, drop, undecided, tasks = resolved.popleft()
            t0 = time.perf_counter()
            for b, task in zip(undecided, tasks):
                res = task.result() if hasattr(task, 'result') else task
                labels[b] = res[0][0]
                if res[0][1]:
                    drop.append(b)
            self.contour_stats['wait_fallback_s'] += time.perf_counter() - t0
            return SegmentedBatch(index, images, labels, sorted(drop))

        # The stage never synchronises (its fixpoint is controlled on the device), so it is enqueued right behind the
        # batch's generator pass, on a HIGH-priority stream of its own: its ~70 short kernels slot in at the next kernel
        # boundary of the other lane's generator instead of queueing behind it, and the finished batch leaves early.
        contour_streams = [torch.cuda.Stream(device=device, priority=-1) for _ in lanes]

        def contour_and_copy(slot):
            cs = contour_streams[slot['lane']]
            with torch.cuda.stream(cs):
                cs.wait_event(slot['generated'])
                label_rgb, flags = stages[slot['lane']].run(slot['stacked'])
                ready = torch.cuda.Event()
                ready.record(cs)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ready)
                slot['image'].copy_(slot['keep'][0], non_blocking=True)
                slot['label'].copy_(label_rgb, non_blocking=True)
                slot['flags'].copy_(flags, non_blocking=True)
                slot['done'] = torch.cuda.Event()
                slot['done'].record(copy_stream)
            slot['keep'] = slot['keep'] + (label_rgb, flags)      # device tensors outlive the asynchronous work on them
            pending.append(slot)

        n = 0
        latent_stream = sharded_latent_stream(self.generator, self.config, self.seed, self.rank, self.world_size, self.replay_stream)
        while True:
            slot = slots[n % n_slots]
            t_enq = time.perf_counter()
            s = self._step(lanes, n % len(lanes), latent_stream, slot['z'], image_u8=True)
            slot['keep'], slot['stacked'], slot['index'] = (s.image, s.latents, s.activations), s.stacked, s.batch_index
            slot['lane'], slot['generated'] = s.lane, s.event
            t_stage = time.perf_counter()
            contour_and_copy(slot)
            self.contour_stats['enqueue_generator_s'] += t_stage - t_enq
            self.contour_stats['enqueue_stage_s'] += time.perf_counter() - t_stage
            n += 1
            if len(pending) > max(lag, len(lanes)):
                resolve(pending.popleft())
                if len(resolved) > fallback_lag:    # a batch's fall-backs get a few batches of time before they are waited for
                    yield collect()

    def _iter_segmented_host(self, depth, pool, lag, cfg) -> Iterator[SegmentedBatch]:
        import collections

        import numpy

        from . import contours
        keys = set(cfg.keys_for_class_determination) | set(cfg.keys_for_finegrained_segmentation)
        pending = collections.deque()

        def collect(entry):
            index, images, tasks = entry
            results = [t.result() if hasattr(t, 'result') else t for t in tasks]
            return SegmentedBatch(index, images, numpy.stack([r[0] for r in results], axis=0),
                                  [b for b, r in enumerate(results) if r[1]])

        for hb in self.iter_host(depth, image_u8=True):
            B = hb.image.shape[0]
            tasks = []
            for b in range(B):
                # the pinned slot is reused depth+1 batches later: every task gets its own copy of its image's masks
                per_image = {layer: {name: hb.masks[layer][j, b:b + 1].numpy().copy() for j, name in enumerate(hb.class_names[layer])}
                             for layer in hb.masks if layer in keys}
                tasks.append(pool.submit(contours._segment_one, (per_image, cfg)) if pool is not None
                             else contours._segment_one((per_image, cfg)))
            pending.append((hb.batch_index, hb.image.numpy().copy(), tasks))
            if len(pending) > lag:
                yield collect(pending.popleft())

    def stats_vector(self) -> torch.Tensor:
        """int64 [sum_k cluster pixel counts per labelled layer | pairs | batches] on the generator's device."""
        device = self.generator.input.input.device
        parts = [self.segmenter.cluster_pixel_counts.get(k, torch.zeros(self.segmenter.catalog[k].k, dtype=torch.int64, device=device))
                 for k in sorted(self.segmenter.catalog)]
        tail = torch.tensor([self.stats['pairs'], self.stats['batches']], dtype=torch.int64, device=device)
        return torch.cat([p.to(device) for p in parts] + [tail])


def reduce_stats(vec: torch.Tensor) -> torch.Tensor:
    """The path's only collective: all-reduce(SUM) of the statistics vector (no-op without a process group)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM)
    return vec


def split_stats(vec: torch.Tensor, catalog_sizes: Dict[str, int]) -> Dict:
    """Inverse of `stats_vector` layout."""
    out, off = {'cluster_pixels': {}}, 0
    for k in sorted(catalog_sizes):
        out['cluster_pixels'][k] = vec[off:off + catalog_sizes[k]].tolist()
        off += catalog_sizes[k]
    out['pairs'], out['batches'] = int(vec[off]), int(vec[off + 1])
    return out
