#!/usr/bin/env python
"""bench.py — labelled image pairs/sec (BASELINE.json metric), one JSON line on rank 0.

A step = one pass of the hot path over one batch of synthetic input: StyleGAN2 generator forward (random-init weights,
noise/bias parameters perturbed so every path is live) with all activation captures, followed by the nearest-centroid
labelling of the workload's layers (k=4, 3 classes) into cluster-id maps and S x S class masks.  N ranks = N independent
batch shards (weak scaling); the only collective is the final all-reduce of the statistics vector.

  --config 2 (default, the headline)  BASELINE configs[1]: 256^2, batch 32, layers 8,9,12,13
  --config 3                          BASELINE configs[2]: 512^2 config-f, batch 16, layers 8..15 (64-512 px maps)
  --config 4                          BASELINE configs[3]: 1024^2, batch 8, truncation 0.7 + style mixing, layers 12,13,16,17
  --extra-configs 3,4 (default with --config 2): short runs of the other configs, reported in the line's `configs` array

  value      pairs/s with the step's inputs (latents, noise) already resident in HBM
  e2e        same metric through the public API with HOST buffers: pinned-host latents copied in every step, noise
             drawn on the device as the reference does, image + id maps + masks copied back to pinned host memory every step
  roofline   dominant kernel (tcgen05 modulated-conv GEMM): algorithmic conv FLOPs / its CUDA-event time
  parity     2 samples of the first timed batch (the in-forward fused labelling kernels' own outputs) against the oracle
  cpu_baseline  the oracle (CPU restatement of the reference) on this box's host cores, bounded sample
  --impl reference   the oracle alone, all host threads (the reference has no CPU path of its own; BASELINE.md §1)
  gpu_reference      (N=1) the reference's graph on this GPU as the reference runs it, SURVEY §8(d), TF32 off and on
  --leg contours | dataset_gan | dataset   stage benchmarks of the rows after the hot path (SURVEY §8(f)), own JSON line
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

STYLE_DIM, N_MLP = 512, 8
CLASS_MAP = {'0': 'background', '1': 'printed_text', '2': 'handwritten_text', '3': 'background'}
COLORS = {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'}
UNIT = 'pairs/s'
K_CLUSTERS = 4

# BASELINE.json configs[1..3].  `layers`: labelled activation indices (class determination + fine-grained keys, as the
# creation JSON splits them); `mix`: crossover index of the style-mixing extension (None = single style).
WORKLOADS = {
    2: {'size': 256, 'batch': 32, 'class_keys': ['8', '9'], 'fine_keys': ['12', '13'], 'truncation': False, 'mix': None,
        'baseline': 'configs[1]',
        'text': 'StyleGAN2 256x256 random-init generator, batch 32 per GPU, 14 activation captures, nearest-centroid labelling '
                'of layers 8,9,12,13 (k=4) to id maps + 256x256 class masks (BASELINE configs[1])'},
    3: {'size': 512, 'batch': 16, 'class_keys': ['8', '9', '10', '11'], 'fine_keys': ['12', '13', '14', '15'], 'truncation': False,
        'mix': None, 'baseline': 'configs[2]',
        'text': 'StyleGAN2 512x512 config-f random-init generator, batch 16 per GPU, 16 activation captures, nearest-centroid '
                'labelling of layers 8..15 (64-512 px maps, k=4) to id maps + 512x512 class masks (BASELINE configs[2])'},
    4: {'size': 1024, 'batch': 8, 'class_keys': ['12', '13'], 'fine_keys': ['16', '17'], 'truncation': True, 'mix': 9,
        'baseline': 'configs[3]',
        'text': 'StyleGAN2 1024x1024 random-init generator, batch 8 per GPU, truncation 0.7 (mean latent of 4096 samples, fixed seed) '
                '+ style mixing (crossover index 9), 18 activation captures, nearest-centroid labelling of layers 12,13,16,17 '
                '(k=4) to id maps + 1024x1024 class masks, batch-index sharded (BASELINE configs[3])'},
}


def wl_layers(wl):
    return wl['class_keys'] + wl['fine_keys']


def metric_name(wl):
    return f'labelled image pairs/sec at {wl["size"]}^2'


def layer_res(layer):
    return 4 if int(layer) <= 1 else 2 ** ((int(layer) - 2) // 2 + 3)


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_burst': d['bf16_tflops'], 'bf16_sustained': d['bf16_tflops_sustained'], 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_burst': 1590.0, 'bf16_sustained': 1400.0, 'source': 'fallback'}


def build_info():
    """What `__graft_entry__.build()` did last (written by synthesis_in_style_b200/build.py next to the library)."""
    p = os.path.join(ROOT, 'synthesis_in_style_b200', 'lib', 'build_stamp.json')
    info = {}
    if os.path.exists(p):
        with open(p) as f:
            info = json.load(f)
    so = os.path.join(ROOT, 'synthesis_in_style_b200', 'lib', 'libsis_b200.so')
    if os.path.exists(so):
        import hashlib
        with open(so, 'rb') as f:
            info['so_sha16'] = hashlib.sha256(f.read()).hexdigest()[:16]
        info['so_bytes'] = os.path.getsize(so)
    return info


def synthetic_catalog(wl, seed=5):
    """SURVEY.md §8d: unit-norm centroids, torch.manual_seed(5); F.normalize(randn(k, C))."""
    from oracle import stylegan2_oracle as so
    ch = so.get_channels(2)
    g = torch.Generator().manual_seed(seed)
    return {layer: torch.nn.functional.normalize(torch.randn(K_CLUSTERS, ch[layer_res(layer)], generator=g), dim=1)
            for layer in wl_layers(wl)}


def oracle_state(size):
    from oracle import stylegan2_oracle as so
    spec = so.GeneratorSpec(size, STYLE_DIM, N_MLP, 2)
    sd = so.perturb_zero_params(so.init_state_dict(spec, seed=0), seed=1234)
    return spec, sd


def oracle_forward(wl, spec, sd, z, z2, noise, mean_latent):
    """The reference's path on the CPU (oracle): generator with captures (+ truncation / mixing of the workload)."""
    from oracle import stylegan2_oracle as so
    styles = [z] if wl['mix'] is None else [z, z2]
    return so.generator_forward(sd, spec, styles, noise=noise, return_intermediate_activations=True,
                                inject_index=wl['mix'], truncation=0.7 if wl['truncation'] else 1,
                                truncation_latent=mean_latent if wl['truncation'] else None)


def oracle_step(wl, spec, sd, catalog, inv_map, batch, mean_latent):
    """One CPU pass of the reference's path (generator + labelling) on `batch` samples."""
    from oracle import labelling_oracle as lo
    from oracle import stylegan2_oracle as so
    z = torch.randn(batch, STYLE_DIM)
    noise = so.make_noise(spec)
    img, acts = oracle_forward(wl, spec, sd, z, torch.roll(z, 1, 0), noise, mean_latent)
    masks = lo.prepare_image_segmentation(acts, catalog, inv_map, wl['size'])
    return img, masks


def time_oracle(wl, steps, warmup, batch):
    from oracle import labelling_oracle as lo
    from oracle import stylegan2_oracle as so
    torch.set_num_threads(os.cpu_count() or 1)
    spec, sd = oracle_state(wl['size'])
    catalog = synthetic_catalog(wl)
    inv = lo.invert_class_label_map({layer: CLASS_MAP for layer in wl_layers(wl)})
    torch.manual_seed(7)
    ml = so.mean_latent(sd, spec, 4096) if wl['truncation'] else None
    torch.manual_seed(1)
    for _ in range(warmup):
        oracle_step(wl, spec, sd, catalog, inv, batch, ml)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle_step(wl, spec, sd, catalog, inv, batch, ml)
    dt = time.perf_counter() - t0
    return steps * batch / dt, dt / steps * 1e3


def load_ref_kernels():
    """The reference's own two CUDA ops compiled by oracle/build_ref.py (None when oracle/_ref is absent)."""
    import importlib.util
    mods = {}
    for name in ('ref_fused', 'ref_upfirdn2d'):
        path = os.path.join(ROOT, 'oracle', '_ref', f'{name}.so')
        if not os.path.exists(path):
            return None
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mods[name] = mod
    return mods


def time_reference_gpu(wl, dev, steps, warmup, batch, tf32):
    """SURVEY.md §8(d) "GPU reference path": the reference's graph on THIS GPU, as the reference runs it -- cuDNN/cuBLAS
    fp32 convs, its own fused_bias_act / upfirdn2d kernels (oracle/_ref), ~150 launches per forward, then
    FactorCatalog.predict with its CPU round trip (factor_catalog.py:47-62: A.cpu(), distances + argmin on the host,
    ids .cuda()), class merge and nearest resize on the GPU.  `tf32=False` is the fp32 graph the parity criterion is
    stated against; `tf32=True` is what stock torch does to the UNMODIFIED reference (torch.backends.cudnn.allow_tf32
    defaults to True, SURVEY §8a A4).  A reported baseline (bench leg), never the product path."""
    from oracle import labelling_oracle as lo
    from oracle import stylegan2_oracle as so
    saved_flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = bool(tf32)
    torch.backends.cuda.matmul.allow_tf32 = False      # torch's default for matmul stays False
    torch.set_num_threads(os.cpu_count() or 1)
    spec, sd = oracle_state(wl['size'])
    sd = {k: v.to(dev) for k, v in sd.items()}
    catalog = synthetic_catalog(wl)
    inv = lo.invert_class_label_map({layer: CLASS_MAP for layer in wl_layers(wl)})
    ref = load_ref_kernels()
    saved = (so.fused_bias_act, so.upfirdn2d_op, lo.predict)

    def predict_round_trip(x, centroids):
        b, _, h, w = x.shape
        flat = lo.partial_flat(x).cpu()
        ids = torch.argmin(lo.pairwise_distances(flat, centroids.cpu()), dim=1)
        return ids.to(x.device).reshape(b, h, w)

    def step():
        z = torch.randn(batch, STYLE_DIM).to(dev)
        noise = [n.to(dev) for n in so.make_noise(spec)]
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        with torch.no_grad():
            img, acts = so.generator_forward(sd, spec, [z], noise=noise, return_intermediate_activations=True)
            torch.cuda.synchronize(dev)
            t1 = time.perf_counter()
            lo.prepare_image_segmentation(acts, catalog, inv, wl['size'])
        torch.cuda.synchronize(dev)
        return t1 - t0, time.perf_counter() - t0

    try:
        if ref is not None:
            so.fused_bias_act = ref['ref_fused'].fused_bias_act
            so.upfirdn2d_op = ref['ref_upfirdn2d'].upfirdn2d
        lo.predict = predict_round_trip
        torch.manual_seed(1)
        for _ in range(warmup):
            step()
        fwd = tot = 0.0
        for _ in range(steps):
            a, b = step()
            fwd += a
            tot += b
    finally:
        so.fused_bias_act, so.upfirdn2d_op, lo.predict = saved
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved_flags
    return {'value': steps * batch / tot, 'unit': UNIT, 'forward_only_images_per_s': steps * batch / fwd,
            'ms_per_step': tot / steps * 1e3, 'forward_ms_per_step': fwd / steps * 1e3, 'cudnn_allow_tf32': bool(tf32),
            'kind': f'reference graph on this GPU: cuDNN/cuBLAS fp32 (cudnn.allow_tf32={bool(tf32)}) + '
                    + ("the reference's compiled fused_bias_act/upfirdn2d kernels" if ref is not None else 'torch restatement of its two ops')
                    + ', labelling through its CPU round trip (factor_catalog.py:47-62)',
            'cores': torch.get_num_threads(), 'sample': f'{steps} timed + {warmup} warm-up steps of {batch} images, wall clock around synchronize'}


class ClockSampler:
    """SM clock and clock-event (throttle) reasons during the timed region: NVML polled every ~10 ms from a thread
    (the B200_PROFILING.md recipe's `nvidia-smi -lms 100` line gives only 1-2 samples in a 0.2 s region); falls back to
    that nvidia-smi loop when pynvml is unavailable."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    BITS = {'sw_power_cap': 0x4, 'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40,
            'hw_power_brake_slowdown': 0x80}

    def __init__(self, device):
        self.device, self.proc, self.lines, self.samples = device, None, [], []
        self.nvml, self.handle, self.stop_flag, self.thread, self.smax = None, None, False, None, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.device).uuid)
            uuid = uuid if uuid.startswith('GPU-') else 'GPU-' + uuid
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, 'encode') else uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.device.index or 0)
        return pynvml, h

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.smax = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.device.index or 0)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        reasons_fn = getattr(n, 'nvmlDeviceGetCurrentClocksEventReasons', None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.samples.append((time.perf_counter(), float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)),
                                     int(reasons_fn(self.handle))))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin, t_end):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            rows = [s for s in self.samples if t_begin <= s[0] <= t_end] or self.samples
            sm = sorted(r[1] for r in rows)
            reasons = sorted(name for name, bit in self.BITS.items() if any(r[2] & bit for r in rows))
            return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.smax, 'reasons': reasons, 'samples': len(sm),
                    'source': 'nvml, 10 ms poll'}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        rows = [l for (t, l) in self.lines if t_begin <= t <= t_end] or [l for (_, l) in self.lines]
        for l in rows:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': len(sm),
                'source': 'nvidia-smi -lms 100'}


def make_config(wl, world, batch_per_step, arm):
    """`config` of the JSON line.  The workload keys are the same for both arms; `batch_per_step` is what ONE step of
    THIS arm processes (the reference arm times a bounded sample of the workload, not its full batch)."""
    return {'workload': wl['text'], 'baseline_config': wl['baseline'], 'image_size': wl['size'], 'k': K_CLUSTERS,
            'label_layers': wl_layers(wl), 'truncation': 0.7 if wl['truncation'] else 1.0, 'style_mixing_index': wl['mix'],
            'workload_batch_per_gpu': wl['batch'], 'batch_per_step': batch_per_step, 'global_batch': batch_per_step * world,
            'arm': arm,
            'parallelism': f'batch-index sharding over {world} GPU(s), no data-path collective',
            'l2': 'per-step working set (>= 3.9 GB of captured activations) exceeds the 126 MB L2; no explicit flush'}


REFERENCE_ARM_BATCH = 4     # SURVEY §8(d) "CPU baseline timing": B = 1 and B = 4; bounded so K steps end within minutes


def run_reference(args, wl, rank, world, out):
    """Reference arm: the oracle port on the host cores (rank 0 only)."""
    if rank != 0:
        return
    batch = REFERENCE_ARM_BATCH if wl['size'] <= 256 else 1
    value, ms = time_oracle(wl, args.steps, max(1, min(args.warmup, 2)), batch)
    cores = torch.get_num_threads()
    sample = (f'each step = {batch} image(s) (a bounded sample; the GPU arm steps {wl["batch"]}) of the {wl["size"]}^2 workload '
              f'(generator + labelling of layers {",".join(wl_layers(wl))}), oracle fp32, {cores} threads')
    line = {'impl': 'reference', 'metric': metric_name(wl), 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': make_config(wl, max(1, world), batch, 'reference (CPU oracle port, bounded sample per step)'),
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), file=out, flush=True)


def run_leg_contours(args, out):
    """`--leg contours`: CPU timing of the contour stage (SURVEY §8(f) row 1) on synthetic document-like masks: product
    (synthesis_in_style_b200/contours.py) vs the restatement of the reference's algorithm (oracle/contour_oracle.py),
    same inputs, results asserted equal.  No GPU needed."""
    from concurrent.futures import ProcessPoolExecutor

    import numpy

    from oracle import contour_oracle as co
    from synthesis_in_style_b200 import contours as pc
    colors = {'background': (0, 0, 0), 'printed_text': (0, 0, 255), 'handwritten_text': (255, 0, 0)}
    images_n, oracle_n, size = 16, 4, 256
    workers = min(8, os.cpu_count() or 1)
    pred = co.synthetic_document_masks(21, images_n, size)
    cfg = pc.ContourConfig(size, colors, ['8', '9'], ['12', '13'], True, 10)
    pc.segment_masks({k: {n: m[:1] for n, m in v.items()} for k, v in pred.items()}, 1, cfg)     # warm-up
    t0 = time.perf_counter()
    images, drop = pc.segment_masks(pred, images_n, cfg)
    t_prod = time.perf_counter() - t0
    with ProcessPoolExecutor(workers) as pool:
        for _ in range(3):
            pc.segment_masks_parallel(pred, images_n, cfg, pool)                                  # workers start lazily
        t0 = time.perf_counter()
        for _ in range(3):
            images_p, drop_p = pc.segment_masks_parallel(pred, images_n, cfg, pool)
        t_par = (time.perf_counter() - t0) / 3
    assert numpy.array_equal(images, images_p) and sorted(drop) == sorted(drop_p)
    sub = {k: {nm: m[:oracle_n] for nm, m in v.items()} for k, v in pred.items()}
    t0 = time.perf_counter()
    o_images, o_drop = co.create_segmentation_image(sub, oracle_n, size, colors, ['8', '9'], ['12', '13'], True, 10)
    t_or = time.perf_counter() - t0
    assert numpy.array_equal(o_images, images[:oracle_n]) and sorted(o_drop) == sorted(d for d in drop if d < oracle_n)
    print(json.dumps({'leg': 'contours', 'image_size': size, 'images': images_n,
                      'product_ms_per_image_1_core': round(t_prod / images_n * 1e3, 2),
                      'product_images_per_s_pool': round(images_n / t_par, 1), 'pool_workers': workers,
                      'reference_algorithm_ms_per_image_1_core': round(t_or / oracle_n * 1e3, 1),
                      'speedup_1_core': round((t_or / oracle_n) / (t_prod / images_n), 1), 'results_equal': True}), file=out, flush=True)


def run_leg_dataset_gan(args, out):
    """`--leg dataset_gan`: throughput of the DatasetGAN labeller (SURVEY §8(f) row 3) at the BASELINE shape: 256^2,
    14 captures (F = 5888), 3 networks, 3 classes; captures from the B200 generator.  Timed with CUDA events:
    sis_pixel_ensemble_label over a batch and its per-category split; beside it the reference's algorithm in PyTorch on
    the same device (materialised [B,S,S,F] features, three fp32 MLPs, TF32 off) on a small batch, labels compared."""
    from oracle import dataset_gan_oracle as dg
    from oracle import stylegan2_oracle as so
    from synthesis_in_style_b200 import _lib
    from synthesis_in_style_b200 import dataset_gan as pg
    from synthesis_in_style_b200.model import Generator
    assert torch.cuda.is_available(), 'this leg needs a CUDA device'
    dev = torch.device('cuda:0')
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    batch, ref_batch, iters, SIZE = args.batch or 32, 2, 5, 256
    spec, sd = oracle_state(SIZE)
    g = Generator(SIZE, STYLE_DIM, N_MLP)
    g.load_state_dict(sd)
    g = g.to(dev).eval()
    torch.manual_seed(1)
    with torch.no_grad():
        _, acts = g([torch.randn(batch, STYLE_DIM).to(dev)], return_intermediate_activations=True, noise=[n.to(dev) for n in so.make_noise(spec)])
    feat = sum(t.shape[1] for t in acts.values())
    states = [dg.init_classifier_state(feat, 3, seed=50 + i, base_seed=49) for i in range(3)]
    ens = pg.PixelEnsembleClassifier(3, 0, 0)
    for st in states:
        net = pg.PixelClassifier(3, feat)
        net.load_state_dict(st)
        ens.add_network(net.eval())
    for _ in range(2):
        labels, _, _ = ens.predict_label_images(acts, SIZE)
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    _lib.profile_collect()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        labels, _, _ = ens.predict_label_images(acts, SIZE)
    e1.record()
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    ens.check(dev)
    ms = e0.elapsed_time(e1) / iters
    models = [dg.ClassifierParams({k: v.to(dev) for k, v in st.items()}) for st in states]
    sub = {k: v[:ref_batch] for k, v in acts.items()}
    with torch.no_grad():
        dg.predict_labels(models, sub, SIZE)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        want, margin, _ = dg.predict_labels(models, sub, SIZE)
        r1.record()
        torch.cuda.synchronize()
    ref_ms = r0.elapsed_time(r1)
    safe = margin > 1e-3
    got = labels[:ref_batch].float()
    flops = 2.0 * batch * 384 * sum(t.shape[1] * t.shape[-1] ** 2 for t in acts.values())
    print(json.dumps({'leg': 'dataset_gan', 'image_size': SIZE, 'batch': batch, 'features': feat, 'networks': 3,
                      'ms_per_batch': round(ms, 3), 'images_per_s': round(batch / ms * 1e3, 1),
                      'ms_by_category': {k: round(v[0] / iters, 3) for k, v in prof.items() if v[1]},
                      'first_layer_alg_TFLOP/s': round(flops / (prof['conv_tc'][0] / iters * 1e-3) / 1e12, 1),
                      'reference_algorithm_same_gpu': {'batch': ref_batch, 'ms_per_image': round(ref_ms / ref_batch, 2),
                                                       'images_per_s': round(ref_batch / ref_ms * 1e3, 1),
                                                       'note': 'materialised [B,S,S,F] features + three fp32 MLPs in PyTorch (TF32 off)'},
                      'labels_equal_where_margin_gt_1e-3': bool((got[safe] == want[safe]).all()),
                      'label_agreement': round(float((got == want).float().mean()), 6)}), file=out, flush=True)



def run_leg_dataset(args, dev, rank, world, out):
    """`--leg dataset`: `dataset_writer.build_dataset` end to end on config 2 -- generate -> label (GPU) -> contour stage
    (process pool) -> side-by-side PNGs (thread pool) into a scratch directory, `--steps` batches per rank.  Wall clock from
    the first batch to the last flushed file, MAX over ranks; beside it the GPU-only pair rate of the same pipeline
    (`iter_host`, nothing downstream), so the line shows what the host stages cost.  The random-init generator with
    random centroids gives noise-like masks: their contour counts are far above those of document-like masks (the
    `--leg contours` inputs), which is the worst case for the host stage."""
    import multiprocessing
    import shutil
    import tempfile
    from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

    import torch.distributed as dist
    from synthesis_in_style_b200 import dataset_creation as dc, dataset_writer as dw, labelling
    from synthesis_in_style_b200.model import Generator
    wl = WORKLOADS[2]
    B, S = (args.batch or wl['batch']), wl['size']
    if args.png:
        dw.PNG_ENCODER = args.png
    spec, sd = oracle_state(S)
    g = Generator(S, STYLE_DIM, N_MLP, precision=args.precision)
    g.load_state_dict(sd)
    g = g.to(dev).eval()
    catalog = {k: labelling.FactorCatalog(v.shape[0], v) for k, v in synthetic_catalog(wl).items()}
    seg = labelling.ClusterSegmenter(None, S, COLORS, keys_for_class_determination=wl['class_keys'],
                                     keys_for_finegrained_segmentation=wl['fine_keys'], num_clusters=K_CLUSTERS, keys_to_merge={},
                                     catalog=catalog, class_label_map={layer: CLASS_MAP for layer in wl_layers(wl)},
                                     min_class_contour_area=10)
    cfg = {'batch_size': B, 'latent_size': STYLE_DIM}
    cores = os.cpu_count() or 1
    per_rank = max(2, cores // world)
    n_contour, n_png = max(1, per_rank * 3 // 4), max(1, per_rank // 4)
    if args.contours != 'host':          # contour stage on the device: the host cores go to the PNG encoder
        n_contour, n_png = max(1, per_rank // 4), max(1, per_rank * 3 // 4)
    base = tempfile.mkdtemp(prefix=f'sis_dataset_r{rank}_', dir='/dev/shm' if os.path.isdir('/dev/shm') else None)

    def sync_max(seconds):
        t = torch.tensor([seconds], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    try:
        spawn = multiprocessing.get_context('spawn')
        # one process per contour worker (Python-heavy tasks); with device contours they only serve the rare fall-backs
        with ProcessPoolExecutor(n_contour, mp_context=spawn) as cpool, ThreadPoolExecutor(n_png) as wpool:
            # GPU-only rate of the same pipeline (host buffers out, nothing downstream)
            pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, rank=rank, world_size=world, in_flight=args.in_flight)
            it = pipe.iter_host(depth=2, image_u8=True)
            for _ in range(4):
                next(it)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                next(it)
            gpu_only = sync_max(time.perf_counter() - t0)
            del it, pipe
            # warm the worker processes, then the timed end-to-end run
            device_contours = {'device': True, 'host': False, 'auto': None}[args.contours]
            warm = dc.LabelledPairGenerator(g, seg, cfg, seed=3, rank=rank, world_size=world, in_flight=args.in_flight)
            dw.build_dataset(warm, os.path.join(base, 'warm'), 2 * B * world, cpool, wpool, device_contours=device_contours)
            del warm
            # the contour stage alone (device): one batch of this pipeline's masks, CUDA events around sis_contour_stage
            contour_ms = None
            if device_contours is not False:
                from synthesis_in_style_b200 import contours_device as cd
                probe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, rank=rank, world_size=world)
                jobs = seg.make_label_jobs(g, B)
                batch0 = next(iter(probe))
                stacked = {k: (list(v), torch.stack([m.view(torch.uint8) for m in v.values()])) for k, v in batch0.masks.items()}
                stage = cd.DeviceContourStage(seg.contour_config())
                stage.run(stacked)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    stage.run(stacked)
                e1.record()
                torch.cuda.synchronize()
                contour_ms = e0.elapsed_time(e1) / 5
                contour_info = {'ms_per_batch': round(contour_ms, 3), 'shapes': stage.last_info[0], 'fixpoint_rounds': stage.last_info[1]}
                del probe, batch0, stacked, stage, jobs
            pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, rank=rank, world_size=world, in_flight=args.in_flight)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            stats = dw.build_dataset(pipe, os.path.join(base, 'run'), args.steps * B * world, cpool, wpool, device_contours=device_contours)
            total = sync_max(time.perf_counter() - t0)
        generated = torch.tensor([stats['batches_this_rank'] * B], device=dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(generated)
        if rank == 0:
            n_gen = int(generated.item())
            print(json.dumps({'leg': 'dataset', 'metric': 'labelled pairs/s through build_dataset (generate -> label -> contours -> PNG)',
                              'value': n_gen / total, 'unit': UNIT, 'n_gpus': world, 'image_size': S, 'batch_per_gpu': B,
                              'pairs_generated': n_gen, 'images_kept_all_ranks': stats['images_kept_all_ranks'],
                              'seconds': total, 'gpu_only_pairs_per_s': world * args.steps * B / gpu_only,
                              'fraction_of_gpu_rate': (n_gen / total) / (world * args.steps * B / gpu_only),
                              'host_cores': cores, 'contour_workers_per_rank': n_contour, 'png_threads_per_rank': n_png,
                              'png_encoder': dw.PNG_ENCODER, 'contours': args.contours, 'contour_stage': stats.get('contour_stage'), 'seconds_by_part': stats.get('seconds'),
                              'device_contour_stage': contour_info if contour_ms is not None else None,
                              'scratch': 'tmpfs' if base.startswith('/dev/shm') else 'disk',
                              'note': 'wall clock, max over ranks; noise-like masks of a random-init generator (worst case for the contour stage)'}),
                  file=out, flush=True)
    finally:
        shutil.rmtree(base, ignore_errors=True)


def claim_stdout():
    """Native libraries (NCCL's version banner, ...) write to fd 1; the contract is ONE JSON line on stdout.  Keep a
    private handle on the real stdout for that line and point fd 1 at stderr for everything else."""
    real = os.fdopen(os.dup(1), 'w')
    sys.stdout.flush()
    os.dup2(2, 1)
    return real


def conv_layer_table(spec):
    """[(cin, cout, res_in, res_out, up)] of the StyledConv layers in execution order (model.py:394-441)."""
    layers = [(spec.channels[4], spec.channels[4], 4, 4, False)]
    cin = spec.channels[4]
    for i in range(3, spec.log_size + 1):
        res, cout = 2 ** i, spec.channels[2 ** i]
        layers += [(cin, cout, res // 2, res, True), (cout, cout, res, res, False)]
        cin = cout
    return layers


def parity_check(wl, spec, sd, lat, image, jobs, mean_latent, n=2):
    """`n` samples of one batch, as the timed step produced them (image + the in-forward fused labelling kernels' id
    maps), against the oracle on the same latents / noise: the north-star criteria (image max-abs error <= 2e-2 and
    PSNR >= 40 dB on the clamped images, ids bit-exact where the oracle's margin exceeds 1e-3, >= 99.9 % overall)."""
    from oracle import labelling_oracle as lo
    torch.set_num_threads(os.cpu_count() or 1)
    z_all = lat.latent.detach().cpu()
    z, z2 = z_all[:n], torch.roll(z_all, 1, 0)[:n]
    noise = [t.detach().cpu() for t in lat.noise]
    want_img, want_acts = oracle_forward(wl, spec, sd, z, z2, noise, mean_latent.cpu() if mean_latent is not None else None)
    got_img = image[:n].detach().cpu()
    err = float((got_img - want_img).abs().max())
    mse = float(((got_img.clamp(-1, 1) - want_img.clamp(-1, 1)) ** 2).mean())
    psnr = 10.0 * torch.log10(torch.tensor(4.0 / max(mse, 1e-30))).item()
    catalog = synthetic_catalog(wl)
    total = agree = unsafe = bad = 0
    for job in jobs:
        layer = str(job.activation_idx)
        ids_want, margin = lo.predict_with_margin(want_acts[int(layer)], catalog[layer])
        ids_got = job.ids_u8[:n].detach().cpu().long()
        safe = margin > 1e-3
        bad += int((ids_got[safe] != ids_want[safe]).sum())
        unsafe += int((~safe).sum())
        total += ids_want.numel()
        agree += int((ids_got == ids_want).sum())
    ok = err <= 2e-2 and psnr >= 40.0 and bad == 0 and agree / total >= 0.999
    return {'samples': n, 'batch_index': 'first timed batch of rank 0', 'image_max_abs_err': err, 'image_psnr_db_peak2': psnr,
            'label_pixels': total, 'label_agreement': agree / total, 'label_mismatches_at_margin_gt_1e-3': bad,
            'pixels_with_margin_le_1e-3': unsafe, 'ok': bool(ok),
            'source': 'id maps written by the in-forward label jobs of the timed step (label_wide_kernel / label_native_kernel)'}


DUMP_BYTES = 60 << 20        # 64 MB with room for the .npy headers


def dump_outputs(path, image, jobs):
    """`--dump-outputs`: what one step of the timed path returned -- the image, then per labelled layer the cluster-id
    map (`ids_<layer>`) and the class masks (`masks_<layer>`) -- as float32 `<name>.npy` files of at most DUMP_BYTES in
    all.  The budget is shared out smallest array first; an array that does not fit whole is stored as a flat sample at
    indices drawn with seed 0, so two runs with the same arguments sample the same elements."""
    import numpy
    arrays = {'image': image}
    for j in jobs:
        arrays[f'ids_{j.activation_idx}'] = j.ids_u8
        arrays[f'masks_{j.activation_idx}'] = j.masks
    os.makedirs(path, exist_ok=True)
    left, n_left = DUMP_BYTES // 4, len(arrays)
    for name, t in sorted(arrays.items(), key=lambda kv: kv[1].numel()):
        keep = min(t.numel(), left // n_left)
        a = t.detach().float().cpu().numpy()
        if keep < a.size:
            idx = numpy.sort(numpy.random.default_rng(0).choice(a.size, size=keep, replace=False))
            a = a.reshape(-1)[idx]
            print(f'--dump-outputs: {name} {list(t.shape)} stored as a sample of {keep} elements', file=sys.stderr)
        numpy.save(os.path.join(path, f'{name}.npy'), a)
        left, n_left = left - keep, n_left - 1


def measure(wl, args, dev, rank, world, steps, warmup, profile_steps, with_e2e=True, with_parity=True, dump_dir=None):
    """One workload on this rank: resident `value`, host-buffer `e2e`, per-kernel roofline, parity of the timed path.
    `dump_dir`: rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    import copy

    import torch.distributed as dist
    from synthesis_in_style_b200 import _lib, dataset_creation as dc, labelling
    from synthesis_in_style_b200.model import Generator
    from oracle import stylegan2_oracle as so   # shared synthetic-weight recipe + the parity checker

    B, S = (args.batch or wl['batch']), wl['size']
    layers = wl_layers(wl)
    spec, sd = oracle_state(S)
    g = Generator(S, STYLE_DIM, N_MLP, precision=args.precision)
    g.load_state_dict(sd)
    g = g.to(dev).eval()
    catalog = {k: labelling.FactorCatalog(v.shape[0], v) for k, v in synthetic_catalog(wl).items()}
    seg = labelling.ClusterSegmenter(None, S, COLORS, keys_for_class_determination=wl['class_keys'],
                                     keys_for_finegrained_segmentation=wl['fine_keys'], num_clusters=K_CLUSTERS, keys_to_merge={},
                                     catalog=catalog, class_label_map={layer: CLASS_MAP for layer in layers})
    mean_latent = None
    if wl['truncation']:
        torch.manual_seed(7)                       # the reference draws it unseeded; fixed here so every rank agrees
        with torch.no_grad():
            mean_latent = g.mean_latent(4096)
    cfg = {'batch_size': B, 'latent_size': STYLE_DIM}
    total_steps = warmup + steps
    # this rank's shard of the reference's single (latent, noise) stream: batch index = rank + i*world
    stream = dc.sharded_latent_stream(g, cfg, seed=1, rank=rank, world_size=world)
    batches = [next(stream)[1].to(dev) for _ in range(total_steps)]

    # `--in-flight` lanes: independent batches alternate over CUDA streams, each lane with its own generator workspace
    # (a replica: same weights, separate native plan), exactly what LabelledPairGenerator(in_flight=...) does
    n_lanes = max(1, args.in_flight)
    gens = [g] + [copy.deepcopy(g).eval() for _ in range(n_lanes - 1)]
    lane_streams = [torch.cuda.Stream(device=dev) for _ in range(n_lanes)] if n_lanes > 1 else [None]
    lane_out = [None] * n_lanes
    first_timed = {}

    def step_resident(lat, lane=0):
        # one native call per batch: generator + in-forward labelling (fused with ToRGB where both read the same tensor)
        jobs = seg.make_label_jobs(gens[lane], B)
        acts, img = dc.generate_images(lat, gens[lane], device=dev, mean_latent=mean_latent, label_jobs=jobs,
                                       mix_inject_index=wl['mix'])
        return img, jobs

    def run_steps(first, count, keep_first=False):
        cur = torch.cuda.current_stream(dev)
        if n_lanes == 1:
            for i in range(count):
                lane_out[0] = step_resident(batches[first + i])
                if keep_first and i == 0:
                    first_timed['out'] = lane_out[0]
            return
        for st in lane_streams:
            st.wait_stream(cur)
        done = []
        for i in range(count):
            lane = i % n_lanes
            if i >= n_lanes:
                done[i - n_lanes].synchronize()     # one batch in flight per lane: the lanes stay half a step apart
            with torch.cuda.stream(lane_streams[lane]):
                lane_out[lane] = step_resident(batches[first + i], lane)
                if keep_first and i == 0:
                    first_timed['out'] = lane_out[lane]
                ev = torch.cuda.Event()
                ev.record(lane_streams[lane])
                done.append(ev)
        for st in lane_streams:
            cur.wait_stream(st)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms_value):
        ms = torch.tensor([ms_value], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---------------------------------------------------------------- value: inputs resident in HBM
    run_steps(0, warmup, keep_first=True)     # the first warm-up batch is held like the first timed one will be, then released:
    first_timed.clear()                       # the allocator's cache then already holds blocks of those sizes
    if world > 1:                             # the timed region ends with this all-reduce: its first call (NCCL sets up the
        dc.reduce_stats(torch.cat([seg.cluster_pixel_counts[k] for k in sorted(seg.cluster_pixel_counts)]).clone())   # int64 path lazily) belongs to the warm-up
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
    import gc
    gc.collect()
    gc.disable()                              # no collector pause on the thread that enqueues the timed steps
    barrier()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    run_steps(warmup, steps, keep_first=True)
    stats = dc.reduce_stats(torch.cat([seg.cluster_pixel_counts[k] for k in sorted(seg.cluster_pixel_counts)]).clone())
    e1.record()
    barrier()
    t_end = time.perf_counter()
    gc.enable()
    launches = _lib.launch_count() - launches0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    res = {'value': world * steps * B / (ms_total / 1e3), 'ms_per_step': ms_total / steps, 'gpu_launches': launches, 'clocks': clocks,
           'stats_allreduce_sum': int(stats.sum().item()), 'batch': B, 'lanes': n_lanes}
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, *lane_out[(steps - 1) % n_lanes])      # step i ran on lane i % n_lanes

    # ---------------------------------------------------------------- parity of the timed path (rank 0)
    if with_parity and rank == 0:
        img0, jobs0 = first_timed['out']
        res['parity'] = parity_check(wl, spec, sd, batches[warmup], img0, jobs0, mean_latent)
    first_timed.clear()

    # ---------------------------------------------------------------- e2e: host buffers in and out
    # Public API: LabelledPairGenerator.iter_host — pinned-host latents in, device noise as the reference draws it,
    # fp32 image + uint8 id maps + [3, B, S, S] uint8 mask stacks out to pinned host memory every step (side stream).
    if with_e2e:
        n_cls = len(COLORS)
        h2d = B * STYLE_DIM * 4
        d2h = B * 3 * S * S * 4 + len(layers) * n_cls * B * S * S + sum(B * layer_res(l) ** 2 for l in layers)
        pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, mean_latent=mean_latent, rank=rank, world_size=world, in_flight=n_lanes,
                                        mix_inject_index=wl['mix'])
        host_iter = pipe.iter_host(depth=2)
        for _ in range(8):                               # past the one-time costs (replica plans, pinned slots): steady state
            next(host_iter)
        barrier()
        checksum = 0
        last = layers[-1]
        e0.record()
        for _ in range(steps):
            hb = next(host_iter)
            checksum += int(hb.masks[last][1, 0, 0, 0]) + int(hb.ids[last][0, 0, 0])     # touch the host result of every step
        e1.record()
        barrier()
        ms2 = max_over_ranks(e0.elapsed_time(e1))
        res['e2e'] = {'value': world * steps * B / (ms2 / 1e3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                      'ms_per_step': ms2 / steps}
        del host_iter, pipe

    # ---------------------------------------------------------------- roofline: per-kernel CUDA-event times (rank 0)
    if rank == 0 and profile_steps > 0:
        peaks = load_peaks()
        _lib.profile_enable(True)
        torch.cuda.synchronize()
        _lib.profile_collect()
        for i in range(profile_steps):
            step_resident(batches[warmup + (i % steps)])
        torch.cuda.synchronize()
        prof = _lib.profile_collect()
        _lib.profile_enable(False)
        n = profile_steps
        kernels = {k: {'ms_per_step': v[0] / n, 'launches_per_step': v[1] / n} for k, v in prof.items() if v[1]}
        table = conv_layer_table(spec)
        flops = {'wide': 0.0, 'narrow': 0.0}
        narrow_bytes = 0.0
        for cin, cout, r_in, r_out, up in table:
            which = 'narrow' if cout <= 64 else 'wide'
            flops[which] += 2.0 * B * (r_in if up else r_out) ** 2 * 9 * cin * cout
            if cout <= 64:
                narrow_bytes += 4.0 * B * (cin * r_in * r_in + cout * r_out * r_out)
        tc = args.precision == 'bf16x3'
        wide_ms = kernels.get('conv_tc' if tc else 'conv_simt', {'ms_per_step': 0.0})['ms_per_step']
        narrow_ms = kernels.get('conv_tc_narrow', {'ms_per_step': 0.0})['ms_per_step'] if tc else 0.0
        conv_ms = wide_ms + narrow_ms
        conv_flops = flops['wide'] + flops['narrow']
        achieved = conv_flops / (conv_ms / 1e3) / 1e12
        peak = peaks['bf16_sustained']
        traffic = None
        tp = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tp) and S == 256 and B == 32:
            with open(tp) as f:
                traffic = json.load(f).get('conv_tc' if tc else 'conv_simt')
        step_sum = sum(v['ms_per_step'] for v in kernels.values())
        roofline = {'bound': 'tensor', 'kernel': 'modconv_tc_* (tcgen05 implicit-GEMM modulated conv)' if tc else 'modconv3x3_simt_kernel',
                    'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak, 'traffic': traffic,
                    'peak_source': f'{peaks["source"]} bf16 sustained (kernel timed inside a long step)',
                    'passes': 3 if tc else 1, 'mma_pass_TFLOP/s': achieved * (3 if tc else 1),
                    'frac_of_split_cap': achieved * (3 if tc else 1) / peak,
                    'note': f'algorithmic FLOPs (2*MACs, SURVEY 8d) of the {len(table)} StyledConv layers per step / their summed CUDA-event '
                            'time over the profiled steps; the bf16x3 split issues 3 MMA passes per algorithmic FLOP (SURVEY §7: one '
                            'bf16 / tf32 pass cannot meet the label criterion), so `frac` is capped at 1/3 and `frac_of_split_cap` '
                            'is the tensor-pipe view',
                    'profiled_steps': n, 'share_of_step': conv_ms / step_sum}
        if flops['narrow'] > 0 and narrow_ms > 0:
            roofline['wide_layers'] = {'TFLOP/s': flops['wide'] / (wide_ms / 1e3) / 1e12, 'ms_per_step': wide_ms}
            gbs = narrow_bytes / (narrow_ms / 1e3) / 1e9
            roofline['narrow_layers'] = {'what': 'StyledConv layers with Cout <= 64 (AI <= 144 FLOP/B in fp32: SURVEY §8d ridge check reports '
                                                 'them against HBM)', 'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                                         'frac': gbs / peaks['hbm_gbs'], 'TFLOP/s': flops['narrow'] / (narrow_ms / 1e3) / 1e12,
                                         'ms_per_step': narrow_ms,
                                         'bytes_model': '4 B x (B*Cin*Hin^2 + B*Cout*Hout^2): each layer reads its input once and writes its output once'}
        # HBM-side view of the memory-bound kernels (bytes model in DESIGN.md)
        hbm = {}
        ch = spec.channels
        n_cls = len(COLORS)
        lbl_bytes = sum(B * ch[layer_res(l)] * layer_res(l) ** 2 * 4 + B * layer_res(l) ** 2 + n_cls * B * S * S for l in layers)
        resolutions = [2 ** i for i in range(2, spec.log_size + 1)]
        rgb_bytes = sum(B * ch[r] * r * r * 4 + B * 3 * r * r * 4 + B * 3 * (r // 2) ** 2 * 4 for r in resolutions)
        # a ToRGB rides in the labelling pass of the same tensor (odd layers = second conv of a block) when the map is wide enough
        fused_saved = sum(B * ch[layer_res(l)] * layer_res(l) ** 2 * 4 for l in layers
                          if int(l) % 2 == 1 and B * layer_res(l) ** 2 // 4 >= 148 * 160)
        lr_ms = kernels.get('label', {'ms_per_step': 0})['ms_per_step'] + kernels.get('torgb', {'ms_per_step': 0})['ms_per_step']
        if lr_ms > 0:
            hbm['label+torgb'] = {'GB/s': (lbl_bytes + rgb_bytes - fused_saved) / (lr_ms / 1e3) / 1e9,
                                  'note': 'labelling launches (ToRGB of the same tensor fused in where the map is wide) + the remaining '
                                          'ToRGB launches; the tiny 4^2..32^2 ToRGB launches are latency-bound'}
        if 'blur_split' in kernels:
            bl_bytes = sum(B * ch[r] * ((r + 1) ** 2 * 4 + r * r * 8) for r in resolutions[1:])
            hbm['blur_split'] = {'GB/s': bl_bytes / (kernels['blur_split']['ms_per_step'] / 1e3) / 1e9}
        for v in hbm.values():
            v['frac_of_hbm_peak'] = v['GB/s'] / peaks['hbm_gbs']
        roofline['memory_bound_kernels'] = hbm
        roofline['captured_activation_bytes_per_step'] = sum(B * ch[layer_res(i)] * layer_res(i) ** 2 * 4 for i in range(spec.n_latent))
        res['roofline'], res['kernels'] = roofline, kernels
    del gens, g, batches
    torch.cuda.empty_cache()
    return res


def main():
    out = claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--precision', default='bf16x3', choices=['bf16x3', 'fp32'])
    ap.add_argument('--config', type=int, default=2, choices=sorted(WORKLOADS), help='BASELINE.json workload (2 = configs[1], the headline)')
    ap.add_argument('--extra-configs', default=None,
                    help='comma list of further workloads measured briefly into the `configs` array (default "3,4" with --config 2; "" = none)')
    ap.add_argument('--batch', type=int, default=0, help='override the workload batch per GPU (0 = the BASELINE batch)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--profile-steps', type=int, default=10)
    ap.add_argument('--in-flight', type=int, default=2, choices=[1, 2],
                    help='batches in flight on separate CUDA streams / generator workspaces (3 measured slower: do not)')
    ap.add_argument('--png', default='', choices=['', 'fast', 'stored', 'cv2', 'pil'],
                    help='--leg dataset: PNG writer (dataset_writer.PNG_ENCODER; default: the module default)')
    ap.add_argument('--contours', default='auto', choices=['auto', 'device', 'host'],
                    help='--leg dataset: contour stage on the device (sis_contour_stage) or as host tasks')
    ap.add_argument('--leg', default='', choices=['', 'contours', 'dataset_gan', 'dataset'],
                    help='run one of the extra stage benchmarks (rows after the hot path) instead of the headline metric')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='write the image, id maps and class masks of the last timed step of --config to DIR/<name>.npy '
                         '(float32, <= 64 MB in all, larger arrays as a fixed seeded sample; rank 0)')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == 'reference' or args.leg):
        ap.error('--dump-outputs writes the outputs of the headline measurement (--impl b200, no --leg)')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    wl = WORKLOADS[args.config]

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        run_reference(args, wl, rank, world, out)
        return
    if args.leg in ('contours', 'dataset_gan'):
        if rank == 0:
            (run_leg_contours if args.leg == 'contours' else run_leg_dataset_gan)(args, out)
        return

    import torch.distributed as dist

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    if args.leg == 'dataset':
        run_leg_dataset(args, dev, rank, world, out)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    main_res = measure(wl, args, dev, rank, world, args.steps, args.warmup, args.profile_steps, dump_dir=args.dump_outputs)

    extra = []
    extra_ids = args.extra_configs if args.extra_configs is not None else ('3,4' if args.config == 2 and not args.batch else '')
    for cid in [int(c) for c in extra_ids.split(',') if c.strip()]:
        if cid == args.config or cid not in WORKLOADS:
            continue
        w2 = WORKLOADS[cid]
        try:
            r = measure(w2, args, dev, rank, world, min(args.steps, 10), 3, min(args.profile_steps, 5))
            entry = {'config': cid, 'metric': metric_name(w2), 'unit': UNIT, 'workload': w2['text'], 'n_gpus': world,
                     'steps': min(args.steps, 10), 'warmup': 3}
            entry.update(r)
        except Exception as exc:   # an extra workload must never take the headline down
            entry = {'config': cid, 'metric': metric_name(w2), 'error': f'{type(exc).__name__}: {exc}'[:400]}
            torch.cuda.empty_cache()
        extra.append(entry)

    # ---------------------------------------------------------------- CPU baseline + reference graph on this GPU (rank 0, N=1 only)
    cpu = gpu_ref = gpu_ref_tf32 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, ms_cpu = time_oracle(wl, 10, 1, 1)
        cpu = {'value': v, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
               'sample': f'10 timed + 1 warm-up steps of 1 image ({wl["size"]}^2 generator + labelling of layers {",".join(wl_layers(wl))}), oracle fp32'}
        B = args.batch or wl['batch']
        gpu_ref = time_reference_gpu(wl, dev, 5, 1, B, tf32=False)
        gpu_ref_tf32 = time_reference_gpu(wl, dev, 5, 1, B, tf32=True)

    if rank == 0:
        B = main_res['batch']
        line = {'metric': metric_name(wl), 'value': main_res['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': main_res['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16x3 (3-term bf16 split, fp32 accumulate)' if args.precision == 'bf16x3' else 'f32', 'data': 'synthetic',
                'config': dict(make_config(wl, world, B, 'b200'), in_flight_batches=main_res['lanes'],
                               pipelining=f'{main_res["lanes"]} independent batches in flight per GPU on separate CUDA streams / generator workspaces'),
                'e2e': main_res.get('e2e'), 'gpu_launches': main_res['gpu_launches'], 'clocks': main_res['clocks'],
                'roofline': main_res.get('roofline'), 'kernels': main_res.get('kernels'), 'parity': main_res.get('parity'),
                'cpu_baseline': cpu, 'gpu_reference': gpu_ref, 'gpu_reference_tf32': gpu_ref_tf32,
                'stats_allreduce_sum': main_res['stats_allreduce_sum'], 'configs': extra, 'build': build_info()}
        print(json.dumps(line), file=out, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
