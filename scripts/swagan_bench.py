"""SWAGAN 256^2 on the fused plan: resident labelled-pair rate, per-category kernel time, launches per step and parity
against the CPU oracle, with the StyleGAN2 256^2 rate of the same labelling setup beside it.  Prints one JSON line.

Workload (both generators): random-init weights with the zero-init parameters perturbed (bench.oracle_state's recipe),
batch 32, every activation captured, nearest-centroid labelling (k = 4) of layers 8, 9 (64^2, 512 ch; class
determination) and 10, 11 (128^2, 256 ch; fine-grained) to id maps and 256^2 class masks inside the forward, two batches
in flight on two CUDA streams, timed with CUDA events after a warm-up.

    python scripts/swagan_bench.py [--steps 400] [--warmup 20]
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import CLASS_MAP, COLORS, K_CLUSTERS, N_MLP, STYLE_DIM  # noqa: E402
from oracle import labelling_oracle as lo  # noqa: E402
from oracle import stylegan2_oracle as so  # noqa: E402
from oracle import swagan_oracle as sw  # noqa: E402
from synthesis_in_style_b200 import _lib, labelling, model, swagan  # noqa: E402
from synthesis_in_style_b200 import dataset_creation as dc  # noqa: E402

SIZE, BATCH, LANES = 256, 32, 2
CLASS_KEYS, FINE_KEYS = ['8', '9'], ['10', '11']
LAYERS = CLASS_KEYS + FINE_KEYS
POOL = 8          # distinct input batches, cycled: the work per step does not depend on the values


def gpu_info(dev):
    info = {'gpu': torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(dev.index or 0), '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as err:
        info['power_limit_and_max_sm_clock'] = f'not read: {err}'
    return info


def build(kind, dev):
    if kind == 'swagan':
        spec = sw.SwaganSpec(SIZE, STYLE_DIM, N_MLP)
        sd = so.perturb_zero_params(sw.init_state_dict(spec, seed=0), seed=1234)
        g = swagan.Generator(SIZE, STYLE_DIM, N_MLP)
    else:
        spec = so.GeneratorSpec(SIZE, STYLE_DIM, N_MLP, 2)
        sd = so.perturb_zero_params(so.init_state_dict(spec, seed=0), seed=1234)
        g = model.Generator(SIZE, STYLE_DIM, N_MLP)
    g.load_state_dict(sd)
    g = g.to(dev).eval()
    gen = torch.Generator().manual_seed(5)
    catalog = {}
    for layer in LAYERS:
        c, _ = g.activation_shape(int(layer))
        catalog[layer] = labelling.FactorCatalog(K_CLUSTERS, torch.nn.functional.normalize(torch.randn(K_CLUSTERS, c, generator=gen), dim=1))
    seg = labelling.ClusterSegmenter(None, SIZE, COLORS, keys_for_class_determination=CLASS_KEYS, keys_for_finegrained_segmentation=FINE_KEYS,
                                     num_clusters=K_CLUSTERS, keys_to_merge={}, catalog=catalog,
                                     class_label_map={layer: CLASS_MAP for layer in LAYERS})
    return spec, sd, g, seg


def measure(kind, dev, steps, warmup, profile_steps):
    spec, sd, g, seg = build(kind, dev)
    stream = dc.sharded_latent_stream(g, {'batch_size': BATCH, 'latent_size': STYLE_DIM}, seed=1, rank=0, world_size=1)
    batches = [next(stream)[1].to(dev) for _ in range(POOL)]
    gens = [g] + [copy.deepcopy(g).eval() for _ in range(LANES - 1)]
    lane_streams = [torch.cuda.Stream(device=dev) for _ in range(LANES)]

    def step(lat, lane):
        jobs = seg.make_label_jobs(gens[lane], BATCH)
        _, img = dc.generate_images(lat, gens[lane], device=dev, label_jobs=jobs)
        return img, jobs

    def run(count):
        """`count` steps alternating over the lanes, one batch in flight per lane (LabelledPairGenerator(in_flight=2))."""
        cur = torch.cuda.current_stream(dev)
        for st in lane_streams:
            st.wait_stream(cur)
        done, out = [], None
        for i in range(count):
            lane = i % LANES
            if i >= LANES:
                done[i - LANES].synchronize()
            with torch.cuda.stream(lane_streams[lane]):
                out = step(batches[i % POOL], lane)
                ev = torch.cuda.Event()
                ev.record(lane_streams[lane])
                done.append(ev)
        for st in lane_streams:
            cur.wait_stream(st)
        return out

    run(warmup)
    torch.cuda.synchronize()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    for x in gens:
        x.check()
    res = {'pairs_per_s': round(steps * BATCH / (ms / 1e3), 1), 'ms_per_step': round(ms / steps, 3),
           'timed_s': round(ms / 1e3, 2), 'launches_per_step': (_lib.launch_count() - launches0) / steps}
    # per-category kernel time: a separate run (events around every launch slow the host)
    _lib.profile_collect()
    _lib.profile_enable(True)
    run(profile_steps)
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    res['kernel_ms_per_step'] = {k: round(v[0] / profile_steps, 3) for k, v in prof.items() if v[1]}
    res['launches_per_step_by_category'] = {k: v[1] / profile_steps for k, v in prof.items() if v[1]}
    if kind == 'swagan':
        res['parity'] = parity(spec, sd, g, seg, batches[0], dev)
    return res


def parity(spec, sd, g, seg, lat, dev, n=2):
    """`n` samples against oracle/swagan_oracle.py on the same latents and noise, with bench.parity_check's criterion:
    image max-abs error <= 2e-2 and PSNR >= 40 dB on the clamped images, ids bit-exact where the oracle's margin exceeds
    1e-3, >= 99.9 % agreement overall."""
    jobs = seg.make_label_jobs(g, BATCH)
    _, img = dc.generate_images(lat, g, device=dev, label_jobs=jobs)
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    want_img, want_acts = sw.generator_forward(sd, spec, [lat.latent[:n].cpu()], noise=[t.cpu() for t in lat.noise],
                                               return_intermediate_activations=True)
    got = img[:n].cpu()
    err = float((got - want_img).abs().max())
    mse = float(((got.clamp(-1, 1) - want_img.clamp(-1, 1)) ** 2).mean())
    psnr = 10.0 * torch.log10(torch.tensor(4.0 / max(mse, 1e-30))).item()
    total = agree = bad = 0
    for job in jobs:
        ids_want, margin = lo.predict_with_margin(want_acts[job.activation_idx], job.centroids.cpu())
        ids_got = job.ids_u8[:n].cpu().long()
        safe = margin > 1e-3
        bad += int((ids_got[safe] != ids_want[safe]).sum())
        total += ids_want.numel()
        agree += int((ids_got == ids_want).sum())
    ok = err <= 2e-2 and psnr >= 40.0 and bad == 0 and agree / total >= 0.999
    return {'status': 'ok' if ok else 'FAIL', 'samples': n, 'image_max_abs_err': err, 'psnr_db': round(psnr, 2),
            'ids_mismatch_where_margin_gt_1e-3': bad, 'label_agreement': round(agree / total, 6)}


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--steps', type=int, default=400)
    p.add_argument('--warmup', type=int, default=20)
    p.add_argument('--profile-steps', type=int, default=20)
    args = p.parse_args()
    assert torch.cuda.is_available(), 'swagan_bench needs a CUDA device'
    dev = torch.device('cuda:0')
    torch.manual_seed(0)
    t0 = time.time()
    out = {'workload': f'SWAGAN {SIZE}x{SIZE} random-init, batch {BATCH}, captures 0..11, nearest-centroid labelling (k={K_CLUSTERS}) '
                       f'of layers 8,9 (class) + 10,11 (fine) to id maps + {SIZE}x{SIZE} masks, {LANES} batches in flight',
           **gpu_info(dev)}
    out['swagan'] = measure('swagan', dev, args.steps, args.warmup, args.profile_steps)
    out['stylegan2_same_setup'] = measure('stylegan2', dev, args.steps, args.warmup, args.profile_steps)
    out['swagan_over_stylegan2'] = round(out['swagan']['pairs_per_s'] / out['stylegan2_same_setup']['pairs_per_s'], 3)
    out['wall_s'] = round(time.time() - t0, 1)
    print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
