"""Catalog creation at 256^2: sampling time, then per layer the k-means step loop of every k run two ways on the same
inputs, alternated in one process -- the library's batched loop (`sis_kmeans_steps`, one launch per chunk of
KMEANS_CHUNK_STEPS steps for all k, one host read per chunk) and the host-driven loop (oracle/kmeans_oracle.py in fp32 on
the GPU: one fit after the other, about 15 small launches and at least two host synchronisations per step) -- and the
whole `fit_catalogs` (seeding, steps, labelling) per layer.  Prints one JSON line with the card's name and power limit.

    python scripts/catalog_bench.py [-n 100] [--layers 8 9 12 13] [--cluster-range 3 24] [--reps 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import kmeans_oracle as ko                                       # noqa: E402
from synthesis_in_style_b200 import catalog_creation as cc                   # noqa: E402
from synthesis_in_style_b200 import create_catalogs                          # noqa: E402
from synthesis_in_style_b200.model import Generator                          # noqa: E402


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def init_centres(x, ks):
    """The first k rows of a fixed permutation: the same start for both loops."""
    perm = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(0))[:max(ks)].to(x.device)
    return {k: x[perm[:k]].clone() for k in ks}


def device_loop(x, init, batch_size, max_steps):
    fits = [cc.KMeansFit(x, c.clone()) for c in init.values()]
    states = cc.new_states(len(fits), x.device)
    for f, s in zip(fits, states):
        f.state = s
        cc.init_state(f, 0, batch_size, max_steps, 10, 0.01)
    active, launches = list(range(len(fits))), 0
    while active:
        cc.kmeans_steps([fits[i] for i in active], cc.KMEANS_CHUNK_STEPS)
        launches += 1
        done = states[active, 3].cpu().tolist()
        active = [i for i, d in zip(active, done) if not d]
    return {'steps': int(states[:, 1].sum()), 'launches': launches, 'host_syncs': launches}


def oracle_loop(x, init, batch_size, max_steps):
    steps = 0
    for c in init.values():
        _, _, n = ko.fit_steps(x, c.clone(), torch.zeros(c.shape[0], device=x.device), seed=0, batch_size=batch_size,
                               max_steps=max_steps, max_no_improvement=10, ratio=0.01)
        steps += n
    return {'steps': steps}


def main():
    p = argparse.ArgumentParser()
    p.add_argument('-n', '--num-images', type=int, default=100)
    p.add_argument('-b', '--batch-size', type=int, default=10)
    p.add_argument('--size', type=int, default=256)
    p.add_argument('--layers', type=int, nargs='+', default=[8, 9, 12, 13])
    p.add_argument('--cluster-range', type=int, nargs=2, default=[3, 24])
    p.add_argument('--reps', type=int, default=2)
    a = p.parse_args()
    dev = torch.device('cuda', 0)
    ks = list(range(*a.cluster_range))
    torch.manual_seed(0)
    g = Generator(a.size, 512, 8, channel_multiplier=2).to(dev).eval()
    config = {'batch_size': a.batch_size, 'latent_size': 512}
    create_catalogs.sample_activations(g, config, a.batch_size, 1, a.layers, dev)               # warm-up
    t_sample, (acts, _) = timed(lambda: create_catalogs.sample_activations(g, config, a.num_images, 1, a.layers, dev))
    result = {'card': card(), 'size': a.size, 'num_images': a.num_images, 'layers': a.layers, 'ks': [ks[0], ks[-1] + 1],
              'kmeans_chunk_steps': cc.KMEANS_CHUNK_STEPS, 'sample_s': round(t_sample, 3), 'per_layer': {}}
    bs = 100
    for layer in a.layers:
        act = acts[layer]
        x = cc._normalize_rows(act.permute(0, 2, 3, 1).reshape(-1, act.shape[1]).float()).contiguous()
        max_steps = 100 * ((x.shape[0] + bs - 1) // bs)
        init = init_centres(x, ks)
        row = {'points': int(x.shape[0]), 'channels': int(x.shape[1]), 'device_loop_s': [], 'oracle_loop_s': []}
        for _ in range(a.reps):                     # alternated: device, host-driven, device, host-driven, ...
            t, row['device_loop'] = timed(lambda: device_loop(x, init, bs, max_steps))
            row['device_loop_s'].append(round(t, 4))
            t, row['oracle_loop'] = timed(lambda: oracle_loop(x, init, bs, max_steps))
            row['oracle_loop_s'].append(round(t, 4))
        stats = {}
        t, _ = timed(lambda: cc.fit_catalogs({layer: act}, ks, 0, stats=stats))
        row['fit_catalogs_s'], row['fit_catalogs_stats'] = round(t, 3), stats
        result['per_layer'][str(layer)] = row
    print(json.dumps(result))


if __name__ == '__main__':
    main()
