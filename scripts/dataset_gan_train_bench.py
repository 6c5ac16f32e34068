"""Training rate of the DatasetGAN pixel-classifier ensemble at 256^2 with 16 annotated images and 3 networks: the device
trainer (`sis_pixel_train_*`) against the same recipe in plain PyTorch on the same GPU (the feature tensor materialised
in fp32, cuBLAS fp32 GEMMs with TF32 off, torch.optim.Adam), with the card's name and power limit.

    python scripts/dataset_gan_train_bench.py [--steps 2048] [--warmup 256] [--torch-steps 512] [--out result.json]

Steps/s counts steps of the whole ensemble (every network advances one batch).  The device rate is the difference of
two host-timed `fit` calls (--warmup and --warmup + --steps steps), so set-up and the parameter read-back cancel; it
ends in a device synchronise.  The captures (1.9 GB) and the PyTorch feature tensor (24.7 GB) exceed the L2, the
working set of a step (W1 and its Adam moments, 27 MB for three networks) does not.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from synthesis_in_style_b200 import train_dataset_gan as tg  # noqa: E402
from synthesis_in_style_b200.model import Generator  # noqa: E402

N_IMAGES, SIZE, N_MODELS, N_CLASS, BATCH = 16, 256, 3, 4, 64


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0)


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def torch_rate(acts, labels, steps, warmup):
    """The same recipe over the materialised [A*S*S, F] feature tensor."""
    dev = labels.device
    n = labels.numel()
    feats = torch.empty(n, sum(a.shape[1] for a in acts.values()), device=dev)
    off = 0
    for a in acts.values():
        for i in range(a.shape[0]):
            up = F.interpolate(a[i:i + 1], scale_factor=SIZE / a.shape[-1], mode='bilinear')
            feats[i * SIZE * SIZE:(i + 1) * SIZE * SIZE, off:off + a.shape[1]] = up[0].reshape(a.shape[1], -1).t()
        off += a.shape[1]
    y = labels.reshape(-1).long()
    nets, opts, orders = [], [], []
    for m in range(N_MODELS):
        net = tg.initial_network(0, m, N_CLASS, feats.shape[1]).layers.to(dev).train()
        nets.append(net)
        opts.append(torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8))
        orders.append(torch.randperm(n, device=dev))
    loss_fn = torch.nn.CrossEntropyLoss()

    def run(count, start):
        for t in range(start, start + count):
            for net, opt, order in zip(nets, opts, orders):
                idx = order[t * BATCH:(t + 1) * BATCH]
                opt.zero_grad()
                loss_fn(net(feats[idx]), y[idx]).backward()
                opt.step()
    run(warmup, 0)
    dt, _ = timed(lambda: run(steps, warmup))
    return steps / dt


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--steps', type=int, default=2048)
    parser.add_argument('--warmup', type=int, default=256)
    parser.add_argument('--torch-steps', type=int, default=512)
    parser.add_argument('--out', default=None)
    args = parser.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('dataset_gan_train_bench needs a CUDA device')
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device('cuda:0')
    torch.manual_seed(0)
    gen = Generator(SIZE, 512, 8).to(dev).eval()
    g = torch.Generator().manual_seed(1)
    z = torch.randn(N_IMAGES, 512, generator=g)
    noise = [torch.randn(N_IMAGES, 1, 2 ** ((i + 5) // 2), 2 ** ((i + 5) // 2), generator=g) for i in range(gen.num_layers)]
    with torch.no_grad():
        w = gen.get_latent(z.to(dev)).cpu()
    labels = torch.randint(0, N_CLASS, (N_IMAGES, SIZE, SIZE), generator=g, dtype=torch.uint8)
    trainer = tg.PixelEnsembleTrainer(gen, (w, noise, labels), N_CLASS, num_models=N_MODELS, batch_pixels=BATCH)
    t_warm, _ = timed(lambda: trainer.fit(max_steps=args.warmup))
    t_full, _ = timed(lambda: trainer.fit(max_steps=args.warmup + args.steps))
    dev_rate = args.steps / (t_full - t_warm)
    steps_per_epoch = N_IMAGES * SIZE * SIZE // BATCH
    acts = {i: a for i, a in enumerate(trainer.acts)}
    torch_steps = torch_rate(acts, trainer.labels, args.torch_steps, min(args.warmup, 64))
    result = {'card': card(), 'image_size': SIZE, 'annotated_images': N_IMAGES, 'networks': N_MODELS, 'batch_pixels': BATCH,
              'feature_size': trainer.feature_size, 'steps_per_epoch': steps_per_epoch,
              'device': {'steps_per_s': dev_rate, 'pixels_per_s': dev_rate * BATCH * N_MODELS, 's_per_epoch': steps_per_epoch / dev_rate,
                         'timed_steps': args.steps},
              'torch_fp32': {'steps_per_s': torch_steps, 'pixels_per_s': torch_steps * BATCH * N_MODELS,
                             's_per_epoch': steps_per_epoch / torch_steps, 'timed_steps': args.torch_steps}}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
