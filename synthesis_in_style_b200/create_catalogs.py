"""Cluster catalogs from a trained generator: step 1 of the cluster-based workflow (cluster -> label the clusters by hand
in `merged_classes_{k}.json` -> `create_dataset`).  Follows the flow of scf/create_semantic_segmentation.py (SURVEY.md
§3.2): sample images, keep the activations of the selected layers, fit spherical k-means for every k of a range on
every layer, save the catalogs.  Its flags are this project's own and follow `create_dataset`'s names; it makes no
claim to match the reference script's flags or its labelling UI.

    python -m synthesis_in_style_b200.create_catalogs CHECKPOINT -ssd <run>/semantic_segmentation [-op original_config.json]
        [-n 100] [-b 10] [-d cuda] [--truncate] [--seed 1] [--layers 8 9 12 13 | --min-size 32] [--cluster-range 3 24]
        [--random-state 0] [--kmeans-batch-size 100] [--max-iter 100] [--n-init 3] [--init-size N]
        [--reassignment-ratio 0.01] [--max-no-improvement 10]

CHECKPOINT is a generator checkpoint (StyleGAN2 or SWAGAN, as `create_dataset` loads it) or `random-init:<seed>`
(then `-op` names the original config).  Without `-ssd` the output goes to `<checkpoint>/../../semantic_segmentation`.
`--layers` selects activation indices; by default every capture whose map is larger than `--min-size` is used.
`--cluster-range MIN MAX` is half open.  `--max-no-improvement -1` disables early stopping.  Writes
  <ssd>/catalogs/{k}.npz        {layer: float32 [k, C] unit centres}, what `create_dataset` reads
  <ssd>/cluster_arrays/{k}.npz  `images` uint8 [N, S, S, 3] and, per layer, the uint8 [N, H, W] cluster id maps
All fits of all k and layers run together (catalog_creation.fit_catalogs); the captures never leave the device.
"""
import argparse
from pathlib import Path
from typing import Dict

import numpy
import torch

from . import create_dataset as cd
from . import dataset_creation as dc
from .catalog_creation import fit_catalogs, save_catalogs
from .labelling import make_image


def sample_activations(generator, config: Dict, num_images: int, seed: int, layers, device, mean_latent=None):
    """(activations {layer: [N, C, H, W]} on the device, images uint8 [N, S, S, 3] on the host)."""
    acts = {layer: [] for layer in layers}
    images, got = [], 0
    for _, batch in dc.sharded_latent_stream(generator, config, seed, 0, 1):
        activations, image = dc.generate_images(batch, generator, device=device, mean_latent=mean_latent, capture_layers=layers)
        for layer in layers:
            acts[layer].append(activations[layer])
        images.append(make_image(image).cpu().numpy())
        got += image.shape[0]
        if got >= num_images:
            break
    return ({layer: torch.cat(a)[:num_images] for layer, a in acts.items()},
            numpy.concatenate(images)[:num_images])


def main(args: argparse.Namespace) -> Dict:
    ckpt = str(args.checkpoint)
    config = cd.load_config(None if ckpt.startswith('random-init:') else ckpt, args.original_config_path)
    config['batch_size'] = args.batch_size
    if args.semantic_segmentation_base_dir is not None:
        ssd = Path(args.semantic_segmentation_base_dir)
    elif ckpt.startswith('random-init:'):
        raise ValueError('a random-init generator needs -ssd')
    else:
        ssd = Path(ckpt).parent.parent / 'semantic_segmentation'
    k_min, k_max = args.cluster_range
    if not 2 <= k_min < k_max:
        raise ValueError(f'--cluster-range {k_min} {k_max}: need 2 <= MIN < MAX')
    device = cd.resolve_device(args.device)
    with torch.cuda.device(device):
        generator = cd.load_generator(args, config, device)
        layers = args.layers if args.layers else [i for i in range(generator.n_latent)
                                                  if generator.activation_shape(i)[1] > args.min_size]
        mean_latent = None
        if args.truncate:
            with torch.no_grad():
                mean_latent = generator.mean_latent(4096)
        acts, images = sample_activations(generator, config, args.num_images, args.seed, layers, device, mean_latent)
        fitted = fit_catalogs(acts, range(k_min, k_max), args.random_state, batch_size=args.kmeans_batch_size,
                              max_iter=args.max_iter, n_init=args.n_init, init_size=args.init_size,
                              reassignment_ratio=args.reassignment_ratio,
                              max_no_improvement=None if args.max_no_improvement < 0 else args.max_no_improvement)
    written = {}
    for k in range(k_min, k_max):
        save_catalogs({str(layer): fitted[layer][k][0] for layer in layers}, k, ssd / 'catalogs')
        (ssd / 'cluster_arrays').mkdir(parents=True, exist_ok=True)
        numpy.savez(ssd / 'cluster_arrays' / f'{k}.npz', images=images,
                    **{str(layer): fitted[layer][k][1].to(torch.uint8).cpu().numpy() for layer in layers})
        written[k] = ssd / 'catalogs' / f'{k}.npz'
    return {'layers': layers, 'catalogs': written, 'num_images': int(images.shape[0])}


def build_arg_parser() -> argparse.ArgumentParser:
    parser = argparse.ArgumentParser(description='Cluster the activations of a trained generator into catalogs '
                                                 '(<ssd>/catalogs/{k}.npz) for the cluster-based dataset creation.')
    parser.add_argument('checkpoint', help='Path to the trained autoencoder/generator, or random-init:<seed>')
    parser.add_argument('-op', '--original-config-path', type=Path, default=None,
                        help='YAML/JSON config of the original training, if it is not in a sibling directory of the checkpoint')
    parser.add_argument('-n', '--num-images', type=int, default=100, help='Number of images whose activations are clustered')
    parser.add_argument('-b', '--batch-size', default=10, type=int, help='batch size for generation of images on GPU')
    parser.add_argument('-d', '--device', default='cuda', help='CUDA device to use, either any (cuda) or the id of the device')
    parser.add_argument('--truncate', action='store_true', default=False, help='Use truncation trick during generation')
    parser.add_argument('--seed', type=int, default=1, help='seed of the latent and noise stream')
    parser.add_argument('-ssd', '--semantic-segmentation-base-dir', type=Path, default=None,
                        help='where catalogs/ and cluster_arrays/ are written (default: <checkpoint>/../../semantic_segmentation)')
    parser.add_argument('--layers', type=int, nargs='+', default=None, help='activation indices to cluster')
    parser.add_argument('--min-size', type=int, default=32,
                        help='without --layers: cluster every activation whose map is larger than this')
    parser.add_argument('--cluster-range', type=int, nargs=2, default=[3, 24], metavar=('MIN', 'MAX'),
                        help='fit every k in [MIN, MAX)')
    parser.add_argument('--random-state', type=int, default=0, help='seed of the k-means initialisation and draws')
    parser.add_argument('--kmeans-batch-size', type=int, default=100, help='k-means mini-batch size (<= 1024)')
    parser.add_argument('--max-iter', type=int, default=100, help='k-means passes over the data at most')
    parser.add_argument('--n-init', type=int, default=3, help='k-means++ initialisations tried per fit')
    parser.add_argument('--init-size', type=int, default=None, help='rows of each initialisation (default 3 x batch size)')
    parser.add_argument('--reassignment-ratio', type=float, default=0.01, help='count ratio below which a centre is reassigned')
    parser.add_argument('--max-no-improvement', type=int, default=10,
                        help='stop after this many steps without a better smoothed inertia (-1: never)')
    return parser


if __name__ == '__main__':
    main(build_arg_parser().parse_args())
