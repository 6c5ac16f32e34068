"""`create_dataset_for_segmentation.py` on the B200 path: the reference's command line, creation JSON, dispatch on
`segmenter_type`, output tree and ground-truth files, with the per-batch GPU work done by libsis_b200.

Mirrors scf/create_dataset_for_segmentation.py
  :52-81    get_dataset_segmenter          dispatch on creation_config['segmenter_type']
  :109-148  build_dataset                  generate -> create_segmentation_image -> make_image -> drop -> save, running ids
  :169-206  main                           train.json / val.json (90 / 10 after a seeded shuffle) and coco_gt.json
  :209-242  the argument parser            same flags, same defaults
and scf/utils/config.py:12-58 (`load_config`), scf/utils/dataset_creation.py:10-29 (`get_base_dirs`),
scf/networks/__init__.py:24-31,413-423 (`load_weights`, `load_autoencoder_or_generator`: 'autoencoder' / 'g_ema' keys).

    python -m synthesis_in_style_b200.create_dataset CHECKPOINT CREATION_CONFIG.json -n 100000 -b 32 --num-clusters 20 \\
        -ssd <run>/semantic_segmentation [-s OUT] [--truncate] [-op original_config.json]
    torchrun --nproc-per-node 8 -m synthesis_in_style_b200.create_dataset ...     # batch-index sharded over the GPUs

Only the generator half of the reference's autoencoder is built (the script never encodes: `build_latent_and_noise_generator`
yields `Latents`).  Extension: a CHECKPOINT of the form `random-init:<seed>` builds seeded random weights instead of
reading a file (synthetic runs and tests; `-op` must then name the original config).  Multi-GPU runs reproduce the
reference's global running ids (dataset_writer.assign_round_ids); rank 0 writes the JSON files after a barrier.
"""
import argparse
import json
import os
import random
from pathlib import Path
from typing import Dict, Optional, Tuple

import numpy
import torch

from . import dataset_creation as dc
from . import dataset_writer as dw
from .coco_gt import COCOGtCreator, iter_through_images_in
from .labelling import BaseDatasetSegmenter, ClusterSegmenter, make_image
from .model import Generator


# ---------------------------------------------------------------------------------------------- config / paths
def load_config(checkpoint_path: Optional[str] = None, config_path=None) -> dict:
    """utils/config.py:48-58: the original training config, from `-op` (JSON / YAML) or from `<run>/config/` next to the
    checkpoint (`config.json` updated with `args.json`)."""
    if checkpoint_path is None and config_path is None:
        raise RuntimeError('You have to supply either checkpoint path or path to a config file!')
    if config_path is not None:
        config_path = Path(config_path)
        with config_path.open() as f:
            if config_path.suffix == '.json':
                return json.load(f)
            if config_path.suffix == '.yaml':
                import yaml
                return yaml.safe_load(f)
            raise NotImplementedError
    config_dir = Path(checkpoint_path).parent.parent / 'config'
    try:
        with open(config_dir / 'config.json') as f:
            config = json.load(f)
        with open(config_dir / 'args.json') as f:
            config.update(json.load(f))
    except FileNotFoundError as err:
        raise FileNotFoundError('When trying to load a model form a checkpoint assert that the original configs are in ../config. '
                                'Otherwise use the corresponding flag to pass the original config directly.') from err
    return config


def get_base_dirs(args: argparse.Namespace) -> Tuple[Path, Path]:
    """utils/dataset_creation.py:16-29."""
    if getattr(args, 'semantic_segmentation_base_dir', None) is None:
        base_dir = Path(args.checkpoint).parent.parent
        semantic_segmentation_base_dir = base_dir / 'semantic_segmentation'
    else:
        semantic_segmentation_base_dir = Path(args.semantic_segmentation_base_dir)
        base_dir = semantic_segmentation_base_dir.parent
    image_save_base_dir = base_dir / 'generated_images' if args.save_to is None else Path(args.save_to)
    image_save_base_dir.mkdir(parents=True, exist_ok=True)
    return image_save_base_dir, semantic_segmentation_base_dir


def resolve_device(name: str) -> torch.device:
    """`-d cuda` = this rank's GPU (LOCAL_RANK under torchrun), or an explicit device id."""
    if not torch.cuda.is_available():
        raise RuntimeError('create_dataset needs a CUDA device (libsis_b200 has no CPU path)')
    if name == 'cuda':
        return torch.device('cuda', int(os.environ.get('LOCAL_RANK', '0')))
    return torch.device('cuda', int(name)) if str(name).isdigit() else torch.device(name)


# ---------------------------------------------------------------------------------------------- model / segmenter
def load_generator(args: argparse.Namespace, config: dict, device) -> Generator:
    """The decoder of `load_autoencoder_or_generator` (networks/__init__.py:413-423): the StyleGAN2 generator
    (`stylegan_variant` 2, the default) or the SWAGAN generator (`'swagan'`) of `config['image_size']` /
    `config['latent_size']`, weights from the checkpoint's 'autoencoder' entry (its `decoder.*` keys) when the config
    names a `stylegan_checkpoint`, else from 'g_ema'."""
    variant = config.get('stylegan_variant', 2)
    if variant == 2:
        cls = Generator
    elif variant == 'swagan':
        from .swagan import Generator as cls
    else:
        raise NotImplementedError(f'stylegan_variant {variant!r}: the B200 hot path has the StyleGAN2 and SWAGAN generators')
    ckpt = str(args.checkpoint)
    if ckpt.startswith('random-init:'):
        torch.manual_seed(int(ckpt.split(':', 1)[1]))
        return cls(config['image_size'], config['latent_size'], 8, channel_multiplier=2).to(device).eval()
    generator = cls(config['image_size'], config['latent_size'], 8, channel_multiplier=2)
    weights = torch.load(ckpt, map_location='cpu')
    if 'stylegan_checkpoint' in config:
        weights = weights['autoencoder'] if 'autoencoder' in weights else weights
        weights = {k[len('decoder.'):]: v for k, v in weights.items() if k.startswith('decoder.')}
    elif 'g_ema' in weights:
        weights = weights['g_ema']
    generator.load_state_dict(weights)
    return generator.to(device).eval()


def get_dataset_segmenter(args: argparse.Namespace, creation_config: dict, image_size: int,
                          semantic_segmentation_base_dir: Path) -> BaseDatasetSegmenter:
    """create_dataset_for_segmentation.py:52-81."""
    common = dict(base_dir=semantic_segmentation_base_dir, image_size=image_size,
                  class_to_color_map=creation_config['class_to_color_map'])
    if creation_config['segmenter_type'] == 'black_white_handwritten_printed':
        assert 'only_keep_overlapping' in creation_config, 'The key "only_keep_overlapping" must be specified in the config file.'
        return ClusterSegmenter(keys_to_merge=creation_config['keys_to_merge'],
                                only_keep_overlapping=creation_config['only_keep_overlapping'],
                                keys_for_class_determination=creation_config['keys_for_class_determination'],
                                keys_for_finegrained_segmentation=creation_config['keys_for_finegrained_segmentation'],
                                num_clusters=args.num_clusters, min_class_contour_area=creation_config['min_class_contour_area'],
                                **common)
    if creation_config['segmenter_type'] == 'dataset_gan':
        from .dataset_gan import DatasetGANSegmenter
        return DatasetGANSegmenter(classifier_path=args.classifier_path, feature_size=creation_config['feature_size'],
                                   upsamplers=creation_config['upsamplers'], **common)
    raise NotImplementedError


def get_dataset_gan_params(generator: Generator, mean_latent, creation_config: dict, image_size: int, latent_size: int) -> dict:
    """:28-49: one probe forward to learn the feature size and build the per-capture upsamplers."""
    from .dataset_gan import get_dataset_gan_params as params_from
    device = generator.input.input.device
    latent = dc.Latents(torch.randn(1, latent_size), generator.make_noise())
    activations, _ = dc.generate_images(latent, generator, device=device, mean_latent=mean_latent)
    creation_config.update(params_from(activations, image_size))
    return creation_config


# ---------------------------------------------------------------------------------------------- the loop
def _world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def build_dataset(args: argparse.Namespace, creation_config: Dict, original_config_path: Optional[Path] = None,
                  debug: bool = False) -> Dict:
    """:109-148.  The cluster-based segmenter runs on the pipelined path (GPU: generate + label, two batches in flight;
    host pools: contour stage and PNG encoding); the DatasetGAN segmenter labels on the GPU and only encodes PNGs on
    the host.  Returns the counters of `dataset_writer.build_dataset`."""
    from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor
    import multiprocessing
    config = load_config(args.checkpoint if not str(args.checkpoint).startswith('random-init:') else None, original_config_path)
    config['batch_size'] = args.batch_size
    image_save_base_dir, semantic_segmentation_base_dir = get_base_dirs(args)
    device = resolve_device(args.device)
    rank, world = _world()
    with torch.cuda.device(device):
        generator = load_generator(args, config, device)
        mean_latent = None
        if args.truncate:
            with torch.no_grad():
                mean_latent = generator.mean_latent(4096)
            if world > 1:      # the reference draws it unseeded in one process: every rank must use rank 0's
                import torch.distributed as dist
                dist.broadcast(mean_latent, src=0)
        if creation_config['segmenter_type'] == 'dataset_gan':
            creation_config = get_dataset_gan_params(generator, mean_latent, creation_config, config['image_size'], config['latent_size'])
        segmenter = get_dataset_segmenter(args, creation_config, config['image_size'], semantic_segmentation_base_dir)
        cores = max(2, (os.cpu_count() or 2) // world)
        with ThreadPoolExecutor(max(1, cores * 3 // 4)) as png_pool:       # its size = the native writer's encoder threads
            if isinstance(segmenter, ClusterSegmenter) and not debug:
                spawn = multiprocessing.get_context('spawn')      # the workers only run OpenCV / numpy: never fork a CUDA process
                pipe = dc.LabelledPairGenerator(generator, segmenter, config, seed=creation_config['seed'], mean_latent=mean_latent,
                                                rank=rank, world_size=world, capture_only_labelled=True, in_flight=2)
                if pipe.device_contours_supported():
                    # contour stage on the device: the pool only serves the few images that fall back to the host path
                    with ProcessPoolExecutor(max(1, cores // 4), mp_context=spawn) as contour_pool:
                        return dw.build_dataset(pipe, image_save_base_dir, args.num_images, contour_pool, png_pool, device_contours=True)
                with ProcessPoolExecutor(max(1, cores * 3 // 4), mp_context=spawn) as contour_pool:
                    return dw.build_dataset(pipe, image_save_base_dir, args.num_images, contour_pool, png_pool, device_contours=False)
            # generic loop (:127-148): any segmenter with create_segmentation_image; `debug` keeps dropped images
            writer = dw.DatasetWriter(image_save_base_dir, args.num_images, rank, world, png_pool, device=device if world > 1 else None)
            batches = 0
            for _, batch in dc.sharded_latent_stream(generator, config, creation_config['seed'], rank, world):
                activations, generated_images = dc.generate_images(batch, generator, device=device, mean_latent=mean_latent)
                label_images, image_ids_to_drop = segmenter.create_segmentation_image(activations)
                images = make_image(generated_images).cpu().numpy()
                writer.add(images, numpy.asarray(label_images), [] if debug else image_ids_to_drop)
                batches += 1
                if writer.finished:
                    break
            writer.flush()
            return {'images_kept_all_ranks': writer.n, 'files_written_this_rank': writer.files_written, 'batches_this_rank': batches}


def create_dataset_json_data(image_paths, image_root: Path, gt_creator: COCOGtCreator):
    """:151-166: [{'file_name', 'has_<class>'...}] and whether every image could be read."""
    from PIL import Image
    dataset_data = []
    try:
        for image_path in image_paths:
            with Image.open(str(image_path)) as the_image:
                data = {'file_name': str(Path(image_path).relative_to(image_root))}
                data.update(gt_creator.determine_classes_in_image(the_image))
            dataset_data.append(data)
    except Exception:
        import traceback
        print(traceback.format_exc())
        return dataset_data, False
    return dataset_data, True


def main(args: argparse.Namespace) -> Optional[Dict]:
    """:169-206."""
    import torch.distributed as dist
    with open(args.config) as f:
        config = json.load(f)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=resolve_device(args.device))
    stats = None
    if not args.only_create_train_val_split:
        stats = build_dataset(args, config, original_config_path=args.original_config_path, debug=args.debug)
    if world > 1:
        dist.barrier()
    rank, _ = _world()
    if args.debug or rank != 0:
        return stats                                   # no need for gt if only creating debug images
    image_save_base_dir, _ = get_base_dirs(args)
    generated_images = list(iter_through_images_in(image_save_base_dir))
    random.seed(config['seed'])
    random.shuffle(generated_images)
    coco_creator = COCOGtCreator(config['class_to_color_map'], image_root=image_save_base_dir)
    split_index = int(len(generated_images) * 0.9)      # 10 % validation data
    training_images, validation_images = generated_images[:split_index], generated_images[split_index:]
    for name, part in (('train.json', training_images), ('val.json', validation_images)):
        gt, success = create_dataset_json_data(part, image_save_base_dir, coco_creator)
        with (image_save_base_dir / (name if success else name + '.part')).open('w') as f:
            json.dump(gt, f)
    with (image_save_base_dir / 'coco_gt.json').open('w') as f:
        json.dump(coco_creator.create_coco_gt_from_image_paths(validation_images), f)
    return stats


def build_arg_parser() -> argparse.ArgumentParser:
    """:209-238, flag for flag."""
    parser = argparse.ArgumentParser(description='Generate a synthetic dataset using a trained StyleGAN model and the '
                                                 'labelled intermediate layers specified in a config file.')
    parser.add_argument('checkpoint', help='Path to trained autoencoder/generator for dataset creation')
    parser.add_argument('config', help='path to json file containing config for generation')
    parser.add_argument('-op', '--original-config-path', type=Path, default=None,
                        help='Path to the YAML/JSON file that contains the config for the original segmenter training. Has to be '
                             'provided if the config does not lie in a sibling directory of the checkpoint.')
    parser.add_argument('-n', '--num-images', type=int, default=100, help='Number of images to generate')
    parser.add_argument('-s', '--save-to', help='path where to save generated images (default is save in dir of run of used checkpoint)')
    parser.add_argument('-b', '--batch-size', default=10, type=int, help='batch size for generation of images on GPU')
    parser.add_argument('-d', '--device', default='cuda', help='CUDA device to use, either any (cuda) or the id of the device')
    parser.add_argument('--only-create-train-val-split', action='store_true', default=False,
                        help='do not create an entire dataset, rather use the save_path and build a train validation split with '
                             'according COCO GT')
    parser.add_argument('--debug', action='store_true', default=False, help='render debug output during image generation')
    parser.add_argument('--truncate', action='store_true', default=False, help='Use truncation trick during generation')
    parser.add_argument('--num-clusters', type=int, default=-1,
                        help='The number of classes labelled with semantic labeler. Only used with cluster-based segmenters.')
    parser.add_argument('--classifier-path', help='Path to the trained activation classifier. Only used with DatasetGAN segmenters.')
    parser.add_argument('-ssd', '--semantic-segmentation-base-dir', type=Path,
                        help='If a different directory for creating the semantic segmentation was chosen use this flag to provide it')
    return parser


if __name__ == '__main__':
    main(build_arg_parser().parse_args())
