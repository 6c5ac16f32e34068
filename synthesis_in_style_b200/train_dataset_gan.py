"""Train the DatasetGAN segmenter's pixel-classifier ensemble from annotated generated images: the input of
`create_dataset --classifier-path` with `segmenter_type: "dataset_gan"`.

1. Generate an annotation set (the generator's images, and the latents that regenerate their captures exactly):

    python -m synthesis_in_style_b200.train_dataset_gan CHECKPOINT CREATION_CONFIG.json --write-annotation-set 16 -o DIR
        [-op original_config.json] [-b 4] [-d cuda] [--truncate] [--seed 1]

   writes DIR/image_{i:04d}.png and DIR/latents.pt: {'w': fp32 [N, style_dim], the W latents after truncation,
   'noise': [fp32 [N, 1, r, r] per noise layer]}.  `--truncate` draws `mean_latent` once; storing W afterwards makes the
   set reproducible without it.
2. Paint DIR/label_{i:04d}.png (S x S, RGB) in the colours of the creation config's `class_to_color_map`; class ids
   follow the map's order, as the DatasetGAN segmenter's colour images do.  Any other colour is an error.
3. Train and write the checkpoint:

    python -m synthesis_in_style_b200.train_dataset_gan CHECKPOINT CREATION_CONFIG.json --annotations DIR -o classifier.pt
        [-op original_config.json] [-d cuda] [--num-models 3] [--batch-pixels 64] [--epochs 100] [--seed 0]
        [--max-steps N] [--chunk-steps 32]

   writes {'network_i': PixelClassifier state dict}, which `DatasetGANSegmenter.load_ensemble` reads.

The training recipe is this project's own, after DatasetGAN's published train_interpreter.py (the reference's trainer
is not part of the reference checkout, so nothing here is pinned to it): `--num-models` networks with the
`PixelClassifier` layout, initialised with init_weights('normal', 0.02); mean cross-entropy; Adam (lr 1e-3, betas
(0.9, 0.999), eps 1e-8); BatchNorm in training mode; batches of `--batch-pixels` annotated pixels, each network
drawing its own order of all pixels per epoch (a counter-based permutation, trailing partial batch dropped); at most
`--epochs` epochs, and from epoch 4 on a network stops after 51 consecutive steps without a new best loss.  The
features (every capture bilinearly upsampled to S x S and concatenated: 5888 floats per pixel at 256^2) are never
materialised: the captures of the annotated images stay on the device at native resolution and the kernels
(`sis_pixel_train_*`, csrc/dataset_gan_train.cu) gather the drawn pixels.  oracle/dataset_gan_train_oracle.py restates
the recipe in float64 with torch modules.
"""
import argparse
import ctypes
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy
import torch

from . import _lib
from . import create_dataset as cd
from .dataset_gan import PARAM_KEYS, PixelClassifier, PixelEnsembleClassifier
from .labelling import BaseDatasetSegmenter, make_image

MASK64 = (1 << 64) - 1


def _splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & MASK64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & MASK64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & MASK64
    return x ^ (x >> 31)


def network_key(seed: int, index: int) -> int:
    """Draw key of network `index` of an ensemble trained with `seed`."""
    return _splitmix64((_splitmix64(seed & MASK64) + index) & MASK64)


def initial_network(seed: int, index: int, n_class: int, feature_size: int) -> PixelClassifier:
    """Network `index` before training: init_weights('normal', 0.02) from its own seeded stream (the global RNG is left
    as it was)."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(network_key(seed, index) & ((1 << 63) - 1))
        net = PixelClassifier(n_class, feature_size)
        net.init_weights('normal', 0.02)
    return net


# ---------------------------------------------------------------------------------------------- annotation set
def draw_annotation_latents(generator, n: int, seed: int, truncate: bool, batch: int = 8):
    """(W [n, style_dim] after truncation, noise [n,1,r,r] per noise layer) on the host."""
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(n, generator.style_dim, generator=g)
    noise = [torch.randn(n, 1, 2 ** ((layer + 5) // 2), 2 ** ((layer + 5) // 2), generator=g) for layer in range(generator.num_layers)]
    dev = generator.input.input.device
    with torch.no_grad():
        w = torch.cat([generator.get_latent(z[i:i + batch].to(dev)) for i in range(0, n, batch)])
        if truncate:
            torch.manual_seed(seed)
            mean_latent = generator.mean_latent(4096)
            w = mean_latent + 0.7 * (w - mean_latent)
    return w.cpu(), noise


def regenerate(generator, w: torch.Tensor, noise: Sequence[torch.Tensor], batch: int = 4, captures: bool = True):
    """Images [N,3,S,S] and (if `captures`) every capture {layer: fp32 [N, C, r, r]}, on the generator's device."""
    dev = generator.input.input.device
    images, acts = [], []
    with torch.no_grad():
        for i in range(0, w.shape[0], batch):
            image, a = generator([w[i:i + batch].to(dev)], input_is_latent=True, noise=[n[i:i + batch].to(dev) for n in noise],
                                 return_intermediate_activations=captures)
            images.append(image)
            acts.append(a)
    joined = {k: torch.cat([a[k] for a in acts]) for k in acts[0]} if captures else None
    return torch.cat(images), joined


def write_annotation_set(generator, n: int, out_dir: Path, seed: int = 1, truncate: bool = False, batch: int = 4) -> List[Path]:
    from PIL import Image
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    w, noise = draw_annotation_latents(generator, n, seed, truncate)
    torch.save({'w': w, 'noise': noise}, out_dir / 'latents.pt')
    images, _ = regenerate(generator, w, noise, batch, captures=False)
    paths = []
    for i, img in enumerate(make_image(images).cpu().numpy()):
        paths.append(out_dir / f'image_{i:04d}.png')
        Image.fromarray(img).save(paths[-1])
    return paths


def read_label_image(path: Path, class_to_color_map: Dict, image_size: int) -> numpy.ndarray:
    """uint8 [S, S] class ids of a painted label PNG; ids follow the order of `class_to_color_map`."""
    from PIL import Image
    with Image.open(path) as im:
        rgb = numpy.asarray(im.convert('RGB'))
    if rgb.shape[:2] != (image_size, image_size):
        raise ValueError(f'{path}: the label image is {rgb.shape[1]}x{rgb.shape[0]}, the generator makes {image_size}x{image_size}')
    colors = BaseDatasetSegmenter.load_class_to_color_map(class_to_color_map)
    code = (rgb[..., 0].astype(numpy.int64) << 16) | (rgb[..., 1].astype(numpy.int64) << 8) | rgb[..., 2]
    ids = numpy.full(code.shape, 255, dtype=numpy.uint8)
    for class_id, (r, g, b) in reversed(list(enumerate(colors.values()))):     # the first class of a repeated colour wins
        ids[code == ((r << 16) | (g << 8) | b)] = class_id
    bad = numpy.argwhere(ids == 255)
    if len(bad):
        y, x = (int(v) for v in bad[0])
        raise ValueError(f'{path}: pixel (x={x}, y={y}) has colour {tuple(int(v) for v in rgb[y, x])}, which is not in '
                         f'class_to_color_map {dict(colors)}')
    return ids


def load_annotation_set(directory: Path, class_to_color_map: Dict, image_size: int):
    """(W, noise, labels uint8 [N, S, S]) of an annotation set; every image needs its label PNG."""
    directory = Path(directory)
    saved = torch.load(directory / 'latents.pt', map_location='cpu')
    w, noise = saved['w'], saved['noise']
    labels = numpy.stack([read_label_image(directory / f'label_{i:04d}.png', class_to_color_map, image_size) for i in range(w.shape[0])])
    return w, noise, torch.from_numpy(labels)


# ---------------------------------------------------------------------------------------------- training
class PixelEnsembleTrainer:
    """Trains `num_models` PixelClassifiers (or the networks `networks` of such an ensemble: network i's initial weights
    and draws depend only on (seed, i)) on the annotated pixels, on the device."""

    def __init__(self, generator, annotations: Union[str, Path, Tuple[torch.Tensor, Sequence[torch.Tensor], torch.Tensor]],
                 n_class: int, class_to_color_map: Optional[Dict] = None, num_models: int = 3, batch_pixels: int = 64,
                 epochs: int = 100, seed: int = 0, networks: Optional[Sequence[int]] = None, chunk_steps: int = 32,
                 activations: Optional[Dict[int, torch.Tensor]] = None):
        """`annotations` is an annotation directory (then `class_to_color_map` decodes its label PNGs) or (W, noise,
        labels [N, S, S]).  `activations` ({layer: fp32 [N, C, r, r]} on the device) replaces the regenerated captures
        and then `generator` may be None; `annotations` must then be the labels alone."""
        if activations is not None:
            labels = torch.as_tensor(annotations)
            acts = activations
        else:
            if isinstance(annotations, (str, Path)):
                if class_to_color_map is None:
                    raise ValueError('an annotation directory needs class_to_color_map')
                w, noise, labels = load_annotation_set(Path(annotations), class_to_color_map, generator.size)
            else:
                w, noise, labels = annotations
            if tuple(labels.shape[1:]) != (generator.size, generator.size):
                raise ValueError(f'labels are {tuple(labels.shape[1:])}, the generator makes {generator.size}x{generator.size}')
            _, acts = regenerate(generator, w, noise)
        if labels.dim() != 3 or labels.shape[1] != labels.shape[2]:
            raise ValueError(f'labels must be [N, S, S] (got {tuple(labels.shape)})')
        if int(labels.max()) >= n_class or int(labels.min()) < 0:
            raise ValueError(f'labels hold class ids outside [0, {n_class})')
        self.acts = [a.contiguous().float() for a in acts.values()]
        for t in self.acts:
            _lib.require_cuda(t, 'activation')
        self.device = self.acts[0].device
        self.labels = labels.to(self.device, torch.uint8).contiguous()
        self.n_class, self.batch_pixels, self.epochs, self.seed = n_class, batch_pixels, epochs, seed
        self.networks = list(range(num_models)) if networks is None else [int(i) for i in networks]
        self.chunk_steps = chunk_steps
        self.feature_size = sum(t.shape[1] for t in self.acts)
        self.image_size = self.labels.shape[-1]
        self.ensemble: Optional[PixelEnsembleClassifier] = None
        self.losses: List[numpy.ndarray] = []

    def fit(self, max_steps: Optional[int] = None):
        """Train from the initial weights; `max_steps` caps the steps of every network.  Returns the trained
        `PixelEnsembleClassifier` (networks in eval mode) and each network's per-step losses."""
        lib = _lib.load()
        M, F = len(self.networks), self.feature_size
        stream = _lib.current_stream_ptr(self.device)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(lib.sis_pixel_train_create(ctypes.byref(handle), M, F, self.n_class, self.batch_pixels))
            try:
                for m, index in enumerate(self.networks):
                    sd = initial_network(self.seed, index, self.n_class, F).state_dict()
                    for key in PARAM_KEYS:
                        t = sd[key].detach().float().contiguous()
                        _lib.check(lib.sis_pixel_train_set_param(handle, m, key.encode(), ctypes.c_void_p(t.data_ptr()), t.numel()))
                n = len(self.acts)
                ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in self.acts])
                chans = (ctypes.c_int * n)(*[t.shape[1] for t in self.acts])
                ress = (ctypes.c_int * n)(*[t.shape[-1] for t in self.acts])
                _lib.check(lib.sis_pixel_train_set_data(handle, n, ptrs, chans, ress, self.labels.shape[0], self.image_size,
                                                        _lib.ptr(self.labels)))
                keys = (ctypes.c_uint64 * M)(*[network_key(self.seed, i) for i in self.networks])
                _lib.check(lib.sis_pixel_train_prepare(handle, keys, self.epochs, stream))
                done = (ctypes.c_int32 * M)()
                steps_done = (ctypes.c_int64 * M)()
                issued = 0
                while max_steps is None or issued < max_steps:
                    chunk = self.chunk_steps if max_steps is None else min(self.chunk_steps, max_steps - issued)
                    _lib.check(lib.sis_pixel_train_steps(handle, chunk, stream))
                    issued += chunk
                    _lib.check(lib.sis_pixel_train_status(handle, done, steps_done, stream))      # once per chunk
                    if all(done):
                        break
                ensemble = PixelEnsembleClassifier(self.n_class, F, 0)
                self.losses = []
                for m in range(M):
                    net = PixelClassifier(self.n_class, F)
                    sd = net.state_dict()
                    for key in PARAM_KEYS:
                        out = torch.empty_like(sd[key], dtype=torch.float32).contiguous()
                        _lib.check(lib.sis_pixel_train_read_param(handle, m, key.encode(), ctypes.c_void_p(out.data_ptr()),
                                                                  out.numel(), stream))
                        sd[key] = out
                    sd['layers.2.num_batches_tracked'] = torch.tensor(steps_done[m])
                    sd['layers.5.num_batches_tracked'] = torch.tensor(steps_done[m])
                    net.load_state_dict(sd)
                    net.eval()
                    ensemble.set_network(f'network_{m}', net)
                    losses = numpy.empty(steps_done[m], dtype=numpy.float32)
                    _lib.check(lib.sis_pixel_train_read_losses(handle, m, ctypes.c_void_p(losses.ctypes.data), len(losses), stream))
                    self.losses.append(losses)
            finally:
                lib.sis_pixel_train_destroy(handle)
        self.ensemble = ensemble
        return ensemble, self.losses

    def save(self, path: Union[str, Path]):
        """{'network_i': state dict} with the keys of PixelClassifier, as DatasetGANSegmenter.load_ensemble reads it."""
        if self.ensemble is None:
            raise RuntimeError('call fit() first')
        save_checkpoint(self.ensemble, path)


def save_checkpoint(ensemble: PixelEnsembleClassifier, path: Union[str, Path]):
    torch.save({f'network_{i}': net.state_dict() for i, net in enumerate(ensemble.get_networks().values())}, str(path))


# ---------------------------------------------------------------------------------------------- command line
def main(args: argparse.Namespace) -> Dict:
    import json
    ckpt = str(args.checkpoint)
    config = cd.load_config(None if ckpt.startswith('random-init:') else ckpt, args.original_config_path)
    with open(args.config) as f:
        creation_config = json.load(f)
    class_to_color_map = creation_config['class_to_color_map']
    if (args.write_annotation_set is None) == (args.annotations is None):
        raise ValueError('give exactly one of --write-annotation-set N and --annotations DIR')
    annotations = None
    if args.annotations is not None:
        annotations = load_annotation_set(args.annotations, class_to_color_map, config['image_size'])
    device = cd.resolve_device(args.device)
    with torch.cuda.device(device):
        generator = cd.load_generator(args, config, device)
        if args.write_annotation_set is not None:
            paths = write_annotation_set(generator, args.write_annotation_set, args.output, seed=args.seed, truncate=args.truncate,
                                         batch=args.batch_size)
            return {'images': paths}
        trainer = PixelEnsembleTrainer(generator, annotations, len(class_to_color_map), num_models=args.num_models,
                                       batch_pixels=args.batch_pixels, epochs=args.epochs, seed=args.seed,
                                       chunk_steps=args.chunk_steps)
        _, losses = trainer.fit(args.max_steps)
        trainer.save(args.output)
    return {'checkpoint': Path(args.output), 'steps': [len(l) for l in losses],
            'final_loss': [float(l[-1]) if len(l) else None for l in losses]}


def build_arg_parser() -> argparse.ArgumentParser:
    parser = argparse.ArgumentParser(description='Write an annotation set of generated images, or train the DatasetGAN '
                                                 'pixel-classifier ensemble on an annotated one.')
    parser.add_argument('checkpoint', help='Path to the trained autoencoder/generator, or random-init:<seed>')
    parser.add_argument('config', help='creation config (JSON) whose class_to_color_map the labels are painted in')
    parser.add_argument('-op', '--original-config-path', type=Path, default=None,
                        help='YAML/JSON config of the original training, if it is not in a sibling directory of the checkpoint')
    parser.add_argument('-o', '--output', type=Path, required=True,
                        help='annotation directory (with --write-annotation-set) or checkpoint file (with --annotations)')
    parser.add_argument('--write-annotation-set', type=int, default=None, metavar='N', help='generate N images to annotate')
    parser.add_argument('--annotations', type=Path, default=None, help='annotated set to train on')
    parser.add_argument('-b', '--batch-size', default=4, type=int, help='batch size for generation of images on GPU')
    parser.add_argument('-d', '--device', default='cuda', help='CUDA device to use, either any (cuda) or the id of the device')
    parser.add_argument('--truncate', action='store_true', default=False, help='Use truncation trick during generation')
    parser.add_argument('--seed', type=int, default=None,
                        help='seed of the latents (default 1) or of the networks\' initialisation and draws (default 0)')
    parser.add_argument('--num-models', type=int, default=3, help='networks of the ensemble')
    parser.add_argument('--batch-pixels', type=int, default=64, help='annotated pixels per step (2..64)')
    parser.add_argument('--epochs', type=int, default=100, help='passes over the annotated pixels at most')
    parser.add_argument('--max-steps', type=int, default=None, help='stop every network after this many steps')
    parser.add_argument('--chunk-steps', type=int, default=32, help='steps enqueued between two reads of the stop words')
    return parser


def parse_args(argv=None) -> argparse.Namespace:
    args = build_arg_parser().parse_args(argv)
    if args.seed is None:
        args.seed = 1 if args.write_annotation_set is not None else 0
    return args


if __name__ == '__main__':
    main(parse_args())
