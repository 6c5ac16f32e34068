"""CPU restatement of the DatasetGAN pixel-classifier training of synthesis_in_style_b200/train_dataset_gan.py
(`sis_pixel_train_*`, csrc/dataset_gan_train.cu).  TEST INFRASTRUCTURE ONLY.

The recipe follows DatasetGAN's train_interpreter.py with this project's batch order:
  - network m's order of the N = A*S*S annotated pixels in epoch e is a 4-round Feistel permutation keyed by its key
    and e, cycle-walked into [0, N) (`permute`); step t takes positions (t mod steps_per_epoch) * B .. + B - 1 of epoch
    t // steps_per_epoch, steps_per_epoch = N // B (the trailing partial batch is dropped);
  - features: dataset_gan_oracle.scale_activations of every capture, concatenated in capture order;
  - one step: nn.Sequential identical to PixelClassifier in training mode, nn.CrossEntropyLoss, torch.optim.Adam
    (lr 1e-3, betas (0.9, 0.999), eps 1e-8), in float64;
  - stop rule (`StopRule`): from epoch 4 on, count the steps whose loss is not below the best so far (reset on a new
    best); stop once the count exceeds 50, or after the last step of the last epoch.
"""
from typing import Dict, List, Sequence

import numpy
import torch
from torch import nn

from oracle.dataset_gan_oracle import scale_activations

MASK64 = numpy.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x):
    x = numpy.asarray(x, dtype=numpy.uint64)
    with numpy.errstate(over='ignore'):
        x = x + numpy.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> numpy.uint64(30))) * numpy.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> numpy.uint64(27))) * numpy.uint64(0x94D049BB133111EB)
    return x ^ (x >> numpy.uint64(31))


def half_bits(n: int) -> int:
    bits = 2
    while bits < 62 and (1 << bits) < n:
        bits += 2
    return bits // 2


def permute(key: int, epoch: int, positions, n: int) -> numpy.ndarray:
    """Pixel index at each of `positions` of the epoch's order (vectorised)."""
    half = half_bits(n)
    mask = numpy.uint64((1 << half) - 1)
    ekey = splitmix64(numpy.uint64(key) ^ splitmix64(numpy.uint64(epoch)))
    x = numpy.asarray(positions, dtype=numpy.uint64).copy()
    todo = numpy.ones(x.shape, dtype=bool)
    while todo.any():
        v = x[todo]
        left, right = v >> numpy.uint64(half), v & mask
        for rnd in range(4):
            f = splitmix64(ekey ^ (numpy.uint64(rnd) << numpy.uint64(56)) ^ right) & mask
            left, right = right, left ^ f
        x[todo] = (left << numpy.uint64(half)) | right
        todo = x >= numpy.uint64(n)
    return x.astype(numpy.int64)


def step_pixels(key: int, step: int, n: int, batch: int) -> numpy.ndarray:
    spe = n // batch
    epoch, pos = divmod(step, spe)
    return permute(key, epoch, numpy.arange(pos * batch, (pos + 1) * batch), n)


class StopRule:
    """DatasetGAN's early stop, evaluated after each optimiser step."""

    def __init__(self, steps_per_epoch: int, epochs: int, first_epoch: int = 4, patience: int = 50):
        self.spe, self.max_steps, self.first_epoch, self.patience = steps_per_epoch, epochs * steps_per_epoch, first_epoch, patience
        self.best, self.count, self.steps = 10000000.0, 0, 0

    def update(self, loss: float) -> bool:
        """Record the loss of the next step; True when the network stops after it."""
        if self.steps // self.spe >= self.first_epoch:
            if loss < self.best:
                self.best, self.count = loss, 0
            else:
                self.count += 1
        self.steps += 1
        return self.count > self.patience or self.steps >= self.max_steps


def make_network(state_dict: Dict[str, torch.Tensor], n_class: int, feature_size: int) -> nn.Sequential:
    """PixelClassifier's layers (model.py:60-86, n_class < 32) in float64, loaded from `state_dict`'s `layers.*` keys."""
    net = nn.Sequential(nn.Linear(feature_size, 128), nn.ReLU(), nn.BatchNorm1d(num_features=128), nn.Linear(128, 32), nn.ReLU(),
                        nn.BatchNorm1d(num_features=32), nn.Linear(32, n_class)).double()
    net.load_state_dict({k[len('layers.'):]: v.double() if v.is_floating_point() else v for k, v in state_dict.items()})
    return net


def state_dict_of(net: nn.Sequential) -> Dict[str, torch.Tensor]:
    return {f'layers.{k}': v.detach().clone() for k, v in net.state_dict().items()}


def pixel_features(activations: Dict[int, torch.Tensor], image_size: int, pixels: numpy.ndarray) -> torch.Tensor:
    """float64 [len(pixels), F]: the rows of scale_activations at flat pixel indices (image * S * S + y * S + x), one
    image and one capture at a time."""
    pixels = numpy.asarray(pixels, dtype=numpy.int64)
    acts = list(activations.values())
    out = torch.empty(len(pixels), sum(a.shape[1] for a in acts), dtype=torch.float64)
    plane = image_size * image_size
    for img in numpy.unique(pixels // plane):
        rows = numpy.nonzero(pixels // plane == img)[0]
        local = torch.from_numpy(pixels[rows] % plane)
        off = 0
        for i, a in enumerate(acts):
            up = scale_activations({i: a[int(img):int(img) + 1].detach().cpu().double()}, image_size)[0].reshape(plane, -1)
            out[torch.from_numpy(rows), off:off + a.shape[1]] = up[local]
            off += a.shape[1]
    return out


class OracleTrainer:
    """Trains networks from given initial state dicts on the same draws as the device trainer."""

    def __init__(self, initial: Sequence[Dict[str, torch.Tensor]], keys: Sequence[int], activations: Dict[int, torch.Tensor],
                 labels: torch.Tensor, n_class: int, batch: int = 64, epochs: int = 100, dtype=torch.float64):
        """`dtype=torch.float32` runs the same steps in fp32 (features, modules, optimiser): a twin that shows how far
        fp32 rounding alone moves the trajectory away from the float64 one."""
        self.dtype = dtype
        self.labels = labels.reshape(-1).long().cpu()
        self.n, self.batch, self.keys = self.labels.numel(), batch, list(keys)
        self.image_size = labels.shape[-1]
        self.activations = activations
        feature_size = sum(a.shape[1] for a in activations.values())
        self.nets = [make_network(sd, n_class, feature_size).to(dtype).train() for sd in initial]
        self.opts = [torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8) for net in self.nets]
        self.rules = [StopRule(self.n // batch, epochs) for _ in self.nets]
        self.done = [False] * len(self.nets)
        self.losses: List[List[float]] = [[] for _ in self.nets]
        self.loss_fn = nn.CrossEntropyLoss()
        self._features = {}
        # per network and trainable tensor: the smallest nonzero |gradient| any step saw, elementwise (where Adam's
        # g / (|g| + eps) turns the last bits of a gradient near eps into a visible change of the step)
        self.min_abs_grad = [{} for _ in self.nets]

    def _pixel_features(self, idx) -> torch.Tensor:
        rows = pixel_features(self.activations, self.image_size, idx)
        return rows.to(self.dtype)

    def prefetch(self, steps: int):
        """Compute the features of every pixel the first `steps` steps of every network draw, in one pass."""
        idx = numpy.unique(numpy.concatenate([step_pixels(k, t, self.n, self.batch) for k in self.keys for t in range(steps)]))
        idx = numpy.array([i for i in idx if int(i) not in self._features], dtype=numpy.int64)
        if len(idx):
            rows = self._pixel_features(idx)
            for i, r in zip(idx.tolist(), rows):
                self._features[i] = r

    def step(self):
        for m, (net, opt) in enumerate(zip(self.nets, self.opts)):
            if self.done[m]:
                continue
            t = self.rules[m].steps
            idx = step_pixels(self.keys[m], t, self.n, self.batch)
            missing = [int(i) for i in idx if int(i) not in self._features]
            if missing:
                for i, r in zip(missing, self._pixel_features(numpy.array(missing))):
                    self._features[i] = r
            x = torch.stack([self._features[int(i)] for i in idx])
            y = self.labels[torch.from_numpy(idx)]
            opt.zero_grad()
            loss = self.loss_fn(net(x), y)
            loss.backward()
            for name, p in net.named_parameters():
                g = p.grad.detach().abs()
                g = torch.where(g == 0, torch.full_like(g, float('inf')), g)
                key = f'layers.{name}'
                self.min_abs_grad[m][key] = torch.minimum(self.min_abs_grad[m][key], g) if key in self.min_abs_grad[m] else g.clone()
            opt.step()
            self.losses[m].append(float(loss.item()))
            self.done[m] = self.rules[m].update(float(loss.item()))

    def state_dicts(self) -> List[Dict[str, torch.Tensor]]:
        return [state_dict_of(net) for net in self.nets]
