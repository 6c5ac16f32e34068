"""DatasetGAN classifier training without a GPU: the pixel permutation and the stop rule of the oracle, annotation PNG
decoding, the checkpoint writer, the command line up to the device, and the argument checks `sis_pixel_train_*` make
before any CUDA call."""
import ctypes
import json

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import dataset_gan_train_oracle as to
from synthesis_in_style_b200 import _lib
from synthesis_in_style_b200 import create_dataset as cd
from synthesis_in_style_b200 import train_dataset_gan as tg
from synthesis_in_style_b200.dataset_gan import PARAM_KEYS, DatasetGANSegmenter, PixelClassifier, PixelEnsembleClassifier

COLORS = {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'}


@pytest.mark.parametrize('n', [64, 1000, 4096, 3 * 256 * 256])
def test_permutation_visits_every_pixel_once_per_epoch(n):
    key0, key1 = tg.network_key(0, 0), tg.network_key(0, 1)
    orders = {}
    for key in (key0, key1):
        for epoch in (0, 1):
            order = to.permute(key, epoch, np.arange(n), n)
            assert order.min() == 0 and order.max() == n - 1 and len(np.unique(order)) == n
            orders[key, epoch] = order
    assert not np.array_equal(orders[key0, 0], orders[key1, 0])          # networks draw their own orders
    assert not np.array_equal(orders[key0, 0], orders[key0, 1])          # and a new one every epoch
    # a step takes the next batch of its epoch's order; the trailing partial batch is dropped
    spe = n // 64
    assert np.array_equal(to.step_pixels(key0, spe - 1, n, 64), orders[key0, 0][(spe - 1) * 64:spe * 64])
    assert np.array_equal(to.step_pixels(key0, spe, n, 64), orders[key0, 1][:64])


def test_network_keys_are_pinned():
    assert tg.network_key(0, 0) == int(to.splitmix64(to.splitmix64(np.uint64(0))))
    assert len({tg.network_key(s, i) for s in range(3) for i in range(8)}) == 24


def test_stop_rule_on_a_scripted_loss_sequence():
    rule = to.StopRule(steps_per_epoch=10, epochs=100)
    losses = [5.0 - 0.01 * t for t in range(40)]         # epochs 0..3: the rule is not evaluated
    losses += [1.0, 1.5, 0.9]                            # epoch 4: best 1.0, one miss, new best 0.9 resets the count
    losses += [0.9] * 51                                 # equal is not better: the 51st miss stops
    stops = [rule.update(v) for v in losses]
    assert stops.index(True) == len(losses) - 1 == 40 + 3 + 50
    assert rule.best == 0.9 and rule.count == 51
    short = to.StopRule(steps_per_epoch=3, epochs=2)
    assert [short.update(1.0) for _ in range(6)] == [False] * 5 + [True]     # the last step of the last epoch


def test_initial_networks():
    a, b = tg.initial_network(0, 1, 3, 64), tg.initial_network(0, 1, 3, 64)
    c = tg.initial_network(0, 2, 3, 64)
    torch.testing.assert_close(a.state_dict(), b.state_dict(), rtol=0, atol=0)
    assert not torch.equal(a.layers[0].weight, c.layers[0].weight)
    sd = a.state_dict()
    assert abs(float(sd['layers.0.weight'].std()) - 0.02) < 0.002 and float(sd['layers.0.bias'].abs().max()) == 0.0
    assert float(sd['layers.2.weight'].min()) == 1.0 and float(sd['layers.2.running_var'].min()) == 1.0


def paint(path, ids, colors):
    table = np.array([[int(c[i:i + 2], 16) for i in (1, 3, 5)] for c in colors.values()], dtype=np.uint8)
    Image.fromarray(table[ids]).save(path)


def test_label_pngs_decode_to_class_ids(tmp_path):
    ids = (np.arange(16 * 16).reshape(16, 16) % 3).astype(np.uint8)
    paint(tmp_path / 'label_0000.png', ids, COLORS)
    assert np.array_equal(tg.read_label_image(tmp_path / 'label_0000.png', COLORS, 16), ids)
    rgb = np.asarray(Image.open(tmp_path / 'label_0000.png')).copy()
    rgb[5, 7] = (1, 2, 3)
    Image.fromarray(rgb).save(tmp_path / 'label_0001.png')
    with pytest.raises(ValueError, match=r'label_0001\.png: pixel \(x=7, y=5\) has colour \(1, 2, 3\)'):
        tg.read_label_image(tmp_path / 'label_0001.png', COLORS, 16)
    with pytest.raises(ValueError, match=r'label_0000\.png: the label image is 16x16, the generator makes 32x32'):
        tg.read_label_image(tmp_path / 'label_0000.png', COLORS, 32)


def test_checkpoint_loads_into_pixel_classifier_and_the_segmenter(tmp_path):
    ens = PixelEnsembleClassifier(3, 64, 0)
    for i in range(3):
        ens.set_network(f'network_{i}', tg.initial_network(7, i, 3, 64))
    tg.save_checkpoint(ens, tmp_path / 'classifier.pt')
    ckpt = torch.load(tmp_path / 'classifier.pt')
    assert sorted(ckpt) == ['network_0', 'network_1', 'network_2']
    for sd in ckpt.values():
        assert set(sd) == set(PixelClassifier(3, 64).state_dict()) and set(PARAM_KEYS) <= set(sd)
        PixelClassifier(3, 64).load_state_dict(sd)
    seg = DatasetGANSegmenter(tmp_path, 16, COLORS, classifier_path=str(tmp_path / 'classifier.pt'), feature_size=64)
    nets = list(seg.ensemble.get_networks().values())
    assert len(nets) == 3 and not nets[0].training
    torch.testing.assert_close(nets[2].layers[0].weight, ckpt['network_2']['layers.0.weight'])


class _Boundary(Exception):
    pass


def test_cli_parses_and_runs_to_the_device(tmp_path, monkeypatch):
    orig = tmp_path / 'orig.json'
    orig.write_text(json.dumps({'image_size': 32, 'latent_size': 512, 'stylegan_variant': 2}))
    creation = tmp_path / 'creation.json'
    creation.write_text(json.dumps({'segmenter_type': 'dataset_gan', 'class_to_color_map': COLORS, 'seed': 1}))
    ann = tmp_path / 'ann'
    ann.mkdir()
    torch.save({'w': torch.zeros(2, 512), 'noise': [torch.zeros(2, 1, 4, 4)]}, ann / 'latents.pt')
    for i in range(2):
        paint(ann / f'label_{i:04d}.png', np.full((32, 32), i, dtype=np.uint8), COLORS)
    reached = []

    def boundary(name):
        reached.append(name)
        raise _Boundary
    monkeypatch.setattr(cd, 'resolve_device', boundary)

    args = tg.parse_args(['random-init:0', str(creation), '-op', str(orig), '--annotations', str(ann), '-o', str(tmp_path / 'c.pt'),
                          '--num-models', '2', '--epochs', '5', '--max-steps', '100', '-d', '1'])
    assert (args.num_models, args.batch_pixels, args.epochs, args.max_steps, args.seed, args.chunk_steps) == (2, 64, 5, 100, 0, 32)
    with pytest.raises(_Boundary):
        tg.main(args)
    args = tg.parse_args(['random-init:0', str(creation), '-op', str(orig), '--write-annotation-set', '4', '-o', str(ann), '--truncate'])
    assert (args.write_annotation_set, args.seed, args.truncate, args.num_models) == (4, 1, True, 3)
    with pytest.raises(_Boundary):
        tg.main(args)
    assert reached == ['1', 'cuda']
    with pytest.raises(ValueError, match='exactly one'):
        tg.main(tg.parse_args(['random-init:0', str(creation), '-op', str(orig), '-o', str(ann)]))
    paint(ann / 'label_0001.png', np.zeros((16, 16), dtype=np.uint8), COLORS)
    with pytest.raises(ValueError, match='label_0001.png'):
        tg.main(tg.parse_args(['random-init:0', str(creation), '-op', str(orig), '--annotations', str(ann), '-o', str(tmp_path / 'c.pt')]))


def test_library_rejects_sizes_it_cannot_take():
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.sis_pixel_train_create(ctypes.byref(h), 3, 5888, 32, 64) != 0 and b'n_class' in lib.sis_last_error()
    assert lib.sis_pixel_train_create(ctypes.byref(h), 9, 5888, 4, 64) != 0 and b'networks' in lib.sis_last_error()
    assert lib.sis_pixel_train_create(ctypes.byref(h), 3, 100, 4, 64) != 0 and b'multiple of 32' in lib.sis_last_error()
    assert lib.sis_pixel_train_create(ctypes.byref(h), 3, 128, 4, 65) != 0 and b'batch' in lib.sis_last_error()
    assert lib.sis_pixel_train_create(ctypes.byref(h), 3, 128, 4, 64) == 0
    fake = (ctypes.c_void_p * 2)(16, 32)
    chans, ress = (ctypes.c_int * 2)(64, 64), (ctypes.c_int * 2)(4, 8)
    assert lib.sis_pixel_train_set_data(h, 2, fake, chans, ress, 1, 4, ctypes.c_void_p(64)) != 0
    assert b'fewer than one batch' in lib.sis_last_error()
    assert lib.sis_pixel_train_set_data(h, 2, fake, chans, ress, 1, 4096, ctypes.c_void_p(64)) == 0
    chans[1] = 32
    assert lib.sis_pixel_train_set_data(h, 2, fake, chans, ress, 1, 4096, ctypes.c_void_p(64)) != 0
    assert b'captures carry 96 features' in lib.sis_last_error()
    assert lib.sis_pixel_train_set_data(h, 2, fake, chans, ress, 1 << 16, 256, ctypes.c_void_p(64)) != 0
    assert b'exceed 2^31' in lib.sis_last_error()
    assert lib.sis_pixel_train_steps(h, 1, None) != 0 and b'prepare' in lib.sis_last_error()
    lib.sis_pixel_train_destroy(h)
