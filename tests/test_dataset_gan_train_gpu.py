"""DatasetGAN classifier training on the GPU (`sis_pixel_train_*`, csrc/dataset_gan_train.cu): step parity with the
float64 oracle (oracle/dataset_gan_train_oracle.py) on the same draws, independence of a network from the launch it
shares and from the chunk size, the device stop rule, a teacher -> student run at 256^2, and annotation set ->
training -> `create_dataset` end to end."""
import json

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import dataset_gan_oracle as dg
from oracle import dataset_gan_train_oracle as to
from synthesis_in_style_b200 import create_dataset as cd
from synthesis_in_style_b200 import train_dataset_gan as tg
from synthesis_in_style_b200.dataset_gan import PARAM_KEYS, PixelClassifier, PixelEnsembleClassifier
from synthesis_in_style_b200.model import Generator

pytestmark = pytest.mark.gpu

COLORS = {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'}
# Held-out agreement with the teacher of three networks trained 200 steps by the float64 oracle on the same draws
# (teacher_student_setup, labelled through the device labeller), measured on a B200.  The teacher labels 95.4 % of the
# held-out pixels with its majority class.
ORACLE_TEACHER_AGREEMENT = 0.95781


def synthetic_case(dev, n_images, size, layers, n_class, seed, learnable=False):
    """Random captures and noise labels, or (`learnable`) labels that a fixed linear map of the features determines."""
    g = torch.Generator().manual_seed(seed)
    acts = {i: torch.randn(n_images, c, r, r, generator=g).to(dev) for i, (c, r) in enumerate(layers)}
    labels = torch.randint(0, n_class, (n_images, size, size), generator=g, dtype=torch.uint8)
    if learnable:
        x = to.pixel_features(acts, size, np.arange(n_images * size * size))
        proj = torch.randn(x.shape[1], n_class, generator=g, dtype=torch.float64)
        labels = (x @ proj).argmax(1).to(torch.uint8).reshape(n_images, size, size)
    return acts, labels


def generator_case(dev, n_images, seed):
    torch.manual_seed(0)
    gen = Generator(256, 512, 8).to(dev).eval()
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(n_images, 512, generator=g)
    noise = [torch.randn(n_images, 1, 2 ** ((i + 5) // 2), 2 ** ((i + 5) // 2), generator=g) for i in range(gen.num_layers)]
    with torch.no_grad():
        w = gen.get_latent(z.to(dev)).cpu()
    images, acts = tg.regenerate(gen, w, noise)
    grey = images.mean(1).cpu()
    labels = torch.bucketize(grey, torch.tensor([-0.1, 0.1])).to(torch.uint8)       # three brightness classes
    return gen, acts, labels


def device_trainer(acts, labels, n_class, **kw):
    return tg.PixelEnsembleTrainer(None, labels, n_class, activations=acts, **kw)


def oracle_for(acts, labels, n_class, networks, seed=0, epochs=100, dtype=torch.float64):
    F = sum(a.shape[1] for a in acts.values())
    init = [tg.initial_network(seed, i, n_class, F).state_dict() for i in networks]
    return to.OracleTrainer(init, [tg.network_key(seed, i) for i in networks], {k: v.cpu() for k, v in acts.items()}, labels,
                            n_class, epochs=epochs, dtype=dtype)


def assert_state_close(ensemble, oracle, rtol, atol, steps):
    """Every parameter, running statistic and step count within rtol + atol of the oracle's, with two exceptions that
    fp32 against float64 cannot avoid, both bounded by the 2 * lr * steps Adam can move an element at most:
      - Adam moves an element by lr * g / (|g| + eps): where a step's nonzero gradient is within ~100 eps of zero, an
        fp32 gradient (error ~1e-9) changes that ratio visibly;
      - a first-layer output within rounding of 0 takes the other side of the ReLU, which changes that pixel's
        contribution to a row of dW1: at most 1 in 10^4 elements of a tensor."""
    lr = 1e-3
    for net, ref, min_grad in zip(ensemble.get_networks().values(), oracle.state_dicts(), oracle.min_abs_grad):
        sd = net.state_dict()
        for key in PARAM_KEYS:
            got, want = sd[key].double(), ref[key]
            diff = (got - want).abs()
            ok = diff <= atol + rtol * want.abs()
            if key in min_grad:
                bounded = diff <= 2 * lr * steps
                ok = ok | ((min_grad[key] < 1e-6) & bounded)
                flips = ~ok
                assert bool(bounded.all()) and int(flips.sum()) <= want.numel() // 10000, \
                    f'{key}: {int(flips.sum())} elements differ, max |diff| {float(diff.max()):.3g}'
            else:
                # running statistics: batch means and variances of first-layer rows the exceptions above moved
                ok = diff <= 1e-4 + rtol * want.abs()
                assert bool(ok.all()), f'{key}: {int((~ok).sum())} elements differ, max |diff| {float(diff.max()):.3g}'
        assert int(sd['layers.2.num_batches_tracked']) == int(ref['layers.2.num_batches_tracked']) == steps


CASES = {'F160': dict(layers=[(32, 8), (64, 16), (64, 32)], size=32, n_images=3),
         'F5888': None}


@pytest.fixture(scope='module', params=sorted(CASES))
def parity_case(request, cuda_device):
    if request.param == 'F5888':
        _, acts, labels = generator_case(cuda_device, 3, seed=5)
        n_class = 3
    else:
        c = CASES[request.param]
        acts, labels = synthetic_case(cuda_device, c['n_images'], c['size'], c['layers'], 4, seed=1, learnable=True)
        n_class = 4
    train = {k: v[:-1].contiguous() for k, v in acts.items()}
    held = {k: v[-1:].contiguous() for k, v in acts.items()}
    return train, labels[:-1].contiguous(), held, n_class


def test_steps_match_the_float64_oracle(parity_case):
    train, labels, held, n_class = parity_case
    oracle = oracle_for(train, labels, n_class, [0, 1])
    oracle.prefetch(200)
    done = 0
    for steps in (1, 5):
        ens, losses = device_trainer(train, labels, n_class, num_models=2).fit(max_steps=steps)
        while done < steps:
            oracle.step()
            done += 1
        assert_state_close(ens, oracle, rtol=1e-5, atol=1e-6, steps=steps)
        for m in range(2):
            np.testing.assert_allclose(losses[m], oracle.losses[m], rtol=1e-5, atol=1e-6)
    ens, losses = device_trainer(train, labels, n_class, num_models=2).fit(max_steps=200)
    # Over many steps the trajectories drift apart: Adam's sign-like steps turn last-bit differences of small gradients
    # into whole steps.  The recipe does that to itself: the same steps run in fp32 on the CPU (a twin, with other
    # summation orders than the device's) drift from the float64 oracle in the same way.  So the device must stay as close to the oracle as the twin does, with a
    # margin for the chaotic spread between two perturbed runs: the first 10 losses to 1e-4, the mean of the last 50
    # within 3x the twin's difference (+ 0.5 %), held-out labels agreeing at most 3 points less often than the twin's.
    twin = oracle_for(train, labels, n_class, [0, 1], dtype=torch.float32)
    twin.prefetch(200)
    for _ in range(200):
        twin.step()
    while done < 200:
        oracle.step()
        done += 1
    size = labels.shape[-1]
    pixels = np.random.default_rng(0).choice(size * size, min(size * size, 20000), replace=False)
    x = to.pixel_features(held, size, pixels)
    F = x.shape[1]

    def labels_of(sd):
        with torch.no_grad():
            return to.make_network({k: v.double() if v.is_floating_point() else v for k, v in sd.items()}, n_class, F).eval()(x).argmax(1)

    for m, (net, ref, twin_sd) in enumerate(zip(ens.get_networks().values(), oracle.state_dicts(), twin.state_dicts())):
        assert len(losses[m]) == 200
        np.testing.assert_allclose(losses[m][:10], oracle.losses[m][:10], rtol=1e-4)
        late, late_ref, late_twin = (float(np.mean(l[-50:])) for l in (losses[m], oracle.losses[m], twin.losses[m]))
        want = labels_of(ref)
        agree = float((labels_of(dict(net.state_dict())) == want).double().mean())
        agree_twin = float((labels_of(twin_sd) == want).double().mean())
        print(f'network {m}: mean of the last 50 losses {late:.5f}, oracle {late_ref:.5f}, twin {late_twin:.5f}; '
              f'held-out labels equal to the oracle\'s {agree:.5f}, twin {agree_twin:.5f}')
        assert abs(late - late_ref) <= 3 * abs(late_twin - late_ref) + 0.005 * late_ref
        assert agree >= agree_twin - 0.03


def test_a_network_does_not_depend_on_its_launch_or_chunk(cuda_device):
    acts, labels = synthetic_case(cuda_device, 2, 32, [(32, 8), (96, 16), (128, 32)], 5, seed=2)
    runs = {}
    for networks, chunk in (((0, 1, 2), 32), ((0, 1, 2), 1), ((1,), 32), ((1,), 1)):
        ens, losses = device_trainer(acts, labels, 5, networks=networks, chunk_steps=chunk).fit(max_steps=40)
        nets = list(ens.get_networks().values())
        runs[networks, chunk] = (nets[networks.index(1)].state_dict(), losses[networks.index(1)])
    ref_sd, ref_losses = runs[(0, 1, 2), 32]
    for (networks, chunk), (sd, losses) in runs.items():
        assert np.array_equal(losses, ref_losses), (networks, chunk)
        for key in PARAM_KEYS:
            assert torch.equal(sd[key], ref_sd[key]), (networks, chunk, key)


def test_device_stop_rule(cuda_device):
    # 256 annotated pixels, 4 steps per epoch: the rule starts at step 16.  1 x 1 captures give every pixel the same
    # features, so the loss only follows each batch's draw of noise labels and stops improving
    acts, labels = synthetic_case(cuda_device, 1, 16, [(32, 1), (32, 1)], 3, seed=3)
    ens, losses = device_trainer(acts, labels, 3, num_models=3, epochs=1000, chunk_steps=7).fit()
    for m, l in enumerate(losses):
        rule = to.StopRule(4, 1000)
        stops = [rule.update(float(v)) for v in l]
        assert stops[-1] and not any(stops[:-1]), m
        assert 16 + 51 < len(l) < 4000
        assert int(list(ens.get_networks().values())[m].state_dict()['layers.5.num_batches_tracked']) == len(l)


def teacher_student_setup(dev):
    """(generator, training captures, teacher labels, held-out captures, held-out teacher labels) at 256^2."""
    gen, acts, _ = generator_case(dev, 16, seed=11)
    F = sum(a.shape[1] for a in acts.values())
    teacher = PixelEnsembleClassifier(3, F, 0)
    for i in range(3):
        net = PixelClassifier(3, F)
        net.load_state_dict(dg.init_classifier_state(F, 3, seed=i + 1, base_seed=100))
        teacher.set_network(f'network_{i}', net.eval())
    labels = torch.cat([teacher.predict_label_images({k: v[i:i + 4] for k, v in acts.items()}, 256)[0].cpu() for i in (0, 4, 8, 12)])
    train = {k: v[:8].contiguous() for k, v in acts.items()}
    held = {k: v[8:].contiguous() for k, v in acts.items()}
    return train, labels[:8].contiguous(), held, labels[8:].contiguous()


def agreement(ensemble, held, held_labels):
    got = torch.cat([ensemble.predict_label_images({k: v[i:i + 4] for k, v in held.items()}, 256)[0].cpu() for i in (0, 4)])
    return float((got == held_labels).double().mean())


def test_student_reaches_the_oracle_agreement_with_its_teacher(cuda_device):
    train, labels, held, held_labels = teacher_student_setup(cuda_device)
    ens, losses = device_trainer(train, labels, 3, num_models=3).fit(max_steps=200)
    got = agreement(ens, held, held_labels)
    print(f'student agreement with the teacher: {got:.5f}')
    assert abs(got - ORACLE_TEACHER_AGREEMENT) <= 0.005


def test_annotation_set_to_training_to_create_dataset(cuda_device, tmp_path):
    orig = tmp_path / 'orig.json'
    orig.write_text(json.dumps({'image_size': 32, 'latent_size': 512, 'stylegan_variant': 2}))
    creation = tmp_path / 'creation.json'
    creation.write_text(json.dumps({'segmenter_type': 'dataset_gan', 'class_to_color_map': COLORS, 'seed': 1}))
    ann = tmp_path / 'ann'
    common = ['random-init:0', str(creation), '-op', str(orig)]
    out = tg.main(tg.parse_args(common + ['--write-annotation-set', '3', '-o', str(ann), '-b', '2', '--truncate']))
    assert [p.name for p in out['images']] == ['image_0000.png', 'image_0001.png', 'image_0002.png']
    saved = torch.load(ann / 'latents.pt')
    assert saved['w'].shape == (3, 512) and len(saved['noise']) == 7 and saved['noise'][-1].shape == (3, 1, 32, 32)
    # the stored W and noise regenerate the written images exactly
    gen = cd.load_generator(tg.parse_args(common + ['--annotations', str(ann), '-o', 'x']), {'image_size': 32, 'latent_size': 512},
                            cuda_device)
    images, _ = tg.regenerate(gen, saved['w'], saved['noise'], captures=False)
    from synthesis_in_style_b200.labelling import make_image
    pngs = np.stack([np.asarray(Image.open(p)) for p in out['images']])
    assert np.array_equal(make_image(images).cpu().numpy(), pngs)
    table = np.array([[0, 0, 0], [0, 0, 255], [255, 0, 0]], dtype=np.uint8)
    for i, png in enumerate(pngs):
        ids = np.digitize(png.mean(-1), [85, 170])                                 # "annotate" by brightness
        Image.fromarray(table[ids]).save(ann / f'label_{i:04d}.png')
    ckpt = tmp_path / 'classifier.pt'
    res = tg.main(tg.parse_args(common + ['--annotations', str(ann), '-o', str(ckpt), '--num-models', '2', '--max-steps', '20']))
    assert res['steps'] == [20, 20] and all(np.isfinite(res['final_loss']))
    images_out = tmp_path / 'out'
    stats = cd.main(cd.build_arg_parser().parse_args(['random-init:0', str(creation), '-op', str(orig), '-n', '4', '-b', '2',
                                                      '-s', str(images_out), '--classifier-path', str(ckpt),
                                                      '-ssd', str(tmp_path / 'sem')]))
    files = sorted(images_out.glob('**/*.png'))
    assert stats['images_kept_all_ranks'] == 4 and len(files) >= 4
    for name in ('train.json', 'val.json', 'coco_gt.json'):
        assert (images_out / name).is_file()
