"""SWAGAN on the fused plan (`sis_generator_create_swagan`, `sis_wavelet_to_rgb`): CPU checks of the plan's shapes and of
`create_dataset.load_generator` with `stylegan_variant: 'swagan'`; on the GPU the one-pass wavelet ToRGB against the
oracle's `to_rgb`, the plan against the oracle at 256^2, in-forward labelling, the launch schedule, the labelled-pair
pipeline and `create_dataset.main` end to end."""
import ctypes
import json
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import labelling_oracle as lo
from oracle import stylegan2_oracle as so
from oracle import swagan_oracle as sw
from synthesis_in_style_b200 import _lib, labelling, swagan
from synthesis_in_style_b200 import create_dataset as cd

NAMES = {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'}
CLASS_MAP = {'0': 'background', '1': 'printed_text', '2': 'handwritten_text', '3': 'background'}


# ------------------------------------------------------------------------------------------------------------ CPU
def test_create_swagan_checks_size_and_reports_the_oracle_shapes():
    lib = _lib.load()
    h = ctypes.c_void_p()
    for bad in (8, 24, 100, 2048):
        assert lib.sis_generator_create_swagan(bad, 64, 2, 2, ctypes.byref(h)) != 0
        assert b'power of two in [16, 1024]' in lib.sis_last_error()
    assert lib.sis_generator_create_swagan(32, 64, 2, 2, ctypes.byref(h)) == 0
    spec = sw.SwaganSpec(32, 64, 2)
    assert lib.sis_generator_n_latent(h) == spec.n_latent == 6 and lib.sis_generator_num_layers(h) == spec.num_layers == 5
    g = swagan.Generator(32, 64, 2)
    c, r = ctypes.c_int(), ctypes.c_int()
    for idx in range(spec.n_latent):
        assert lib.sis_generator_activation_shape(h, idx, ctypes.byref(c), ctypes.byref(r)) == 0
        res = 4 if idx <= 1 else 2 ** ((idx - 2) // 2 + 3)
        assert (c.value, r.value) == (spec.channels[res], res) == g.activation_shape(idx)
    assert lib.sis_generator_activation_shape(h, spec.n_latent, ctypes.byref(c), ctypes.byref(r)) != 0
    assert lib.sis_generator_destroy(h) == 0


def test_load_generator_builds_swagan(tmp_path):
    config = {'image_size': 32, 'latent_size': 64, 'stylegan_variant': 'swagan'}
    g = cd.load_generator(Namespace(checkpoint='random-init:0'), config, 'cpu')
    assert isinstance(g, swagan.Generator) and g.size == 32 and g.n_latent == 6
    ref = sw.init_state_dict(sw.SwaganSpec(32, 64, 8), seed=0)
    sd = g.state_dict()
    assert set(sd) == set(ref)
    assert all(torch.equal(sd[k], ref[k]) for k in ref)
    # a saved g_ema checkpoint, and an autoencoder checkpoint with decoder.* keys, round-trip
    want = so.perturb_zero_params(sw.init_state_dict(sw.SwaganSpec(32, 64, 8), seed=3), seed=7)
    torch.save({'g_ema': want}, tmp_path / 'g.pt')
    torch.save({'autoencoder': {**{f'decoder.{k}': v for k, v in want.items()}, 'encoder.w': torch.zeros(1)}}, tmp_path / 'ae.pt')
    for path, cfg in ((tmp_path / 'g.pt', config), (tmp_path / 'ae.pt', dict(config, stylegan_checkpoint='x'))):
        got = cd.load_generator(Namespace(checkpoint=str(path)), cfg, 'cpu').state_dict()
        assert set(got) == set(want) and all(torch.equal(got[k], want[k]) for k in want)
    for variant in (1, 3, 'stylegan1'):
        with pytest.raises(NotImplementedError):
            cd.load_generator(Namespace(checkpoint='random-init:0'), dict(config, stylegan_variant=variant), 'cpu')


# ------------------------------------------------------------------------------------------------------------ GPU
def close(got, want, tol):
    want = want.detach().cpu()
    return float((got.detach().cpu() - want).abs().max()) <= tol * max(1.0, float(want.abs().max()))


@pytest.mark.gpu
@pytest.mark.parametrize('res', [4, 8, 16, 64, 128])
@pytest.mark.parametrize('with_skip', [False, True])
def test_wavelet_to_rgb_matches_oracle(cuda_device, res, with_skip):
    cin = {4: 512, 8: 512, 16: 512, 64: 512, 128: 256}[res]
    torch.manual_seed(res)
    m = swagan.ToRGB(cin, 64, upsample=True)
    with torch.no_grad():
        m.bias.normal_(0, 0.1)
        m.conv.modulation.bias.add_(torch.randn(cin) * 0.1)
    sd = {f't.{k}': v.clone() for k, v in m.state_dict().items()}
    x, style = torch.randn(3, cin, res, res), torch.randn(3, 64)
    skip = torch.randn(3, 12, res // 2, res // 2) if with_skip else None
    want = sw.to_rgb(sd, 't', x, style, skip)
    m = m.to(cuda_device)
    with torch.no_grad():
        got = m(x.to(cuda_device), style.to(cuda_device), skip.to(cuda_device) if with_skip else None)
    assert got.shape == want.shape == (3, 12, res, res)
    assert close(got, want, 1e-5), float((got.cpu() - want).abs().max())


@pytest.fixture(scope='module')
def plan256():
    spec = sw.SwaganSpec(256, 512, 8)
    sd = so.perturb_zero_params(sw.init_state_dict(spec, seed=0), seed=1234)
    gen = torch.Generator().manual_seed(11)
    z, z2 = torch.randn(2, 512, generator=gen), torch.randn(2, 512, generator=gen)
    noise = [torch.randn(n.shape, generator=gen) for n in sw.make_noise(spec)]
    ml = so.style_mlp(sd, spec, torch.randn(64, 512, generator=gen)).mean(0, keepdim=True)
    wplus = torch.randn(2, spec.n_latent, 512, generator=gen)
    cases = {'plain': dict(styles=[z], noise=noise),
             'truncmix': dict(styles=[z, z2], noise=noise, inject_index=5, truncation=0.7, truncation_latent=ml),
             'wplus': dict(styles=[wplus], noise=noise, input_is_latent=True),
             'fixed_noise': dict(styles=[z], randomize_noise=False)}
    want = {name: sw.generator_forward(sd, spec, return_intermediate_activations=True, **kw) for name, kw in cases.items()}
    want['latents'] = sw.generator_forward(sd, spec, return_latents=True, **cases['truncmix'])
    return spec, sd, cases, want


def to_dev(kw, dev):
    out = {}
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            v = v.to(dev)
        elif isinstance(v, list):
            v = [t.to(dev) for t in v]
        out[k] = v
    return out


def make_swagan(sd, size, dev, precision='bf16x3'):
    g = swagan.Generator(size, 512, 8, precision=precision)
    g.load_state_dict(sd)
    return g.to(dev).eval()


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'bf16x3'])
def test_plan_matches_oracle_at_256(cuda_device, plan256, precision):
    spec, sd, cases, want = plan256
    g = make_swagan(sd, 256, cuda_device, precision)
    tol = 2e-4 if precision == 'fp32' else 2e-3
    for name, kw in cases.items():
        with torch.no_grad():
            img, acts = g(return_intermediate_activations=True, **to_dev(kw, cuda_device))
        g.check()
        want_img, want_acts = want[name]
        assert img.shape == (2, 3, 256, 256)
        assert close(img, want_img, tol), (name, float((img.cpu() - want_img).abs().max()))
        assert sorted(acts) == list(range(spec.n_latent))
        for k, a in acts.items():
            assert close(a, want_acts[k], tol), (name, k)
    with torch.no_grad():
        img, latent = g(return_latents=True, **to_dev(cases['truncmix'], cuda_device))
    assert close(img, want['latents'][0], tol) and close(latent, want['latents'][1], tol)


def make_segmenter(g, size, layers):
    gen = torch.Generator().manual_seed(5)
    cents = {}
    for layer in layers:
        c, _ = g.activation_shape(int(layer))
        cents[layer] = torch.nn.functional.normalize(torch.randn(4, c, generator=gen), dim=1)
    seg = labelling.ClusterSegmenter(None, size, NAMES, keys_for_class_determination=layers[:2], keys_for_finegrained_segmentation=layers[2:],
                                     num_clusters=4, keys_to_merge={}, catalog={k: labelling.FactorCatalog(4, v) for k, v in cents.items()},
                                     class_label_map={k: CLASS_MAP for k in layers})
    return seg, cents


@pytest.mark.gpu
def test_in_forward_labelling_equals_separate_labelling_and_oracle(cuda_device, plan256):
    spec, sd, cases, want = plan256
    g = make_swagan(sd, 256, cuda_device)
    layers = ['8', '9', '10', '11']
    seg, cents = make_segmenter(g, 256, layers)
    jobs = seg.make_label_jobs(g, 2, want_margin=True)
    with torch.no_grad():
        _, acts = g(return_intermediate_activations=True, capture_layers=[int(l) for l in layers], label_jobs=jobs,
                    **to_dev(cases['plain'], cuda_device))
    g.check()
    assert sorted(acts) == [8, 9, 10, 11]
    _, want_acts = want['plain']
    total = agree = 0
    for job in jobs:
        layer = job.activation_idx
        hist = torch.zeros_like(job.hist)
        _, sep = labelling.label_assign(acts[layer], job.centroids, job.class_bits, job.n_class, job.image_size, want_ids_u8=True,
                                        hist=hist)
        assert torch.equal(sep['ids_u8'], job.ids_u8) and torch.equal(sep['masks'], job.masks) and torch.equal(hist, job.hist), layer
        assert job.masks.shape[-1] == 256
        ids_want, margin = lo.predict_with_margin(want_acts[layer], cents[str(layer)])
        ids_got = job.ids_u8.cpu().long()
        safe = margin > 1e-3
        assert torch.equal(ids_got[safe], ids_want[safe]), layer
        total += ids_want.numel()
        agree += int((ids_got == ids_want).sum())
    assert agree / total >= 0.999


@pytest.mark.gpu
def test_one_wavelet_to_rgb_launch_per_resolution(cuda_device, plan256):
    spec, sd, cases, _ = plan256
    g = make_swagan(sd, 256, cuda_device)
    kw = to_dev(cases['plain'], cuda_device)
    with torch.no_grad():
        g(**kw)
    torch.cuda.synchronize()
    _lib.profile_collect()
    _lib.profile_enable(True)
    try:
        with torch.no_grad(), torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            g(**kw)
            torch.cuda.synchronize()
        counts = _lib.profile_collect()
    finally:
        _lib.profile_enable(False)
    assert spec.log_size - 1 == 6 and counts['torgb'][1] == 6
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert sum('wavelet_torgb' in n for n in names) == 6
    assert not any('upfirdn' in n or 'torgb' in n.replace('wavelet_torgb', '') for n in names), sorted(set(names))


def pipeline_setup(dev):
    spec = sw.SwaganSpec(32, 512, 8)
    sd = so.perturb_zero_params(sw.init_state_dict(spec, seed=0), seed=1234)
    g = make_swagan(sd, 32, dev)
    layers = ['2', '3', '4', '5']
    seg, _ = make_segmenter(g, 32, layers)
    return g, seg, layers


@pytest.mark.gpu
def test_sharded_swagan_run_equals_single_stream(cuda_device):
    from synthesis_in_style_b200 import dataset_creation as dc
    g, seg, layers = pipeline_setup(cuda_device)
    cfg = {'batch_size': 3, 'latent_size': 512}
    single = [b for _, b in zip(range(6), dc.LabelledPairGenerator(g, seg, cfg, seed=1))]
    for rank in range(2):
        pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, rank=rank, world_size=2, capture_only_labelled=True)
        for _, b in zip(range(3), pipe):
            ref_b = single[b.batch_index]
            assert b.batch_index % 2 == rank and b.image.shape == (3, 3, 32, 32)
            assert torch.equal(b.image, ref_b.image)
            for layer in layers:
                assert torch.equal(b.ids[layer], ref_b.ids[layer])
                for cn in NAMES:
                    assert torch.equal(b.masks[layer][cn], ref_b.masks[layer][cn])


@pytest.mark.gpu
def test_two_swagan_batches_in_flight_equal_single_stream(cuda_device):
    from synthesis_in_style_b200 import dataset_creation as dc
    g, seg, layers = pipeline_setup(cuda_device)
    cfg = {'batch_size': 3, 'latent_size': 512}
    single = [b for _, b in zip(range(5), dc.LabelledPairGenerator(g, seg, cfg, seed=1))]
    double = [b for _, b in zip(range(5), dc.LabelledPairGenerator(g, seg, cfg, seed=1, in_flight=2))]
    torch.cuda.synchronize()
    for a, b in zip(single, double):
        assert a.batch_index == b.batch_index
        assert torch.equal(a.image, b.image)
        for k in a.activations:
            assert torch.equal(a.activations[k], b.activations[k])
        for layer in layers:
            for cn in NAMES:
                assert torch.equal(a.masks[layer][cn], b.masks[layer][cn])


@pytest.mark.gpu
def test_create_dataset_end_to_end_with_swagan(cuda_device, tmp_path):
    from PIL import Image
    from synthesis_in_style_b200 import catalog_creation
    creation = {'class_to_color_map': {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'},
                'keys_for_finegrained_segmentation': ['4', '5'], 'keys_for_class_determination': ['2', '3'], 'keys_to_merge': {},
                'segmenter_type': 'black_white_handwritten_printed', 'only_keep_overlapping': False, 'min_class_contour_area': 2, 'seed': 1}
    cfg_path = tmp_path / 'creation.json'
    cfg_path.write_text(json.dumps(creation))
    orig = tmp_path / 'orig.json'
    orig.write_text(json.dumps({'image_size': 32, 'latent_size': 512, 'stylegan_variant': 'swagan'}))
    sem = tmp_path / 'run' / 'semantic_segmentation'
    gen = torch.Generator().manual_seed(5)
    layers = ['2', '3', '4', '5']
    catalog_creation.save_catalogs({l: torch.nn.functional.normalize(torch.randn(4, 512, generator=gen), dim=1).numpy() for l in layers},
                                   4, sem / 'catalogs')
    names = ['background', 'printed_text', 'handwritten_text']
    (sem / 'merged_classes_4.json').write_text(json.dumps({l: {str(i): names[i % 3] for i in range(4)} for l in layers}))
    out = tmp_path / 'out'
    args = cd.build_arg_parser().parse_args(['random-init:0', str(cfg_path), '-op', str(orig), '-n', '24', '-b', '4', '-s', str(out),
                                             '--num-clusters', '4', '-ssd', str(sem), '--truncate'])
    stats = cd.main(args)
    files = sorted(out.glob('**/*.png'))
    assert stats['images_kept_all_ranks'] >= 24 and len(files) == stats['images_kept_all_ranks']
    assert files[0].relative_to(out).as_posix() == '0/0/0000.png'
    assert np.array(Image.open(files[0])).shape == (32, 64, 3)
    train, val = json.loads((out / 'train.json').read_text()), json.loads((out / 'val.json').read_text())
    assert len(train) == int(len(files) * 0.9) and len(train) + len(val) == len(files)
    assert set(train[0]) == {'file_name', 'has_printed_text', 'has_handwritten_text'}
    coco = json.loads((out / 'coco_gt.json').read_text())
    assert len(coco['images']) == len(val) and [c['name'] for c in coco['categories']] == list(creation['class_to_color_map'])
