"""`sis_kmeans_steps` on the GPU: step-by-step against the fp64 oracle, independence from batching, launch count,
done fits, and the catalog command end to end into `create_dataset`."""
import json

import numpy as np
import pytest
import torch

from oracle import kmeans_oracle as ko
from synthesis_in_style_b200 import _lib
from synthesis_in_style_b200 import catalog_creation as cc
from synthesis_in_style_b200 import create_catalogs
from synthesis_in_style_b200 import create_dataset as cd

pytestmark = pytest.mark.gpu


def planted(n_per, k, c, seed=0, noise=0.1):
    """Unit rows around k random directions (offsets of norm ~noise, so every row is far nearer its own direction)."""
    g = torch.Generator().manual_seed(seed)
    dirs = torch.nn.functional.normalize(torch.randn(k, c, generator=g, dtype=torch.float64), dim=1)
    x = dirs.repeat_interleave(n_per, 0) + noise / c ** 0.5 * torch.randn(k * n_per, c, generator=g, dtype=torch.float64)
    perm = torch.randperm(k * n_per, generator=g)
    return ko.normalize_rows(x[perm]), torch.arange(k).repeat_interleave(n_per)[perm]


def new_fit(x64, centers64, device, seed=7, batch_size=100, max_steps=60, max_no_improvement=10, ratio=0.01):
    fit = cc.KMeansFit(x64.float().to(device).contiguous(), centers64.float().to(device).contiguous(),
                       state=cc.new_states(1, device)[0])
    cc.init_state(fit, seed, batch_size, max_steps, max_no_improvement, ratio)
    return fit


@pytest.mark.parametrize('max_no_improvement', [None, 10])
@pytest.mark.parametrize('k', [3, 8, 23])
@pytest.mark.parametrize('c', [32, 128, 512])
def test_steps_match_the_oracle(cuda_device, c, k, max_no_improvement):
    x, truth = planted(40, k, c, seed=c + k)
    init = torch.stack([x[(truth == i).nonzero()[0, 0]] for i in range(k)])
    max_steps = 40
    fit = new_fit(x, init, cuda_device, max_steps=max_steps, max_no_improvement=max_no_improvement)
    before, after, counts, inertia = [], [], [], []
    bi = torch.full((1, 1), float('nan'), device=cuda_device)
    while not fit.done:
        before.append(fit.centers.double().cpu())
        cc.kmeans_steps([fit], 1, batch_inertia=bi)
        after.append(fit.centers.double().cpu())
        counts.append(fit.counts.double().cpu())
        inertia.append(float(bi[0, 0]))
    n_dev = fit.steps_done
    assert n_dev == len(after) and (max_no_improvement is not None or n_dev == max_steps)

    def on_step(t, idx, labels, centers, cnt):
        # the labels the device's own pre-step centres give equal the oracle's; every margin is wide
        d = ((x[idx][:, None, :] - ko.normalize_rows(before[t])[None]) ** 2).sum(2)
        two = d.topk(2, dim=1, largest=False).values
        assert float((two[:, 1] - two[:, 0]).min()) > 1e-2
        assert torch.equal(d.argmin(1), labels), t
        assert torch.equal(cnt, counts[t]), t
        torch.testing.assert_close(centers, after[t], rtol=0, atol=1e-5)

    _, _, n_iter = ko.fit_steps(x, init.clone(), torch.zeros(k, dtype=torch.float64), seed=7, batch_size=100, max_steps=max_steps,
                                max_no_improvement=max_no_improvement, ratio=0.01,
                                batch_inertia=lambda t, own: inertia[t], on_step=on_step)
    assert n_iter == n_dev


def test_reassignment_matches_the_oracle(cuda_device):
    """A centre on no data starves and is replaced at step 10 by the row the stream-1 draws pick."""
    k, c = 6, 64
    x, truth = planted(100, k - 1, c)
    init = torch.cat([torch.stack([x[(truth == i).nonzero()[0, 0]] for i in range(k - 1)]),
                      ko.normalize_rows(torch.randn(1, c, generator=torch.Generator().manual_seed(1), dtype=torch.float64))])
    fit = new_fit(x, init, cuda_device, max_steps=10, max_no_improvement=None)
    cc.kmeans_steps([fit], 10)
    centers, counts, n_iter = ko.fit_steps(x, init.clone(), torch.zeros(k, dtype=torch.float64), seed=7, batch_size=100,
                                           max_steps=10, max_no_improvement=None, ratio=0.01)
    assert n_iter == fit.steps_done == 10
    assert float(counts[k - 1]) > 0 and torch.equal(fit.counts.double().cpu(), counts)
    torch.testing.assert_close(fit.centers.double().cpu(), centers, rtol=0, atol=1e-5)


def test_batched_fits_equal_fits_alone(cuda_device):
    torch.manual_seed(0)
    layers = {8: torch.randn(4, 64, 24, 24, device=cuda_device), 12: torch.randn(2, 128, 32, 32, device=cuda_device)}
    ks = range(3, 24)
    stats = {}
    together = cc.fit_catalogs(layers, ks, random_state=3, stats=stats)
    assert stats['fits'] == 42 and stats['step_launches'] == stats['host_syncs'] >= 1
    for layer, act in layers.items():
        for k in ks:
            alone = cc.fit_catalogs({layer: act}, [k], random_state=3)[layer][k]
            assert np.array_equal(alone[0], together[layer][k][0]), (layer, k)
            assert torch.equal(alone[1], together[layer][k][1]), (layer, k)
            assert alone[1].shape == (act.shape[0],) + act.shape[2:]


def test_one_launch_per_chunk_whatever_the_number_of_fits(cuda_device):
    x, _ = planted(50, 4, 32)
    for n_fits in (1, 40):
        fits = [new_fit(x, x[i:i + 4 + i % 3], cuda_device, seed=i, max_steps=100) for i in range(n_fits)]
        before = _lib.launch_count()
        cc.kmeans_steps(fits, cc.KMEANS_CHUNK_STEPS)
        assert _lib.launch_count() - before == 1
        torch.cuda.synchronize()


def test_done_fits_do_not_move(cuda_device):
    x, _ = planted(50, 4, 48)
    fit = new_fit(x, x[:4], cuda_device, max_steps=5, max_no_improvement=None)
    bi = torch.full((1, 8), float('nan'), device=cuda_device)
    cc.kmeans_steps([fit], 8, batch_inertia=bi)
    assert fit.done and fit.steps_done == 5
    assert bool(torch.isfinite(bi[0, :5]).all()) and bool(torch.isnan(bi[0, 5:]).all())
    centers, counts, state = fit.centers.clone(), fit.counts.clone(), fit.state.clone()
    bi.fill_(float('nan'))
    cc.kmeans_steps([fit], 8, batch_inertia=bi)
    assert torch.equal(fit.centers, centers) and torch.equal(fit.counts, counts) and torch.equal(fit.state, state)
    assert bool(torch.isnan(bi).all())


def test_catalogs_from_a_checkpoint_feed_create_dataset(cuda_device, tmp_path):
    orig = tmp_path / 'orig.json'
    orig.write_text(json.dumps({'image_size': 32, 'latent_size': 512, 'stylegan_variant': 2}))
    sem = tmp_path / 'run' / 'semantic_segmentation'
    args = create_catalogs.build_arg_parser().parse_args(['random-init:0', '-op', str(orig), '-n', '8', '-b', '4', '-ssd', str(sem),
                                                          '--layers', '4', '5', '6', '7', '--cluster-range', '3', '6'])
    out = create_catalogs.main(args)
    assert out['layers'] == [4, 5, 6, 7] and sorted(out['catalogs']) == [3, 4, 5]
    for k in (3, 4, 5):
        cat = np.load(sem / 'catalogs' / f'{k}.npz')
        assert sorted(cat.files) == ['4', '5', '6', '7'] and cat['4'].shape == (k, 512)
        np.testing.assert_allclose(np.linalg.norm(cat['6'], axis=1), 1.0, atol=1e-5)
        arrays = np.load(sem / 'cluster_arrays' / f'{k}.npz')
        assert arrays['images'].shape == (8, 32, 32, 3) and arrays['images'].dtype == np.uint8
        assert arrays['4'].shape == (8, 16, 16) and arrays['6'].shape == (8, 32, 32) and int(arrays['6'].max()) < k
    names = ['background', 'printed_text', 'handwritten_text']
    (sem / 'merged_classes_4.json').write_text(json.dumps({str(l): {str(i): names[i % 3] for i in range(4)} for l in range(4, 8)}))
    creation = {'class_to_color_map': {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'},
                'keys_for_finegrained_segmentation': ['6', '7'], 'keys_for_class_determination': ['4', '5'], 'keys_to_merge': {},
                'segmenter_type': 'black_white_handwritten_printed', 'only_keep_overlapping': False, 'min_class_contour_area': 2, 'seed': 1}
    cfg = tmp_path / 'creation.json'
    cfg.write_text(json.dumps(creation))
    images = tmp_path / 'out'
    stats = cd.main(cd.build_arg_parser().parse_args(['random-init:0', str(cfg), '-op', str(orig), '-n', '8', '-b', '4',
                                                      '-s', str(images), '--num-clusters', '4', '-ssd', str(sem)]))
    files = sorted(images.glob('**/*.png'))
    assert stats['images_kept_all_ranks'] >= 8 and len(files) == stats['images_kept_all_ranks']
    for name in ('train.json', 'val.json', 'coco_gt.json'):
        assert (images / name).is_file()
