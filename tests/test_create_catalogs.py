"""Catalog creation without a GPU: the counter-based draws, the k-means oracle on planted data, the command's flags and
the argument checks `sis_kmeans_steps` / `sis_kmeans_init_state` make before any CUDA call."""
import ctypes

import numpy as np
import torch

from oracle import kmeans_oracle as ko
from synthesis_in_style_b200 import _lib
from synthesis_in_style_b200 import create_catalogs as cc


def test_counter_hash_is_pinned():
    # splitmix64(splitmix64(splitmix64(seed) ^ t) ^ (j << 1 | stream)): the library and the oracle share these values
    assert [int(v) for v in ko.draw(0, 0, 3, 0)] == [0x238275bc38fcbe91, 0xb28c4c30d302532e, 0x7209949bdf4f2159]
    assert [int(v) for v in ko.draw(12345, 7, 2, 1)] == [0x8ffda1ba661f7f87, 0x18c4cda5d7fad75d]
    assert ko.batch_rows(0, 0, 5, 1000).tolist() == [433, 574, 385, 237, 794]
    assert int(ko.splitmix64(np.uint64(0))) == 0xe220a8397b1dcdaf            # the published first output of seed 0


def planted(n_per, k, c, seed=0, noise=0.1):
    g = torch.Generator().manual_seed(seed)
    dirs = torch.nn.functional.normalize(torch.randn(k, c, generator=g, dtype=torch.float64), dim=1)
    x = dirs.repeat_interleave(n_per, 0) + noise / c ** 0.5 * torch.randn(k * n_per, c, generator=g, dtype=torch.float64)
    perm = torch.randperm(k * n_per, generator=g)
    return ko.normalize_rows(x[perm]), torch.arange(k).repeat_interleave(n_per)[perm], dirs


def test_oracle_recovers_planted_clusters():
    k = 5
    x, truth, dirs = planted(200, k, 24)
    # one row of each planted cluster, and one centre on no data: it starves and is reassigned at step 10
    first = torch.stack([x[(truth == i).nonzero()[0, 0]] for i in range(k)])
    centers = torch.cat([first, ko.normalize_rows(torch.randn(1, 24, dtype=torch.float64))])
    counts = torch.zeros(k + 1, dtype=torch.float64)
    seen = []
    centers, counts, n_iter = ko.fit_steps(x, centers, counts, seed=3, batch_size=100, max_steps=200, max_no_improvement=10,
                                           ratio=0.01, on_step=lambda t, idx, lab, c, n: seen.append(float(n.min())))
    assert 10 <= n_iter < 200 and seen[8] == 0 and seen[9] > 0              # the starved centre took a row at t = 9
    torch.testing.assert_close(centers.norm(dim=1), torch.ones(k + 1, dtype=torch.float64))
    sim = centers @ dirs.t()
    assert sorted(set(sim.argmax(1).tolist())) == list(range(k)) and float(sim.max(1).values.min()) > 0.98
    labels, _ = ko.assign(x, centers)
    assert (sim.argmax(1)[labels] == truth).double().mean() > 0.99


def test_command_defaults():
    a = cc.build_arg_parser().parse_args(['run/checkpoints/100.pt'])
    assert (a.num_images, a.batch_size, a.device, a.truncate, a.seed, a.layers, a.min_size, a.cluster_range) == \
        (100, 10, 'cuda', False, 1, None, 32, [3, 24])
    assert (a.random_state, a.kmeans_batch_size, a.max_iter, a.n_init, a.init_size, a.reassignment_ratio, a.max_no_improvement) == \
        (0, 100, 100, 3, None, 0.01, 10)
    assert a.original_config_path is None and a.semantic_segmentation_base_dir is None
    a = cc.build_arg_parser().parse_args(['random-init:0', '-op', 'o.json', '-n', '8', '-b', '4', '-ssd', 'sem', '--layers', '8', '9',
                                          '--cluster-range', '3', '6', '--max-no-improvement', '-1'])
    assert (a.num_images, a.batch_size, a.layers, a.cluster_range, a.max_no_improvement) == (8, 4, [8, 9], [3, 6], -1)


def test_kmeans_arguments_are_checked_without_a_gpu():
    lib = _lib.load()
    assert lib.sis_kmeans_state_bytes() == 64 and ctypes.sizeof(_lib.KmeansFit) == 48
    dummy = 0x1000                                    # never dereferenced: every call below fails its checks first

    def steps(k=4, channels=64, n=100, steps=1, indices=None, n_indices=0, state=dummy):
        fit = _lib.KmeansFit(dummy, n, channels, k, dummy, dummy, state)
        return lib.sis_kmeans_steps((_lib.KmeansFit * 1)(fit), 1, steps, indices, n_indices, None, None)

    for kwargs, msg in [(dict(k=1), b'k = 1 outside [2, 32]'), (dict(k=33), b'k = 33 outside [2, 32]'),
                        (dict(channels=513), b'channels = 513 outside [1, 512]'), (dict(n=3), b'n = 3 < k = 4'),
                        (dict(steps=0), b'steps must be >= 1'), (dict(state=None), b'NULL state'),
                        (dict(indices=dummy, n_indices=1025), b'n_indices 1025 outside [1, 1024]'),
                        (dict(indices=dummy, n_indices=10, steps=2), b'exactly one step')]:
        assert steps(**kwargs) == 1, kwargs
        assert msg in lib.sis_last_error(), (kwargs, lib.sis_last_error())
    assert lib.sis_kmeans_steps(None, 0, 1, None, 0, None, None) == 1 and b'no fits' in lib.sis_last_error()
    assert lib.sis_kmeans_init_state(dummy, 0, 1025, 10, 10, 0.01, None) == 1
    assert b'batch_size 1025 outside [1, 1024]' in lib.sis_last_error()
    assert lib.sis_kmeans_init_state(dummy, 0, 100, 0, 10, 0.01, None) == 1 and b'max_steps' in lib.sis_last_error()
    assert lib.sis_kmeans_init_state(None, 0, 100, 10, 10, 0.01, None) == 1 and b'd_state is NULL' in lib.sis_last_error()
