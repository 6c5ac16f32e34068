"""GPU parity of the TIMED path at the BASELINE batch sizes: BASELINE.json configs[1..3] through
`LabelledPairGenerator(in_flight=2)` with the in-forward label jobs (the kernels bench.py times:
`label_wide_kernel<K, 0|1>` with the ToRGB fused where the tensor is shared, `label_native_kernel` on small maps),
checked against the CPU oracle on the same latents / noise / weights:

  * images: max-abs error <= 2e-2 and PSNR >= 40 dB (peak 2.0, clamped images) -- the north star's tolerance;
  * cluster-id maps WRITTEN BY THE FUSED JOBS: bit-exact wherever the oracle's nearest-centroid margin exceeds 1e-3,
    >= 99.9 % overall; class masks = ids through the class map, nearest-resized (exact, derived from the same ids).

The workload definitions are bench.py's (`WORKLOADS`), so the tests and the benchmark cannot drift apart.
"""
import pytest
import torch

import bench
from oracle import labelling_oracle as lo
from oracle import stylegan2_oracle as so
from synthesis_in_style_b200 import dataset_creation as dc
from synthesis_in_style_b200 import labelling
from synthesis_in_style_b200.model import Generator

pytestmark = pytest.mark.gpu


def build(cfg_id, device, k=bench.K_CLUSTERS, catalog=None):
    wl = bench.WORKLOADS[cfg_id]
    spec, sd = bench.oracle_state(wl['size'])
    g = Generator(wl['size'], bench.STYLE_DIM, bench.N_MLP)
    g.load_state_dict(sd)
    g = g.to(device).eval()
    cents = catalog if catalog is not None else bench.synthetic_catalog(wl)
    layers = bench.wl_layers(wl)
    class_map = {str(i): ('background', 'printed_text', 'handwritten_text')[i % 3] for i in range(k)} if k != 4 else bench.CLASS_MAP
    seg = labelling.ClusterSegmenter(None, wl['size'], bench.COLORS, keys_for_class_determination=wl['class_keys'],
                                     keys_for_finegrained_segmentation=wl['fine_keys'], num_clusters=k, keys_to_merge={},
                                     catalog={l: labelling.FactorCatalog(k, cents[l]) for l in layers},
                                     class_label_map={l: class_map for l in layers})
    return wl, spec, sd, g, seg, cents, class_map


def check_batch(wl, spec, sd, g, seg, cents, class_map, batch, lat, mean_latent):
    """One LabelledBatch of the pipeline against the oracle on the same (latent, noise) batch `lat`."""
    z = lat.latent.cpu()
    noise = [n.cpu() for n in lat.noise]
    want_img, want_acts = bench.oracle_forward(wl, spec, sd, z, torch.roll(z, 1, 0), noise,
                                               mean_latent.cpu() if mean_latent is not None else None)
    got_img = batch.image.cpu()
    assert float((got_img - want_img).abs().max()) <= 2e-2
    mse = float(((got_img.clamp(-1, 1) - want_img.clamp(-1, 1)) ** 2).mean())
    assert 10 * torch.log10(torch.tensor(4.0 / max(mse, 1e-30))) >= 40.0
    inv = lo.invert_class_label_map({l: class_map for l in cents})
    S = wl['size']
    total = agree = 0
    for layer in bench.wl_layers(wl):
        ids_want, margin = lo.predict_with_margin(want_acts[int(layer)], cents[layer])
        ids_got = batch.ids[layer].cpu().long()                      # written by the in-forward label job
        assert ids_got.shape == ids_want.shape
        safe = margin > 1e-3
        assert torch.equal(ids_got[safe], ids_want[safe]), (layer, int((ids_got[safe] != ids_want[safe]).sum()))
        total += ids_want.numel()
        agree += int((ids_got == ids_want).sum())
        # the masks the job wrote are exactly its ids through the class map, nearest-replicated to S x S
        rep = S // ids_got.shape[-1]
        for cn, class_ids in inv[layer].items():
            native = torch.zeros_like(ids_got, dtype=torch.bool)
            for cid in class_ids:
                native |= ids_got == cid
            up = native.repeat_interleave(rep, 1).repeat_interleave(rep, 2)
            assert torch.equal(batch.masks[layer][cn].cpu(), up), (layer, cn)
    assert agree / total >= 0.999, agree / total
    # a fused job of an activation also captured must have labelled that very tensor
    assert set(batch.activations) == set(range(spec.n_latent))
    # every captured activation of every sample, on the kernels the batch size selects (and the plan's epilogues that
    # write the next layer's operand planes), with test_generator_256_against_oracle's per-layer bound
    worst_k, worst_e, worst_frac = None, 0.0, -1.0
    for k, want in want_acts.items():
        e = float((batch.activations[k].cpu() - want).abs().max())
        bound = 2e-3 * max(1.0, float(want.abs().max()))
        assert batch.activations[k].shape == want.shape and e <= bound, (k, e, bound)
        if e / bound > worst_frac:
            worst_k, worst_e, worst_frac = k, e, e / bound
    print(f'\n{S}^2 B={z.shape[0]}: largest activation error {worst_e:.2e} (layer {worst_k}, {worst_frac:.3f} of its bound)')


@pytest.mark.parametrize('cfg_id,batch_index', [(2, 1), (3, 0), (4, 0)])
def test_baseline_config_through_the_timed_path(cuda_device, cfg_id, batch_index):
    """configs[1]: 256^2 B=32; configs[2]: 512^2 B=16, layers 8..15; configs[3]: 1024^2 B=8, truncation 0.7 + style mixing.
    `batch_index` 1 is the second lane of in_flight=2 (the replica generator workspace on its own stream)."""
    wl, spec, sd, g, seg, cents, class_map = build(cfg_id, cuda_device)
    cfg = {'batch_size': wl['batch'], 'latent_size': bench.STYLE_DIM}
    mean_latent = None
    if wl['truncation']:
        torch.manual_seed(7)
        with torch.no_grad():
            mean_latent = g.mean_latent(4096)
    pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, mean_latent=mean_latent, in_flight=2, mix_inject_index=wl['mix'])
    it = iter(pipe)
    for _ in range(batch_index + 1):
        got = next(it)
    assert got.batch_index == batch_index and got.image.shape == (wl['batch'], 3, wl['size'], wl['size'])
    torch.cuda.synchronize()
    g.check()
    # the same stream, replayed (device noise comes from the device generator: draw it again)
    replay = iter(dc.build_latent_and_noise_generator(g, cfg, seed=1))
    for _ in range(batch_index + 1):
        lat = next(replay)
    check_batch(wl, spec, sd, g, seg, cents, class_map, got, lat, mean_latent)


def test_k20_catalog_through_the_timed_path(cuda_device):
    """k = 20 centroids picked FROM generator activations (so every cluster is populated and margins are small), labelled
    by the in-forward jobs (`label_wide_kernel<24, *>`, expanded form) at 256^2, B = 4."""
    wl = bench.WORKLOADS[2]
    spec, sd = bench.oracle_state(256)
    torch.manual_seed(11)
    z0 = torch.randn(1, 512)
    _, acts0 = so.generator_forward(sd, spec, [z0], noise=so.make_noise(spec), return_intermediate_activations=True)
    gen = torch.Generator().manual_seed(3)
    cents = {}
    for layer in bench.wl_layers(wl):
        flat = lo.partial_flat(acts0[int(layer)])
        pick = torch.randperm(flat.shape[0], generator=gen)[:20]
        cents[layer] = torch.nn.functional.normalize(flat[pick].clone(), dim=1)
    wl, spec, sd, g, seg, cents, class_map = build(2, cuda_device, k=20, catalog=cents)
    cfg = {'batch_size': 4, 'latent_size': 512}
    got = next(iter(dc.LabelledPairGenerator(g, seg, cfg, seed=1, in_flight=2)))
    lat = next(iter(dc.build_latent_and_noise_generator(g, cfg, seed=1)))
    check_batch(wl, spec, sd, g, seg, cents, class_map, got, lat, None)
    for layer in bench.wl_layers(wl):
        assert int((seg.cluster_pixel_counts[layer] > 0).sum()) >= 10      # a populated catalog, not one winner


def test_bench_parity_helper(cuda_device):
    """bench.py's `parity` key is computed by `parity_check`: it must agree with the checks above on a small batch."""
    wl, spec, sd, g, seg, cents, class_map = build(2, cuda_device)
    cfg = {'batch_size': 4, 'latent_size': 512}
    lat = next(iter(dc.build_latent_and_noise_generator(g, cfg, seed=1))).to(cuda_device)
    jobs = seg.make_label_jobs(g, 4)
    acts, img = dc.generate_images(lat, g, device=cuda_device, label_jobs=jobs)
    torch.cuda.synchronize()
    rep = bench.parity_check(wl, spec, sd, lat, img, jobs, None, n=2)
    assert rep['ok'] and rep['label_mismatches_at_margin_gt_1e-3'] == 0 and rep['label_agreement'] >= 0.999
    assert rep['image_max_abs_err'] <= 2e-2 and rep['image_psnr_db_peak2'] >= 40
