"""GPU parity of the whole labelled-pair path (generate -> label) against the oracle pipeline on the same seeds, the
equivalence of the sharded run with the single-stream run, and size-independent properties at the full bench size."""
import pytest
import torch

from oracle import labelling_oracle as lo
from oracle import stylegan2_oracle as so
from synthesis_in_style_b200 import dataset_creation as dc
from synthesis_in_style_b200 import labelling
from synthesis_in_style_b200.model import Generator

pytestmark = pytest.mark.gpu
NAMES = {'background': '#000000', 'printed_text': '#0000FF', 'handwritten_text': '#FF0000'}
CLASS_MAP = {'0': 'background', '1': 'printed_text', '2': 'handwritten_text', '3': 'background'}


def make_setup(size, layers, device, precision='bf16x3', seed_centroids=5, keys_to_merge=None):
    spec = so.GeneratorSpec(size, 512, 8, 2)
    sd = so.perturb_zero_params(so.init_state_dict(spec, seed=0), seed=1234)
    g = Generator(size, 512, 8, precision=precision)
    g.load_state_dict(sd)
    g = g.to(device).eval()
    gen = torch.Generator().manual_seed(seed_centroids)
    cents = {}
    for layer in layers:
        c, _ = g.activation_shape(int(layer))
        cents[layer] = torch.nn.functional.normalize(torch.randn(4, c, generator=gen), dim=1)
    seg = labelling.ClusterSegmenter(None, size, NAMES, keys_for_class_determination=layers[:2], keys_for_finegrained_segmentation=layers[2:],
                                     num_clusters=4, keys_to_merge=keys_to_merge or {}, catalog={k: labelling.FactorCatalog(4, v) for k, v in cents.items()},
                                     class_label_map={k: CLASS_MAP for k in layers})
    return spec, sd, g, seg, cents


@pytest.mark.parametrize('precision', ['fp32', 'bf16x3'])
def test_pipeline_matches_oracle_on_same_seeds(cuda_device, precision):
    """Config 2 shape at reduced batch: 256^2, layers 8,9,12,13, k=4; labels bit-exact where margin > 1e-3, >= 99.9 % overall."""
    layers = ['8', '9', '12', '13']
    spec, sd, g, seg, cents = make_setup(256, layers, cuda_device, precision)
    cfg = {'batch_size': 2, 'latent_size': 512}
    pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1)
    got = next(iter(pipe))
    # oracle on the same stream.  The device noise stream (Philox) is replayed by drawing it again on the device.
    it = iter(dc.build_latent_and_noise_generator(g, cfg, seed=1))
    lat = next(it)
    z, noise = lat.latent.cpu(), [n.cpu() for n in lat.noise]
    want_img, want_acts = so.generator_forward(sd, spec, [z], noise=noise, return_intermediate_activations=True)
    inv = lo.invert_class_label_map({k: CLASS_MAP for k in layers})
    want_masks = lo.prepare_image_segmentation(want_acts, cents, inv, 256)
    assert float((got.image.cpu() - want_img).abs().max()) <= 2e-2
    total = agree = 0
    for layer in layers:
        ids_want, margin = lo.predict_with_margin(want_acts[int(layer)], cents[layer])
        ids_got = got.ids[layer].cpu().long()           # the in-forward label job's own id map (the timed kernels)
        assert torch.equal(seg.catalog[layer].predict(got.activations[int(layer)]).cpu()[margin > 1e-3], ids_want[margin > 1e-3])
        safe = margin > 1e-3
        assert torch.equal(ids_got[safe], ids_want[safe]), (layer, int((ids_got[safe] != ids_want[safe]).sum()))
        total += ids_want.numel(); agree += int((ids_got == ids_want).sum())
        for cn in NAMES:
            m = got.masks[layer][cn]
            assert m.shape == (2, 256, 256) and m.dtype == torch.bool
            assert float((m.cpu() == want_masks[layer][cn]).float().mean()) >= 0.999
    assert agree / total >= 0.999


@pytest.mark.parametrize('replay', [False, True])
def test_sharded_run_equals_single_stream(cuda_device, replay):
    """Rank shards reproduce the single-process stream bit for bit: by replaying every draw (`replay=True`) and by
    addressing the streams positionally (default on CUDA: Philox offset jumps for the device noise, one positional CPU
    draw per round for the latents)."""
    layers = ['4', '5', '6', '7']
    spec, sd, g, seg, cents = make_setup(32, layers, cuda_device)
    cfg = {'batch_size': 3, 'latent_size': 512}
    single = []
    for i, b in zip(range(6), dc.LabelledPairGenerator(g, seg, cfg, seed=1)):
        single.append(b)
    it0 = dc.sharded_latent_stream(g, cfg, 1, 1, 3, replay=replay)
    idx, lat = next(it0)
    idx2, lat2 = next(it0)
    ref = list(zip(range(5), dc.build_latent_and_noise_generator(g, cfg, seed=1)))
    assert (idx, idx2) == (1, 4)
    for got, want in ((lat, ref[1][1]), (lat2, ref[4][1])):
        assert torch.equal(got.latent, want.latent)
        assert all(torch.equal(a, b) for a, b in zip(got.noise, want.noise))
    for rank in range(2):
        pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=1, rank=rank, world_size=2, capture_only_labelled=True)
        if replay:
            pipe.replay_stream = True
        for i, b in zip(range(3), pipe):
            ref_b = single[b.batch_index]
            assert b.batch_index % 2 == rank
            assert torch.equal(b.image, ref_b.image)
            assert sorted(b.activations) == [0, 4, 5, 6, 7]
            for layer in layers:
                assert torch.equal(b.ids[layer], ref_b.ids[layer])
                for cn in NAMES:
                    assert torch.equal(b.masks[layer][cn], ref_b.masks[layer][cn])
        vec = pipe.stats_vector()
        assert int(vec[-2]) == 9 and int(vec[-1]) == 3


def test_full_size_properties(cuda_device):
    """BASELINE config 2 at full size (256^2, batch 32): properties that do not need the oracle."""
    layers = ['8', '9', '12', '13']
    spec, sd, g, seg, cents = make_setup(256, layers, cuda_device)
    cfg = {'batch_size': 32, 'latent_size': 512}
    a = next(iter(dc.LabelledPairGenerator(g, seg, cfg, seed=1)))
    b = next(iter(dc.LabelledPairGenerator(g, seg, cfg, seed=1)))
    assert torch.equal(a.image, b.image)                       # deterministic
    assert torch.isfinite(a.image).all()
    for layer in layers:
        stack = torch.stack([a.masks[layer][cn] for cn in NAMES]).to(torch.int32)
        assert int(stack.sum(0).min()) == 1 and int(stack.sum(0).max()) == 1     # classes partition every pixel
        ids = seg.catalog[layer].predict(a.activations[int(layer)])
        h = a.activations[int(layer)].shape[-1]
        # nearest resize: every (256/h)^2 block is constant and equals the native-resolution class
        native = (ids == 1)
        up = native.repeat_interleave(256 // h, 1).repeat_interleave(256 // h, 2)
        assert torch.equal(up, a.masks[layer]['printed_text'])
    # batch independence: sample i of a batch-32 run equals the same latent run alone (noise is shared per batch)
    it = iter(dc.build_latent_and_noise_generator(g, cfg, seed=1))
    lat = next(it).to(cuda_device)
    with torch.no_grad():
        img1, _ = g([lat.latent[5:6]], noise=lat.noise)
    torch.testing.assert_close(img1[0], a.image[5], rtol=0, atol=1e-4)
    counts = seg.cluster_pixel_counts
    assert all(int(counts[l].sum()) % (32 * a.activations[int(l)].shape[-1] ** 2) == 0 for l in layers)


def test_iter_host_equals_device_iteration(cuda_device):
    """The pipelined host-buffer iterator (pinned in/out, side-stream copies) returns the same pairs in order, without
    and with a `keys_to_merge` destination key (the OR of its source layers)."""
    layers = ['4', '5', '6', '7']
    cfg = {'batch_size': 3, 'latent_size': 512}
    for keys_to_merge in ({}, {'merged': ['4', '6']}):
        spec, sd, g, seg, cents = make_setup(32, layers, cuda_device, keys_to_merge=keys_to_merge)
        ref = [b for _, b in zip(range(5), dc.LabelledPairGenerator(g, seg, cfg, seed=1))]
        host = dc.LabelledPairGenerator(g, seg, cfg, seed=1).iter_host(depth=2)
        for i in range(5):
            hb = next(host)
            assert hb.batch_index == ref[i].batch_index == i
            assert hb.image.is_pinned() and torch.equal(hb.image, ref[i].image.cpu())
            assert set(hb.masks) == set(ref[i].masks) == set(layers) | set(keys_to_merge)
            for layer in hb.masks:
                assert hb.class_names[layer] == list(NAMES)
                for j, cn in enumerate(hb.class_names[layer]):
                    assert torch.equal(hb.masks[layer][j].bool(), ref[i].masks[layer][cn].cpu())
            for dst, (a, b) in keys_to_merge.items():
                for cn in NAMES:
                    assert torch.equal(ref[i].masks[dst][cn], ref[i].masks[a][cn] | ref[i].masks[b][cn]), (dst, cn)


def test_in_forward_labelling_equals_separate_calls(cuda_device):
    """label_jobs inside Generator.forward (fused ToRGB + labelling pass on the large maps) gives the same image, masks,
    ids and histograms as the separate sis_label_assign launches (to rounding: the summation orders differ)."""
    layers = ['8', '9', '12', '13']
    spec, sd, g, seg, cents = make_setup(256, layers, cuda_device)
    cfg = {'batch_size': 4, 'latent_size': 512}
    b = next(iter(dc.LabelledPairGenerator(g, seg, cfg, seed=3)))
    counts_b = {k: v.clone() for k, v in seg.cluster_pixel_counts.items()}
    for v in seg.cluster_pixel_counts.values():
        v.zero_()
    # the same latents and noise through the generator without label jobs, then the separate labelling launches
    lat = next(iter(dc.build_latent_and_noise_generator(g, cfg, seed=3)))
    acts, image = dc.generate_images(lat, g, device=cuda_device)
    masks = seg._as_predicted(seg.label_layers_stacked(acts))
    # the fused pass sums the ToRGB channels (and, on large maps, the distances) in a different order than the separate
    # kernels: equal to rounding, not bit for bit
    assert float((image - b.image).abs().max()) <= 2e-5 * float(image.abs().max())
    for layer in layers:
        for cn in NAMES:
            assert float((masks[layer][cn] != b.masks[layer][cn]).float().mean()) <= 1e-4, (layer, cn)
        diff = (seg.cluster_pixel_counts[layer] - counts_b[layer]).abs().sum()
        assert int(diff) <= 1e-4 * int(seg.cluster_pixel_counts[layer].sum()), layer


def test_create_segmentation_image_equals_oracle_contour_stage(cuda_device):
    """§8(f) row 1 on the device pipeline: masks from the B200 labeller, contour stage vs the oracle restatement of the
    reference's create_segmentation_image on the same masks (colour label images and drop list identical)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import contour_oracle as co
    layers = ['4', '5', '6', '7']
    spec, sd, g, seg, cents = make_setup(32, layers, cuda_device)
    seg.min_class_contour_area = 2
    cfg = {'batch_size': 4, 'latent_size': 512}
    lat = next(iter(dc.build_latent_and_noise_generator(g, cfg, seed=1)))
    acts, image = dc.generate_images(lat, g, device=cuda_device)
    label_images, drop = seg.create_segmentation_image(acts)
    assert label_images.shape == (4, 32, 32, 3) and label_images.dtype.name == 'uint8'
    masks = seg.merge_sub_images(seg.prepare_image_segmentation(acts))
    host = {k: {n: m.cpu().numpy() for n, m in v.items()} for k, v in masks.items()}
    want_images, want_drop = co.create_segmentation_image(host, 4, 32, seg.class_to_color_map, layers[:2], layers[2:],
                                                          seg.only_keep_overlapping, seg.min_class_contour_area)
    assert (label_images == want_images).all() and sorted(drop) == sorted(want_drop)
    with ThreadPoolExecutor(2) as pool:
        par_images, par_drop = seg.create_segmentation_image(acts, pool=pool)
    assert (par_images == label_images).all() and sorted(par_drop) == sorted(drop)


@pytest.mark.parametrize('device_contours,in_flight', [(True, 1), (True, 2), (False, 1)])
def test_build_dataset_writes_the_reference_layout(cuda_device, tmp_path, device_contours, in_flight):
    """§8(f) rows 1+2 end to end: pipelined generate -> label -> contours (device stage or host tasks) -> PNG tree; every
    file is make_image || label image of a kept sample, ids are the running count of kept images."""
    import numpy
    from concurrent.futures import ThreadPoolExecutor
    from PIL import Image

    from synthesis_in_style_b200 import dataset_writer as dw
    layers = ['4', '5', '6', '7']
    spec, sd, g, seg, cents = make_setup(32, layers, cuda_device)
    cfg = {'batch_size': 4, 'latent_size': 512}
    with ThreadPoolExecutor(2) as cpool, ThreadPoolExecutor(2) as wpool:
        stats = dw.build_dataset(dc.LabelledPairGenerator(g, seg, cfg, seed=1, in_flight=in_flight), tmp_path, 10, cpool, wpool,
                                 device_contours=device_contours)
    assert ('host' in stats['contour_stage']) == (not device_contours)
    files = sorted(tmp_path.glob('**/*.png'))
    assert stats['images_kept_all_ranks'] >= 10 and len(files) == stats['files_written_this_rank'] == stats['images_kept_all_ranks']
    # replay the stream without the pipeline
    expect = []
    for b, batch in zip(range(stats['batches_this_rank']), dc.LabelledPairGenerator(g, seg, cfg, seed=1)):
        labels, drop = seg.segment_predicted_clusters(batch.masks, 4)
        imgs = labelling.make_image(batch.image).cpu().numpy()
        expect += [numpy.concatenate([imgs[i], labels[i]], axis=1) for i in range(4) if i not in drop]
    assert len(expect) == len(files)
    for i, f in enumerate(files):
        assert f.relative_to(tmp_path).as_posix() == f'0/0/{i:04d}.png'
        assert numpy.array_equal(numpy.array(Image.open(f)), expect[i])


def test_two_batches_in_flight_equal_single_stream(cuda_device):
    """in_flight=2 (two CUDA streams, two generator workspaces) yields the same batches, in order, as one stream."""
    layers = ['4', '5', '6', '7']
    spec, sd, g, seg, cents = make_setup(32, layers, cuda_device)
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
    # the two pipelines share `g`: run them one after the other, not interleaved
    host1 = dc.LabelledPairGenerator(g, seg, cfg, seed=1).iter_host(depth=2)
    want = []
    for _ in range(4):
        h = next(host1)
        want.append((h.batch_index, h.image.clone(), {k: v.clone() for k, v in h.masks.items()}))
    del host1
    torch.cuda.synchronize()
    host2 = dc.LabelledPairGenerator(g, seg, cfg, seed=1, in_flight=2).iter_host(depth=2)
    for idx, image, masks in want:
        h = next(host2)
        assert h.batch_index == idx and torch.equal(h.image, image)
        for layer in layers:
            assert torch.equal(h.masks[layer], masks[layer])


def test_segmented_stream_device_equals_host(cuda_device):
    """The device contour stage inside the pipelined loop gives the host path's batches: same images, label images and
    drop lists, batch for batch (256^2, the BASELINE layers, two lanes)."""
    import itertools
    import numpy
    layers = ['8', '9', '12', '13']
    spec, sd, g, seg, cents = make_setup(256, layers, cuda_device)
    cfg = {'batch_size': 4, 'latent_size': 512}
    host = list(itertools.islice(dc.LabelledPairGenerator(g, seg, cfg, seed=5).iter_segmented(device_contours=False), 3))
    pipe = dc.LabelledPairGenerator(g, seg, cfg, seed=5, in_flight=2)
    dev = list(itertools.islice(pipe.iter_segmented(device_contours=True), 3))
    for h, d in zip(host, dev):
        assert h.batch_index == d.batch_index
        assert numpy.array_equal(h.images, d.images) and numpy.array_equal(h.label_images, d.label_images)
        assert sorted(h.image_ids_to_drop) == sorted(d.image_ids_to_drop)
    assert pipe.contour_stats['images'] >= 12
