"""GPU end-to-end: the reference-shaped API (NGP / render / NGPTrainer / train.py / gui.py) on the CUDA path."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_full_step_matches_oracle_step():
    import __graft_entry__ as g
    g.smoke()


def test_state_dict_keys_match_reference():
    from modules.networks import NGP
    for half in (False, True):
        m = NGP(scale=0.5, max_res=1024, half_opt=half)
        keys = set(m.state_dict().keys())
        want = {'center', 'xyz_min', 'xyz_max', 'half_size', 'density_bitfield', 'density_grid', 'grid_coords',
                'pos_encoder.hash_table', 'xyz_encoder.hidden_layers.0.weight', 'xyz_encoder.output_layer.weight',
                'rgb_net.hidden_layers.0.weight', 'rgb_net.hidden_layers.1.weight', 'rgb_net.output_layer.weight'}
        if half:
            want.add('pos_encoder.hash_grad')  # hash_encoder_half.py:300-306
        assert keys == want, keys ^ want
        assert m.pos_encoder.hash_table.shape == ((5710032, 2) if half else (11420064,))
        assert m.xyz_encoder.output_layer.weight.shape == (16, 64)


def test_fused_mlp_path_equals_torch_path():
    """NGP.forward through the tcgen05 kernel vs the reference's nn.Linear graph under autocast."""
    from modules.networks import NGP
    torch.manual_seed(0)
    m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
    with torch.no_grad():
        m.pos_encoder.hash_table.mul_(3e3)
    x = (torch.rand(5000, 3, device='cuda') - 0.5) * 0.98
    d = torch.randn(5000, 3, device='cuda')
    with torch.autocast('cuda', dtype=torch.float16):
        s_f, c_f = m(x, d)
        m._fusable = lambda _x: False
        s_t, c_t = m(x, d)
    assert (s_f - s_t).abs().max() <= 8e-3 * s_t.abs().max()
    assert (c_f.float() - c_t.float()).abs().max() <= 3e-3


@pytest.mark.parametrize("extra", [[], ['--graph_step']])
def test_training_on_analytic_scene_reaches_psnr(tmp_path, monkeypatch, extra):
    """train.py end to end (small config): PSNR against the analytic teacher's held-out views, through the module /
    autograd step and through the graph-captured step."""
    import train
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(train, 'dataset_dict', {'synthetic': _small_dataset})
    psnrs = train.main(['--dataset_name', 'synthetic', '--half_opt', '--batch_size', '4096', '--max_steps', '400']
                       + extra)
    assert (tmp_path / 'results' / 'model.pth').exists() and (tmp_path / 'results' / 'rgb_000.png').exists()
    assert min(psnrs) > 22.0, psnrs


def _small_dataset(**kw):
    from datasets.synthetic import SyntheticLego
    kw = dict(kw)
    kw.update(img_wh=(100, 100), focal=138.9, n_images=kw.get('n_images', 40))
    return SyntheticLego(**kw)


def test_gui_render_cam():
    import argparse
    from datasets.synthetic import SyntheticLego
    from gui import NGPGUI
    ds = SyntheticLego(img_wh=(64, 64), focal=88.9, n_images=4).to('cuda')
    hp = argparse.Namespace(ckpt_path=None, dataset_name='synthetic')
    gui = NGPGUI(hp, {'scale': 0.5, 'max_res': 1024, 'half_opt': True}, ds.K, ds.img_wh, ds.poses, radius=1.4)
    with torch.autocast('cuda', dtype=torch.float16):
        gui.model.update_density_grid(0.01 * 1024 / 3 ** 0.5, warmup=True)
    img = gui.render_cam()
    assert img.shape == (64, 64, 3) and torch.isfinite(img).all()


def test_render_frame_equals_incremental_loop(lego_bitfield):
    """Batched test-time rendering == the reference-shaped while-loop (chunking must not matter)."""
    import modules.rendering as R
    from datasets.ray_utils import get_ray_directions, get_rays
    from datasets.synthetic import SyntheticLego, hemisphere_poses
    from modules.networks import NGP
    torch.manual_seed(1)
    m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
    with torch.no_grad():
        m.pos_encoder.hash_table.mul_(1e5)  # dense-ish medium so early termination is exercised
        m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
    K = SyntheticLego(n_images=2, img_wh=(160, 160), focal=222.2).K.cuda()
    o, d = get_rays(get_ray_directions(160, 160, K, device='cuda'), hemisphere_poses(3)[2].cuda())
    with torch.autocast('cuda', dtype=torch.float16):
        thr = 0.25    # a high termination threshold so that most rays that hit the medium terminate early
        R._FORCE_LOOP = True
        ref = R.render(m, o, d, test_time=True, T_threshold=thr)
        R._FORCE_LOOP = False
        R._NO_COMPACTION = True
        allsamples = R.render(m, o, d, test_time=True, T_threshold=thr)   # march everything, shade everything, composite
        R._NO_COMPACTION = False
        got = R.render(m, o, d, test_time=True, T_threshold=thr)          # compacting rounds (one CUDA graph per frame)
        got2 = R.render(m, o, d, test_time=True, T_threshold=thr)         # replay of the cached graph
    assert float(ref['opacity'].max()) > 0.5
    terminated = float((ref['opacity'] >= 1 - thr).float().mean())     # rays stopped by the transmittance threshold
    for k in ('rgb', 'opacity', 'depth'):
        assert (ref[k] - allsamples[k]).abs().max() < 2e-3, k
        assert (ref[k] - got[k]).abs().max() < 2e-3, k
        assert torch.equal(got[k], got2[k]), k
    # early termination: rays that hit the dense medium leave the live list, so fewer samples are shaded than marched
    assert terminated > 0.02, terminated
    assert int(got['total_samples']) < int(allsamples['total_samples']), (got['total_samples'], allsamples['total_samples'])
    assert int(got['total_samples']) >= int(ref['total_samples']) * 0.5


@pytest.mark.parametrize("use_graph", [False, True])
def test_static_graph_step_equals_autograd_step(lego_bitfield, monkeypatch, use_graph):
    """The graph-captured sync-free step must produce the same update as the module/autograd step."""
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer

    def build():
        torch.manual_seed(3)
        m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
        with torch.no_grad():
            m.pos_encoder.hash_table.mul_(2e3)
            m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
        return m, NGPTrainer(m, lr=1e-2)

    n = 2048
    o, d = make_rays(n, seed=9)
    o, d = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    gt = torch.rand(n, 3, device='cuda')
    noise = torch.rand(n, device='cuda')

    m1, t1 = build()
    monkeypatch.setattr(torch, 'rand_like', lambda t, **k: noise.clone())
    losses1 = [float(t1.step(o, d, gt)[0]) for _ in range(3)]
    monkeypatch.undo()

    m2, t2 = build()
    fs = StaticTrainStep(t2, n, samples_per_ray_capacity=64, use_graph=use_graph)
    losses2 = [float(fs.step(o, d, gt, noise=noise)) for _ in range(3)]
    assert int(fs.counter[0]) > 1000
    for a, b in zip(losses1, losses2):
        assert abs(a - b) < 2e-3 * max(a, 1e-6), (losses1, losses2)
    for p1, p2 in zip(m1.parameters(), m2.parameters()):
        # Adam's first steps move every touched entry by ~lr regardless of gradient size, so compare the
        # update direction through the parameters themselves with an lr-scaled tolerance
        diff = (p1 - p2).abs()
        assert float((diff > 2e-3).float().mean()) < 2e-3, float(diff.max())
    assert t2.step_count == 3 and int(fs.step_dev) == 3


def test_static_step_capacity_overflow_is_safe(lego_bitfield):
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer
    torch.manual_seed(3)
    m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
    with torch.no_grad():
        m.density_bitfield.fill_(255)  # fully occupied: ~530 samples/ray >> capacity
    n = 1024
    o, d = make_rays(n, seed=10)
    fs = StaticTrainStep(NGPTrainer(m), n, samples_per_ray_capacity=32, use_graph=True)
    loss = fs.step(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), torch.rand(n, 3, device='cuda'))
    assert torch.isfinite(loss).all()
    reserved, dropped = fs.counter.tolist()
    assert reserved > fs.cap and dropped > 0   # rays that did not fit were dropped and counted, never written
    assert all(torch.isfinite(p).all() for p in m.parameters())


@pytest.mark.parametrize("cfg", [
    dict(name="lego_fp32", scale=0.5, half=False, esf=0.0),          # BASELINE configs[0]: fp32 encoder
    dict(name="garden_half", scale=16.0, half=True, esf=1 / 256),    # BASELINE configs[2]: 6 cascades, 4096 layout
])
def test_static_step_other_configs(cfg, monkeypatch):
    """fp32-encoder and multi-cascade (garden-scale) configurations: graph step == module/autograd step."""
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer

    def build():
        torch.manual_seed(4)
        m = NGP(scale=cfg["scale"], max_res=1024 if cfg["scale"] == 0.5 else 4096, half_opt=cfg["half"]).cuda()
        with torch.no_grad():
            if cfg["half"]:
                m.pos_encoder.hash_table.mul_(2e3)
            g = torch.Generator(device='cuda').manual_seed(5)
            m.density_bitfield.copy_((torch.rand(m.density_bitfield.shape, device='cuda', generator=g) < 0.3) *
                                     torch.randint(1, 256, m.density_bitfield.shape, device='cuda', generator=g).to(torch.uint8))
        return m, NGPTrainer(m, lr=1e-2)

    n = 1024
    o, d = make_rays(n, seed=12, radius=1.4 if cfg["scale"] == 0.5 else 3.0)
    o, d = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    gt, noise = torch.rand(n, 3, device='cuda'), torch.rand(n, device='cuda')
    m1, t1 = build()
    assert m1.cascades == (1 if cfg["scale"] == 0.5 else 6)
    monkeypatch.setattr(torch, 'rand_like', lambda t, **k: noise.clone())
    l1 = [float(t1.step(o, d, gt, cfg["esf"])[0].detach()) for _ in range(2)]
    monkeypatch.undo()
    m2, t2 = build()
    fs = StaticTrainStep(t2, n, samples_per_ray_capacity=512, exp_step_factor=cfg["esf"], use_graph=True)
    l2 = [float(fs.step(o, d, gt, noise=noise)) for _ in range(2)]
    assert int(fs.counter[0]) > 1000
    for a, b in zip(l1, l2):
        assert abs(a - b) < 3e-3 * max(a, 1e-6), (l1, l2)
    for p1, p2 in zip(m1.parameters(), m2.parameters()):
        assert float(((p1 - p2).abs() > 2e-3).float().mean()) < 5e-3


def test_device_side_grad_scaler(lego_bitfield):
    """GradScaler semantics on the device: an overflowing step is skipped and halves the scale; clean steps count
    towards the growth interval."""
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer
    torch.manual_seed(3)
    m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
    with torch.no_grad():
        m.pos_encoder.hash_table.mul_(2e3)
        m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
    n = 1024
    o, d = make_rays(n, seed=14)
    o, d = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    fs = StaticTrainStep(NGPTrainer(m), n, samples_per_ray_capacity=64, use_graph=True)
    assert float(fs.scale_state[0]) == 65536.0
    fs.step(o, d, torch.rand(n, 3, device='cuda'))
    assert float(fs.scale_state[0]) == 65536.0 and int(fs.scale_state[1:].view(torch.int32)) == 1
    before = [p.detach().clone() for p in m.parameters()]
    fs.step(o, d, torch.full((n, 3), float('nan'), device='cuda'))     # poisoned targets -> non-finite gradients
    assert float(fs.scale_state[0]) == 32768.0 and int(fs.scale_state[1:].view(torch.int32)) == 0
    for p, b in zip(m.parameters(), before):
        assert torch.equal(p, b)                                         # the step was skipped
    assert abs(float(fs.hyper[2]) - 1 / 32768.0) < 1e-12
    fs.step(o, d, torch.rand(n, 3, device='cuda'))                      # training continues with the halved scale
    assert all(torch.isfinite(p).all() for p in m.parameters())
    assert any(not torch.equal(p, b) for p, b in zip(m.parameters(), before))


@pytest.mark.parametrize("use_graph", [False, True])
def test_static_step_with_device_sampled_batches(lego_bitfield, use_graph):
    """step_sampled() (batch drawn inside the graph from the resident training set) == step() fed with the
    oracle's restatement of the same draw, for three consecutive steps (the draw depends on the device step)."""
    from datasets.synthetic import SyntheticLego
    from modules.networks import NGP
    from oracle import oracle as O
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer

    ds = SyntheticLego(n_images=6, img_wh=(64, 64), focal=88.9, batch_size=1024, seed=2).to('cuda')
    ds.build_image_bank()

    def build():
        torch.manual_seed(3)
        m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
        with torch.no_grad():
            m.pos_encoder.hash_table.mul_(2e3)
            m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
        return m, NGPTrainer(m, lr=1e-2)

    n, seed = 1024, 1234
    m1, t1 = build()
    fs1 = StaticTrainStep(t1, n, samples_per_ray_capacity=64, use_graph=use_graph)
    fs1.attach_ray_source(ds.rays, ds.poses, ds.directions, seed=seed)
    m2, t2 = build()
    fs2 = StaticTrainStep(t2, n, samples_per_ray_capacity=64, use_graph=use_graph)
    bank, poses, dirs = (t.cpu().numpy() for t in (ds.rays, ds.poses, ds.directions))
    for step in range(3):
        l1 = float(fs1.step_sampled())
        b = O.sample_ray_batch(bank, poses, dirs, n, seed=seed, step=step)
        for k in ("rays_o", "rays_d", "noise"):
            np.testing.assert_array_equal(getattr(fs1, k).cpu().numpy(), b[k], err_msg=k)
        np.testing.assert_array_equal(fs1.gt.cpu().numpy(), b["rgb"])
        l2 = float(fs2.step(*(torch.from_numpy(b[k]).cuda() for k in ("rays_o", "rays_d", "rgb", "noise"))))
        assert abs(l1 - l2) < 2e-3 * max(l2, 1e-6), (step, l1, l2)
    assert int(fs1.counter[0]) > 500
    for p1, p2 in zip(m1.parameters(), m2.parameters()):
        assert float(((p1 - p2).abs() > 2e-3).float().mean()) < 2e-3
    if use_graph:
        assert fs1.kernels_per_replay_sampled == fs1.kernels_per_replay + 1 and fs1.replays_sampled == 3
        assert int(fs1.sample_step) == 3


def _shipped_lego_part():
    """The stored part of the reference's shipped, trained Lego deployment model (L=4 F=4 dense grid, 16-wide MLPs;
    oracle/kat_lego.py) as an NGP on the GPU, and the part's other fixture arrays."""
    from modules.networks import NGP
    from modules.utils import load_deployment_model
    from oracle import kat_lego
    P = kat_lego.load_part()
    model = NGP(scale=0.5, pos_encoder_type='hash', levels=4, feature_per_level=4, base_res=32, max_res=128,
                log2_T=21, xyz_net_width=16, rgb_net_width=16, rgb_net_depth=1).cuda()
    load_deployment_model(model, P["blob"])
    return model.eval(), P


def test_shipped_lego_model_renders_on_gpu():
    """Known-answer test on the CUDA path: the part of the reference's shipped, trained Lego deployment model loaded
    with load_deployment_model and rendered through render(test_time=True) must reproduce the oracle's golden image of
    the same rays (made with the full shipped table, tests/golden/make_golden.py)."""
    from modules.rendering import render
    model, P = _shipped_lego_part()
    pose = torch.from_numpy(P["pose"].copy()).cuda()
    directions = torch.from_numpy(P["directions"]).cuda()
    h, w = directions.shape[:2]
    dirs = directions.reshape(-1, 3)
    rays_d = dirs @ pose[:, :3].T
    rays_o = pose[:, 3].expand_as(rays_d).contiguous()
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.float16):
        out = render(model, rays_o, rays_d, test_time=True, T_threshold=1e-2, exp_step_factor=0.0)
    rgb = out['rgb'].float().reshape(h, w, 3).clamp(0, 1).cpu().numpy()   # render() composites onto white
    gold = np.clip(P["gold_rgb"] + (1 - P["gold_opacity"])[..., None], 0, 1)
    assert gold.shape == rgb.shape
    mse = float(((rgb - gold) ** 2).mean())
    psnr = -10 * np.log10(max(mse, 1e-12))
    assert psnr > 35.0, psnr          # fp16 autocast MLP; a layout mistake gives < 15 dB
    opacity = out['opacity'].float().reshape(h, w).cpu().numpy()
    gold_cov = float((P["gold_opacity"] > 0.5).mean())
    assert abs(float((opacity > 0.5).mean()) - gold_cov) < 0.03, gold_cov


@pytest.mark.parametrize("use_graph", [False, True])
def test_static_step_optimizer_overlap_equals_sync_step(lego_bitfield, use_graph):
    """overlap_optimizer=True (Adam of step k on a graph branch beside the marching of step k+1, flush() at the
    end) applies exactly the same sequence of updates as the default step."""
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer

    def build():
        torch.manual_seed(3)
        m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
        with torch.no_grad():
            m.pos_encoder.hash_table.mul_(2e3)
            m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
        return m, NGPTrainer(m, lr=1e-2)

    n = 2048
    batches = []
    for k in range(4):
        o, d = make_rays(n, seed=20 + k)
        g = torch.Generator(device='cuda').manual_seed(k)
        batches.append((torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(),
                        torch.rand(n, 3, device='cuda', generator=g), torch.rand(n, device='cuda', generator=g)))
    m1, t1 = build()
    fs1 = StaticTrainStep(t1, n, samples_per_ray_capacity=64, use_graph=use_graph)
    l1 = [float(fs1.step(*b)) for b in batches]
    m2, t2 = build()
    fs2 = StaticTrainStep(t2, n, samples_per_ray_capacity=64, use_graph=use_graph, overlap_optimizer=True)
    l2 = []
    for k, b in enumerate(batches):
        l2.append(float(fs2.step(*b)))
        assert fs2.pending and int(fs2.step_dev) == k      # the update of step k is still outstanding
        if k == 1:
            fs2.flush()                                      # e.g. before a density-grid update
            assert not fs2.pending and int(fs2.step_dev) == 2
    fs2.flush()
    fs2.flush()                                              # idempotent
    assert int(fs2.step_dev) == 4 == int(fs1.step_dev)
    for a, b in zip(l1, l2):
        assert abs(a - b) < 2e-3 * max(a, 1e-6), (l1, l2)
    for p1, p2 in zip(m1.parameters(), m2.parameters()):
        assert float(((p1 - p2).abs() > 2e-3).float().mean()) < 2e-3
    assert float(t2.flat_grad.abs().max()) == 0.0           # Adam zeroed the gradient buffer


def test_module_path_has_gradscaler_semantics(lego_bitfield):
    """NGPTrainer.step (train.py's default path) follows torch's GradScaler: an inf/NaN gradient skips the Adam
    update, halves the scale and does NOT advance Adam's step count; clean steps advance it; the LR schedule follows
    the iteration count (train.py:197-201)."""
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.trainer import NGPTrainer
    torch.manual_seed(1)
    m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
    with torch.no_grad():
        m.pos_encoder.hash_table.mul_(2e3)
        m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
    tr = NGPTrainer(m, lr=1e-2)
    o, d = make_rays(1024, seed=5)
    o, d = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    gt = torch.rand(1024, 3, device='cuda')
    tr.step(o, d, gt)
    assert float(tr.scale_state[0]) == 65536.0 and int(tr.hyper[3:].view(torch.int32)) == 1
    before = [p.detach().clone() for p in m.parameters()]
    tr.forward_backward(o, d, gt)
    tr.flat_grad[5] = float('inf')                      # an overflowing gradient
    tr.optimizer_step()
    assert float(tr.scale_state[0]) == 32768.0          # backoff x0.5
    assert int(tr.hyper[3:].view(torch.int32)) == 1     # Adam's t did not advance
    assert int(tr.step_dev) == 2                        # the LR schedule did
    for p, b in zip(m.parameters(), before):
        assert torch.equal(p, b)                        # update skipped
    assert float(tr.flat_grad.abs().max()) == 0.0       # gradients zeroed all the same
    tr.step(o, d, gt)
    assert int(tr.hyper[3:].view(torch.int32)) == 2 and abs(float(tr.hyper[2]) - 1 / 32768.0) < 1e-12
    assert any(not torch.equal(p, b) for p, b in zip(m.parameters(), before))
    # aliasing guard: casting / replacing a parameter is reported instead of silently training a stale copy
    m.rgb_net.output_layer.weight.data = m.rgb_net.output_layer.weight.data.clone()
    with pytest.raises(RuntimeError):
        tr.optimizer_step()


def _teacher_crop_psnr(teacher, model, ds, i, margin=4):
    """(PSNR of ``model``, PSNR of an all-white image) against the teacher's view ``i`` of ``ds``, both over the crop
    around the pixels the teacher covers (opacity > 0.01) widened by ``margin`` pixels."""
    from datasets.ray_utils import get_rays
    from modules.rendering import render
    w, h = ds.img_wh
    td = ds[i]
    rays_o, rays_d = get_rays(ds.directions, td['pose'])
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.float16):
        cover = render(teacher, rays_o, rays_d, test_time=True, T_threshold=1e-2, exp_step_factor=0.0)['opacity']
        rgb = render(model, rays_o, rays_d, test_time=True)['rgb']      # as train_vs_teacher evaluates
    cover = cover.float().reshape(h, w) > 0.01
    rows, cols = torch.nonzero(cover.any(1)).flatten(), torch.nonzero(cover.any(0)).flatten()
    r0, r1 = max(int(rows[0]) - margin, 0), min(int(rows[-1]) + 1 + margin, h)
    c0, c1 = max(int(cols[0]) - margin, 0), min(int(cols[-1]) + 1 + margin, w)
    gt = td['rgb'].reshape(h, w, 3)[r0:r1, c0:c1]
    rgb = rgb.float().clamp(0, 1).reshape(h, w, 3)[r0:r1, c0:c1]
    psnr = lambda x: float(-10.0 * torch.log10(((x - gt) ** 2).mean()))   # noqa: E731
    return psnr(rgb), psnr(torch.ones_like(gt))


def test_psnr_vs_teacher():
    """"PSNR vs ref" protocol (SURVEY.md §8c, bench.py's psnr leg: 2000 graph steps on 48 400x400 views): the stock fp16
    model trained on views of the part of the reference's shipped trained Lego model (the teacher) must reach >= 25 dB
    on held-out teacher views.  The part covers only a few per cent of a view, so PSNR is taken over the crop around
    the pixels it covers, where the object fills about as much of the image as the whole model does of a full view:
    there an all-white image, a model that learned only the background, stays ~16 dB below the gate."""
    from taichi_nerfs_b200.psnr import train_vs_teacher
    teacher, _ = _shipped_lego_part()
    r = train_vs_teacher(torch.device('cuda'), steps=2000, train_views=48, test_views=2, downsample=0.5,
                         teacher=teacher)
    assert r is not None
    crops = [_teacher_crop_psnr(teacher, r["model"], r["test_dataset"], i) for i in range(len(r["test_dataset"]))]
    psnr, white = (sum(c[k] for c in crops) / len(crops) for k in (0, 1))
    print(f"teacher-crop PSNR {psnr:.2f} dB, all-white {white:.2f} dB, whole views {r['psnr']:.2f} dB")
    assert white < 25.0 - 12.0, crops       # the gate's margin over a trivial answer
    assert psnr >= 25.0, crops


def test_update_density_grid_is_sync_free_and_matches_reference_statistics():
    """NGP.update_density_grid: zero host synchronisations (torch's sync debug mode raises on any), and the same
    occupancy statistics as the reference's op sequence (different random numbers, same distribution)."""
    from modules.networks import NGP
    torch.manual_seed(11)
    thr = 0.01 * 1024 / 3 ** 0.5

    def fresh():
        torch.manual_seed(11)
        m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
        with torch.no_grad():
            m.pos_encoder.hash_table.mul_(4e4)       # a non-trivial density field
        return m
    a, b = fresh(), fresh()
    a.update_density_grid(thr, warmup=True)          # first call builds the cached workspace / constants
    b.update_density_grid_reference(thr, warmup=True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            a.update_density_grid(thr, warmup=False)
        a.update_density_grid(thr, warmup=True)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for _ in range(3):
        b.update_density_grid_reference(thr, warmup=False)
    b.update_density_grid_reference(thr, warmup=True)
    occ_a = float(np.unpackbits(a.density_bitfield.cpu().numpy()).mean())
    occ_b = float(np.unpackbits(b.density_bitfield.cpu().numpy()).mean())
    assert 0.02 < occ_a < 0.98 and abs(occ_a - occ_b) < 0.02, (occ_a, occ_b)
    ga, gb = a.density_grid.float().cpu().numpy(), b.density_grid.float().cpu().numpy()
    assert abs(ga.mean() - gb.mean()) < 0.02 * abs(gb.mean())
    # identical draws on every rank: two models with the same parameters and update counter get identical grids
    c = fresh()
    c.update_density_grid(thr, warmup=True)
    for _ in range(3):
        c.update_density_grid(thr, warmup=False)
    c.update_density_grid(thr, warmup=True)
    assert torch.equal(a.density_bitfield, c.density_bitfield) and torch.equal(a.density_grid, c.density_grid)


def test_grouped_hash_backward_equals_single_launch(lego_bitfield):
    """The multi-GPU step scatters the hash gradient in level groups (fine hashed, coarse hashed, dense) so that a
    finished group's slice can be all-reduced behind the next group's kernel: the groups together must produce the
    single launch's gradient (each level's atomics are unchanged, levels own disjoint slices)."""
    from modules.networks import NGP
    from oracle.train_step import make_rays
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer

    def run(grouped):
        torch.manual_seed(3)
        m = NGP(scale=0.5, max_res=1024, half_opt=True).cuda()
        with torch.no_grad():
            m.pos_encoder.hash_table.mul_(2e3)
            m.density_bitfield.copy_(torch.from_numpy(lego_bitfield))
        tr = NGPTrainer(m, lr=1e-2)
        fs = StaticTrainStep(tr, 2048, samples_per_ray_capacity=64, use_graph=False, overlap_allreduce=grouped)
        assert fs.overlap_allreduce == grouped
        o, d = make_rays(2048, seed=21)
        g = torch.Generator(device='cuda').manual_seed(0)
        fs.rays_o.copy_(torch.from_numpy(o))
        fs.rays_d.copy_(torch.from_numpy(d))
        fs.gt.copy_(torch.rand(2048, 3, device='cuda', generator=g))
        fs.noise.copy_(torch.rand(2048, device='cuda', generator=g))
        from taichi_nerfs_b200._lib import check, load as L
        check(L().ngp_step_reset(fs.counter.data_ptr(), fs.loss_sum.data_ptr(), tr.found_inf.data_ptr(), None, None))
        fs._enqueue_march()
        fs._enqueue_network()
        torch.cuda.synchronize()
        return tr.flat_grad.clone(), fs
    g1, fs = run(False)
    g2, _ = run(True)
    groups = fs._level_groups()
    assert groups[0][1] == 16 and groups[-1][0] == 0 and sum(b - a for a, b in groups) == 16
    los = sorted(fs._slice_of_levels(a, b) for a, b in groups)
    assert los[0][0] == 0 and los[-1][1] == fs.P and all(x[1] == y[0] for x, y in zip(los, los[1:]))
    scale = float(g1.abs().max())
    assert scale > 0 and float((g1 - g2).abs().max()) <= 1e-5 * scale
