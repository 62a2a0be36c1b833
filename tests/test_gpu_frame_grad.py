"""The per-frame colour-gradient pass (csrc/psl_frame.cu) and what is built on it: the dynamic-radius maps against the host
restatement synth.sobel_radius_map, the candidate list against the oracle (oracle.grad_select.grad_candidates),
the draw without replacement, FusedTracker(sample_with_color_grad=True) and PointSLAM on the TUM configuration."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _frames():
    """One noise-free frame and one with depth noise and 5 % holes (the C4 frame kind), from two poses."""
    from point_slam_b200 import synth
    poses = synth.trajectory(40, seed=5)
    clean = synth.make_frame(poses[3], synth.TUM_INTRINSICS)
    noisy = synth.make_frame(poses[17], synth.TUM_INTRINSICS, noise=True, holes=0.05, seed=17)
    return {'clean': clean, 'noisy': noisy}


def _host_mag(color):
    """The unclipped magnitude inside synth.sobel_radius_map, same expressions."""
    g = color.astype(np.float64) @ np.array([0.2125, 0.7154, 0.0721])
    gy = np.zeros_like(g)
    gx = np.zeros_like(g)
    gy[1:-1, 1:-1] = ((g[2:, :-2] + 2 * g[2:, 1:-1] + g[2:, 2:]) - (g[:-2, :-2] + 2 * g[:-2, 1:-1] + g[:-2, 2:])) / 4.0
    gx[1:-1, 1:-1] = ((g[:-2, 2:] + 2 * g[1:-1, 2:] + g[2:, 2:]) - (g[:-2, :-2] + 2 * g[1:-1, :-2] + g[2:, :-2])) / 4.0
    return np.sqrt(gx ** 2 + gy ** 2)


@pytest.mark.parametrize('kind', ['clean', 'noisy'])
def test_frame_grad_matches_the_host_radius_maps(kind):
    from point_slam_b200 import ops, synth
    from point_slam_b200.default_config import make_cfg
    depth, color = _frames()[kind]
    for ds in ('tum', 'replica'):
        pc = make_cfg(ds, DEV)['pointcloud']
        r_add, r_query = synth.sobel_radius_map(color, pc['radius_add_max'], pc['radius_add_min'], pc['radius_query_ratio'],
                                                pc['color_grad_threshold'])
        g_add, g_query, g_mag = (t.cpu().numpy() for t in ops.frame_grad(torch.from_numpy(color).to(DEV), {'pointcloud': pc}))
        mag = _host_mag(color)
        errs = {k: float(np.abs(a - b).max()) for k, a, b in (('mag', g_mag, mag), ('r_add', g_add, r_add), ('r_query', g_query, r_query))}
        bits = {k: int((a != b).sum()) for k, a, b in (('mag', g_mag, mag), ('r_add', g_add, r_add), ('r_query', g_query, r_query))}
        print(f'{kind}/{ds}: largest |device - host| {errs}, differing values {bits}')
        assert all(e <= 1e-12 for e in errs.values()), errs
        assert (r_add < pc['radius_add_max']).any() and (r_add == pc['radius_add_max']).any()      # both branches of the map taken
    # NULL outputs: mag alone
    _, _, m2 = ops.frame_grad(torch.from_numpy(color).to(DEV), make_cfg('tum', DEV), maps=False)
    assert torch.equal(m2.cpu(), torch.from_numpy(g_mag))


@pytest.mark.parametrize('kind', ['clean', 'noisy'])
def test_grad_candidates_equal_the_oracle(kind):
    from oracle import grad_select as O
    from point_slam_b200 import ops
    from point_slam_b200.default_config import make_cfg
    depth, color = _frames()[kind]
    H, W = depth.shape
    d_dev = torch.from_numpy(depth).to(DEV)
    _, _, mag = ops.frame_grad(torch.from_numpy(color).to(DEV), make_cfg('tum', DEV), maps=False)
    quant = torch.round(mag * 20) / 20                  # a handful of levels: ties at every cut
    for m in (mag, quant):
        mh = m.cpu().numpy()
        for n, window, dmax in ((5000, (20, H - 20, 20, W - 20), None), (1000, None, 5.0), (300, (100, H - 100, 100, W - 100), 3.0)):
            cand, count = ops.grad_candidates(m, d_dev, n, 15, window=window, depth_max=dmax)
            ref = O.grad_candidates(mh, depth, n, 15, window=window, depth_max=dmax)
            c = int(count.item())
            assert c == ref.size, (n, window, dmax, c, ref.size)
            assert np.array_equal(cand[:c].cpu().numpy(), ref), (n, window, dmax)
            assert 0 < c <= 15 * n


def _pick_graph(cand, count, n, W, window):
    from point_slam_b200 import ops
    pix = torch.zeros(n, dtype=torch.int64, device=DEV)
    ops.pick_candidates(cand, count, n, W, window=window, pix=pix)           # warm-up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.pick_candidates(cand, count, n, W, window=window, pix=pix)
    return g, pix


def test_pick_candidates_draws_without_replacement_and_uniformly():
    from scipy import stats
    H, W = 480, 640
    window = (20, H - 20, 30, W - 30)
    ww = W - 60
    cap, n, count_val = 600, 12, 80
    rng = np.random.default_rng(0)
    inside = np.array([y * W + x for y in range(20, H - 20) for x in range(30, W - 30)])
    full = np.sort(rng.choice(inside, cap, replace=False))
    cand = torch.from_numpy(full).to(DEV)
    count = torch.tensor([count_val], dtype=torch.int32, device=DEV)
    g, pix = _pick_graph(cand, count, n, W, window)
    as_rel = lambda p: (p // W - 20) * ww + (p % W - 30)
    valid = set(as_rel(full[:count_val]).tolist())
    hits = np.zeros(count_val)
    slot_of = {v: i for i, v in enumerate(as_rel(full[:count_val]).tolist())}
    R = 4000
    torch.manual_seed(11)
    draws = []
    for _ in range(R):
        g.replay()
        draws.append(pix.clone())
    for p in torch.stack(draws).cpu().numpy():
        assert np.unique(p).size == n and set(p.tolist()) <= valid
        for v in p:
            hits[slot_of[int(v)]] += 1
    expected = R * n / count_val
    chi2 = float(((hits - expected) ** 2 / expected).sum())
    bound = float(stats.chi2.ppf(1 - 1e-6, count_val - 1))
    print(f'chi-square {chi2:.1f} over {count_val - 1} dof (bound {bound:.1f}); frequency range {hits.min() / R:.4f}..{hits.max() / R:.4f} '
          f'(n/count = {n / count_val:.4f})')
    assert chi2 < bound
    # a fixed seed reproduces the draws
    torch.manual_seed(11)
    g.replay()
    assert torch.equal(pix, draws[0])
    # the same graph with another count read from device memory: fewer candidates than samples -> all of them, then -1
    count.fill_(5)
    g.replay()
    p = pix.cpu().numpy()
    assert sorted(p[:5].tolist()) == sorted(as_rel(full[:5]).tolist()) and (p[5:] == -1).all()
    count.fill_(cap)
    g.replay()
    p = pix.cpu().numpy()
    assert np.unique(p).size == n and set(p.tolist()) <= set(as_rel(full).tolist())


def _tum_scene():
    import bench
    return bench, bench.GpuScene(0, DEV, bench.CONFIGS['c4'], 200000, 3)


def test_fused_tracker_colour_gradient_sampling_changes_only_the_pixels():
    """Pixels drawn by psl_pick_candidates inside the captured graph, recorded, and given as `pix` to a uniform-sampling tracker on
    the same frame and pose: loss, pose gradient and the pose after the Adam step are bit-identical.  One capture serves
    frames with different candidate counts."""
    from point_slam_b200 import graphed as G, ops
    bench, scene = _tum_scene()
    npc, dec, ren = scene.npc, scene.decoders, scene.renderer
    n, edge = 1500, (20, 20)
    H, W = bench.INTR['H'], bench.INTR['W']
    cam0 = bench.cam_tensor_from_c2w(scene.frames_host[bench.N_KEYFRAMES]['c2w'], 0.01, scene.rng).to(DEV)
    cur = scene.resident[0]
    a = G.FusedTracker(ren, npc, dec, bench.INTR, n, DEV, edge=edge, sample_with_color_grad=True)
    b = G.FusedTracker(ren, npc, dec, bench.INTR, n, DEV, edge=edge)
    a.load_frame(cur['color'], cur['depth'], cur['dyn_r_query'], cam0)
    a.capture()
    b.pix = torch.zeros(n, dtype=torch.int64, device=DEV)
    b.load_frame(cur['color'], cur['depth'], cur['dyn_r_query'], cam0)
    b.capture()
    a.load_frame(cur['color'], cur['depth'], cur['dyn_r_query'], cam0)
    torch.manual_seed(21)
    a.run(1)
    b.pix.copy_(a.picked)
    b.load_frame(cur['color'], cur['depth'], cur['dyn_r_query'], cam0)
    torch.manual_seed(21)
    torch.randint(2 ** 31 - 1, (a.cand.numel(),), dtype=torch.int32, device=DEV)   # the key draw a's graph made: same RNG offsets after it
    b.run(1)
    torch.cuda.synchronize()
    cand = a.cand[:int(a.cand_count.item())]
    rel = (cand // W - edge[0]) * (W - 2 * edge[1]) + cand % W - edge[1]
    assert torch.isin(a.picked, rel).all() and torch.unique(a.picked).numel() == n
    assert torch.equal(a.loss, b.loss), (a.loss, b.loss)
    assert torch.equal(a.adam.grad, b.adam.grad)
    assert torch.equal(a.cam, b.cam) and float(a.adam.grad.abs().sum()) > 0
    # the pixels are not uniform ones: they sit on the largest gradients
    _, _, mag = ops.frame_grad(cur['color'], npc.cfg, maps=False)
    jj, ii = a.picked // (W - 2 * edge[1]) + edge[0], a.picked % (W - 2 * edge[1]) + edge[1]
    assert float(mag[jj, ii].mean()) > 3 * float(mag[edge[0]:H - edge[0], edge[1]:W - edge[1]].mean())
    # several frames, different candidate counts, one capture
    counts = []
    for k, cut in ((1, None), (2, None), (0, 0.7)):
        f = scene.resident[k]
        depth = f['depth'].clone()
        if cut is not None:
            depth[:, : int(W * cut)] = 0.0                  # most candidates lose their depth
        a.load_frame(f['color'], depth, f['dyn_r_query'], cam0)
        a.run(3)
        counts.append(int(a.cand_count.item()))
        assert torch.isfinite(a.loss) and torch.isfinite(a.best_cam).all()
    print('candidate counts per frame:', counts)
    assert len(set(counts)) == 3 and min(counts) > 0
    assert a.captures == 1


def test_point_slam_tum_runs_on_device_maps_and_gradient_pixels(monkeypatch):
    """PointSLAM on the TUM configuration (tracking.sample_with_color_grad on) with gradient-selected mapping pixels: the radius
    maps come from the device (the host path is never called), the tracker graph is captured once, the schedule is the
    reference's and the tracked poses stay within 3 cm of the ground truth."""
    import types
    from point_slam_b200 import synth
    from point_slam_b200.default_config import make_cfg
    from point_slam_b200.slam import PointSLAM
    from point_slam_b200.src.neural_point import NeuralPointCloud
    from point_slam_b200.src.utils.Renderer import Renderer
    import bench

    def _refuse(*a, **k):
        raise AssertionError('PointSLAM called the host radius maps')
    monkeypatch.setattr(synth, 'sobel_radius_map', _refuse)
    intr = bench.INTR
    cfg = make_cfg('tum', DEV, **{'mapping.every_frame': 2, 'mapping.keyframe_every': 2, 'mapping.mapping_window_size': 4,
                                  'mapping.pixels': 2000, 'mapping.pixels_adding': 6000, 'mapping.pixels_based_on_color_grad': 500,
                                  'tracking.pixels': 1500, 'tracking.iters': 40, 'tracking.ignore_edge_W': 40, 'tracking.ignore_edge_H': 40})
    assert cfg['tracking']['sample_with_color_grad']
    dec = bench.build_decoders(cfg, DEV)
    npc = NeuralPointCloud(cfg)
    npc.reserve(200000)
    ren = Renderer(cfg, None, types.SimpleNamespace(**{k: intr[k] for k in ('H', 'W', 'fx', 'fy', 'cx', 'cy')}))
    ren.sigmoid_coefficient = 0.1
    slam = PointSLAM(cfg, ren, npc, dec, intr, DEV, mapping_iters=100, first_iters=500)
    assert slam.tracker.sample_with_color_grad
    poses = synth.trajectory(400, seed=3)[:8]
    errs = []
    for idx in range(8):
        depth, color = synth.make_frame(poses[idx], intr)
        gt = torch.from_numpy(poses[idx]).float().to(DEV)
        est = slam.process_frame(idx, torch.from_numpy(color).to(DEV), torch.from_numpy(depth).to(DEV), gt)
        errs.append(float((est[:3, 3] - gt[:3, 3]).norm()))
    torch.cuda.synchronize()
    log = slam.log
    print('pose errors (m):', [round(e, 4) for e in errs], 'added:', [e.get('added') for e in log])
    assert [e['mapped'] for e in log] == [True, False, True, False, True, False, True, False]
    assert log[0]['added'] > 3000 and npc.pts_num() == 3 * sum(e.get('added', 0) for e in log)
    assert all(np.isfinite(errs)) and max(errs) < 0.03, errs
    assert slam.tracker.captures == 1
    assert int(slam.tracker.cand_count.item()) > 0
