"""GPU parity against vectors frozen from the reference's own CALLERS (tests/golden/caller_*.npz, render_img_*.npz, written by
oracle/make_golden_callers.py from the unmodified `Tracker.optimize_cam_in_batch`, `Mapper.optimize_map`, `Renderer.render_img`):

  * the fused iteration shells (graphed.FusedTracker / FusedMapper -- what bench.py times) fed the same pixels,
  * the drop-in `Renderer.render_img`,
  * and the reference's OWN Tracker / Mapper code (oracle/_ref, unmodified) running on top of the drop-in modules
    (the module swap of INTEGRATION.md section 1), replaying the same pixel draws.
Achieved errors go to $PSL_PARITY_JSON when it is set (tests/conftest.py writes it at session end)."""
import contextlib
import io
import types

import numpy as np
import pytest
import torch

from tests import callers as K
from tests import cases as C

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
INTR = C.INTR
E = K.Errors


def _t(a, dt=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device=DEV, dtype=dt)


def _objects(dataset='replica', **ov):
    from point_slam_b200.default_config import make_cfg
    from point_slam_b200.src.conv_onet import config as model_config
    from point_slam_b200.src.neural_point import NeuralPointCloud
    from point_slam_b200.src.utils.Renderer import Renderer
    cfg = make_cfg(dataset, DEV, **ov)
    decoders = model_config.get_model(cfg).to(DEV)
    P = C.load_params(False)
    decoders.load_state_dict({k: v for k, v in P.items() if k != 'color_decoder.embedder._B'}, strict=True)
    decoders.color_decoder.embedder._B = P['color_decoder.embedder._B'].to(DEV)
    scene = C.load_scene()
    npc = NeuralPointCloud(cfg)
    npc._cloud_pos = scene['cloud']
    npc._pts_num = scene['cloud'].shape[0]
    npc.geo_feats = scene['geo_feats'].to(DEV).clone()
    npc.col_feats = scene['col_feats'].to(DEV).clone()
    npc.index.add(npc._pos)
    return cfg, decoders, npc, Renderer


def _renderer(Renderer, cfg, intr=INTR):
    r = Renderer(cfg, None, types.SimpleNamespace(**{k: intr[k] for k in ('H', 'W', 'fx', 'fy', 'cx', 'cy')}))
    r.sigmoid_coefficient = 0.1
    return r


def _rand(decoders, g, it_holder):
    decoders.draw_no_neighbor_vectors = lambda stage, device: (_t(g[f'rand_geo{it_holder[0]}']),
                                                               _t(g[f'rand_col{it_holder[0]}']) if stage == 'color' else None)


_TRUTH = {}


def _pose_grad(case, g, k, got):
    """The pose gradient sums ~2000 terms of both signs (|grad| ~ 1e3 from terms ~1e5): the reference's own fp32 result is 1-2e-3
    away from the float64 evaluation of the same iteration.  Rule of tests/test_gpu_parity.py: the error against the float64
    truth may not exceed max(1e-4, 3 x the reference's own error against it)."""
    if k not in _TRUTH:
        _TRUTH[k] = K.tracker_truth(g, k)[1]
    gold = np.concatenate([g[f'grad_quad{k}'], g[f'grad_T{k}']])
    noise = C.rel_err(gold, _TRUTH[k])
    E.check(case, f'pose grad it{k} (vs oracle64; reference fp32 is {noise:.1e} away)', got, _TRUTH[k], 1e-4, noise=noise)
    E.check(case, f'pose grad it{k} (vs reference fp32)', got, gold, 1e-4, noise=noise)


# ---------------------------------------------------------------------------------------------------------------------
# fused shells
# ---------------------------------------------------------------------------------------------------------------------
def test_fused_tracker_matches_reference_optimize_cam_in_batch():
    from point_slam_b200 import graphed as G
    g = K.load('caller_tracker')
    cfg, dec, npc, Renderer = _objects()
    ren = _renderer(Renderer, cfg)
    edge = tuple(int(v) for v in g['edge'])
    ft = G.FusedTracker(ren, npc, dec, INTR, int(g['n_pixels']), DEV, edge=edge, lr=float(g['lr']), w_color=float(g['w_color']), separate_lr=True)
    ft.load_frame(_t(K.full_image(g['color_win'])), _t(K.full_image(g['depth_win'])), _t(K.full_radius(g['r_query_win']), torch.float64),
                  _t(g['cam0']))
    it = [0]
    _rand(dec, g, it)
    best = (1e30, None)
    for k in range(3):
        it[0] = k
        ft.pix = _t(g[f'pix{k}'], torch.int64)
        if k:                  # evaluate at the pose the reference evaluated (they agree to 4e-7; the loss is discontinuous in the
            ft.cam.copy_(_t(g[f'cam_after{k - 1}']))         # pose -- radius cut-offs, outlier mask -- so even that matters)
        cam_before = ft.cam.clone()
        ft._iter()
        torch.cuda.synchronize()
        E.check('caller_tracker', f'loss it{k}', ft.loss, g[f'loss{k}'], 1e-4)
        _pose_grad('caller_tracker', g, k, ft.adam.grad.view(-1))
        E.check('caller_tracker', f'pose after Adam it{k}', ft.cam, g[f'cam_after{k}'], 5e-6)
        if float(g[f'loss{k}']) < best[0]:
            best = (float(g[f'loss{k}']), cam_before)
    # the reference keeps the pose of the iteration with the smallest loss -- with separate_LR the pose that iteration rendered with
    assert torch.equal(ft.best_cam, best[1])


def _end_state(case, what, got, want, start):
    """End state after several Adam steps: the same rows moved, and all but a sliver of the moved entries agree to 1e-3 of the
    feature scale (entries whose gradient history is rounding noise take +-lr steps of either sign in each run)."""
    moved_w, moved_g = (want != start).any(1), (got != start).any(1)
    assert torch.equal(moved_w, moved_g), f'{what}: a different set of rows moved'
    scale = float(want.abs().max())
    frac = float(((got - want).abs() <= 1e-3 * scale)[moved_w].float().mean())
    E.rows.append(dict(case=case, quantity=what + ': share of moved entries within 1e-3 of the reference', err=1.0 - frac, limit=0.02,
                       flat_limit=0.0, fp32_noise=None, ok=frac >= 0.98))
    assert frac >= 0.98, (what, frac)


def _mapper_setup(g):
    cfg, dec, npc, Renderer = _objects()
    ren = _renderer(Renderer, cfg)
    frames = [dict(color=_t(K.full_image(g['color_win'][k])), depth=_t(K.full_image(g['depth_win'][k])), c2w=_t(g['c2w'][k]),
                   dyn_r_query=_t(K.full_radius(g['r_query_win'][k]), torch.float64)) for k in range(3)]
    return cfg, dec, npc, ren, frames


def _add_like_reference(npc, g, cur):
    """The map update optimize_map starts with (Mapper.py:311-319) on the recorded pixels; the fresh feature rows come from the
    device RNG, so they are overwritten with the rows the reference drew."""
    from point_slam_b200.src import common
    with K.replay_randint([g['pix_add']], DEV):
        ro, rd, gd, gc, i, j = common.get_samples(0, INTR['H'], 0, INTR['W'], g['pix_add'].shape[0], INTR['fx'], INTR['fy'], INTR['cx'],
                                                   INTR['cy'], cur['c2w'], cur['depth'], cur['color'], DEV, depth_filter=True, return_index=True)
    r_add = _t(K.full_radius(g['r_add_win'], fill=0.08), torch.float64)[j, i]
    n0 = npc.pts_num()
    k = npc.add_neural_points(ro, rd, gd, gc, dynamic_radius=r_add)
    assert 3 * int(k) == g['added_pos'].shape[0]
    # same kept rays; positions to an ulp (the rays are generated on the device here: torch's CUDA kernels contract a*b+c)
    assert float((npc.cloud_pos_tensor()[n0:].cpu() - torch.from_numpy(g['added_pos'])).abs().max()) < 1e-6
    npc.get_geo_feats()[n0:] = _t(g['added_geo'])
    npc.get_col_feats()[n0:] = _t(g['added_col'])
    return n0


def test_fused_mapper_matches_reference_optimize_map():
    from point_slam_b200 import graphed as G, ops
    g = K.load('caller_mapper')
    cfg, dec, npc, ren, frames = _mapper_setup(g)
    cur = frames[2]
    _add_like_reference(npc, g, cur)
    idx = ops.frustum_select(npc.cloud_pos_tensor(), g['c2w'][2], cur['depth'], INTR['H'], INTR['W'], INTR['fx'], INTR['fy'], INTR['cx'],
                             INTR['cy'], edge=-4)
    assert torch.equal(idx.cpu(), torch.from_numpy(g['indices']))
    U = idx.shape[0]
    fm = G.FusedMapper(ren, npc, dec, INTR, int(g['n_pixels']), DEV, w_color=float(g['w_color']))
    fm.begin_frame(idx, [frames[0], frames[1], cur])                 # the reference's frame order: keyframes, then the current frame
    geo0, col0 = npc.get_geo_feats()[idx].clone(), npc.get_col_feats()[idx].clone()
    it = [0]
    _rand(dec, g, it)
    names = [k for k, _ in dec.color_decoder.named_parameters()]
    for k in range(int(g['n_iters'])):
        it[0] = k
        stage = str(g['stages'][k])
        lr_dec, lr_geo, lr_col = fm.stage_lrs[stage]
        fm.adam_geo.lr, fm.adam_col.lr = lr_geo, lr_col
        for grp in fm.dec_opt.param_groups:
            grp['lr'] = lr_dec
        G.mapper_iteration_fused(ren, npc, dec, fm, fm.keyframes, INTR, int(g['n_pixels']), DEV, stage, npc.cloud_pos_tensor(), fm.loss,
                                 float(g['w_color']), apply_adam=False, pix=_t(g[f'pix{k}'], torch.int64))
        torch.cuda.synchronize()
        # Iteration 0 starts from the reference's state: strict.  From iteration 1 on the two runs are no longer at the same point:
        # Adam's first steps move every touched entry by ~lr * sign(g), and entries whose gradient is rounding noise get the sign
        # of that noise (the reference is not reproducible across GPUs either, README.md:210-211) -- bounded, not bit-comparable.
        lim, lim_l = (1e-4, 1e-4) if k == 0 else (2e-2, 2e-3)
        E.check('caller_mapper', f'loss it{k} ({stage})', fm.loss, g[f'loss{k}'], lim_l)
        E.check('caller_mapper', f'geo feature grad it{k}', fm.adam_geo.grad[:U], K.dense_rows(g[f'grad_geo_rows{k}'], g[f'grad_geo_vals{k}'], U),
                lim, noise=1.7e-4)
        assert float(fm.adam_geo.grad[U:].abs().max()) == 0.0
        fm.adam_geo.step(fm.npc_geo, fm.rows)
        if stage == 'color':
            E.check('caller_mapper', f'col feature grad it{k}', fm.adam_col.grad[:U],
                    K.dense_rows(g[f'grad_col_rows{k}'], g[f'grad_col_vals{k}'], U), lim, noise=1.7e-4)
            worst = 0.0
            for nm, p in zip(names, dec.color_decoder.parameters()):
                key = f'grad_dec{k}.{nm}'
                if key in g:
                    worst = max(worst, C.rel_err(p.grad.cpu(), g[key]))
            E.rows.append(dict(case='caller_mapper', quantity=f'worst colour-decoder grad it{k}', err=worst, limit=2e-2, flat_limit=1e-4,
                               fp32_noise=2.6e-4, ok=worst <= 2e-2))
            assert worst <= 2e-2, worst
            fm.adam_col.step(fm.npc_col, fm.rows)
            fm.dec_opt.step()
    torch.cuda.synchronize()
    want = geo0.cpu().clone(); want[torch.from_numpy(g['geo_after_rows'])] = torch.from_numpy(g['geo_after_vals'])
    _end_state('caller_mapper', 'geometry features after 4 iterations', npc.get_geo_feats()[idx].cpu(), want, geo0.cpu())
    want = col0.cpu().clone(); want[torch.from_numpy(g['col_after_rows'])] = torch.from_numpy(g['col_after_vals'])
    _end_state('caller_mapper', 'colour features after 4 iterations', npc.get_col_feats()[idx].cpu(), want, col0.cpu())
    worst = 0.0
    sd = dec.color_decoder.state_dict()
    for key, v in g.items():
        if key.startswith('dec_after.'):
            worst = max(worst, C.rel_err(sd[key.split('.', 1)[1]].cpu(), v))
    E.rows.append(dict(case='caller_mapper', quantity='worst colour-decoder tensor after 4 iterations', err=worst, limit=5e-2, flat_limit=1e-4,
                       fp32_noise=None, ok=worst <= 5e-2))
    assert worst <= 5e-2, worst


# ---------------------------------------------------------------------------------------------------------------------
# render_img (a3)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['replica', 'tum'])
def test_render_img_matches_reference(name):
    g = K.load(f'render_img_{name}')
    cfg, dec, npc, Renderer = _objects(name)
    H, W, fx, fy, cx, cy = g['intr']
    intr = dict(H=int(H), W=int(W), fx=float(fx), fy=float(fy), cx=float(cx), cy=float(cy))
    ren = _renderer(Renderer, cfg, intr)
    dec.draw_no_neighbor_vectors = lambda stage, device: (_t(g['rand_geo']), _t(g['rand_col']))
    d, u, c = ren.render_img(npc, dec, _t(g['c2w']), DEV, 'color', gt_depth=_t(g['gt_depth']), npc_geo_feats=npc.get_geo_feats(),
                             npc_col_feats=npc.get_col_feats(), dynamic_r_query=_t(g['r_query'], torch.float64), cloud_pos=npc.cloud_pos_tensor())
    assert d.dtype == torch.float64 and u.dtype == torch.float64 and c.dtype == torch.float32 and d.shape == (intr['H'], intr['W'])
    E.check(f'render_img_{name}', 'depth', d, g['depth'], 1e-4)
    E.check(f'render_img_{name}', 'colour', c, g['color'], 1e-4)
    E.check(f'render_img_{name}', 'uncertainty', u, g['uncertainty'], 5e-4)
    if name == 'replica':                                             # zero-depth pixels render depth 0 (Renderer.py:200-201)
        assert bool((d.reshape(-1)[_t(g['gt_depth']).reshape(-1) <= 0] == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
# the reference's own Tracker / Mapper code on the drop-in modules
# ---------------------------------------------------------------------------------------------------------------------
need_ref = pytest.mark.skipif(not K.have_reference_copy(),
                              reason='oracle/_ref missing: __graft_entry__.build() copies the reference sources there where it finds them')


@need_ref
def test_reference_tracker_runs_on_the_drop_in():
    """Unmodified src/Tracker.py:optimize_cam_in_batch (oracle/_ref) + drop-in NeuralPointCloud / POINT / Renderer on the B200,
    same pixels as the golden run -> same losses, pose gradients and poses as the unmodified reference on the CPU."""
    Tracker, _, ref_common, _ = K.install_module_swap()
    g = K.load('caller_tracker')
    cfg, dec, npc, Renderer = _objects()
    ren = _renderer(Renderer, cfg)
    cam0 = _t(g['cam0'])
    quad, T = cam0[:4].clone().requires_grad_(True), cam0[4:].clone().requires_grad_(True)
    lr = float(g['lr'])
    opt = K.recording_adam()([{'params': [T], 'lr': lr}, {'params': [quad], 'lr': lr * 0.2}])
    edge = [int(v) for v in g['edge']]
    me = types.SimpleNamespace(
        device=DEV, npc=npc, H=INTR['H'], W=INTR['W'], fx=INTR['fx'], fy=INTR['fy'], cx=INTR['cx'], cy=INTR['cy'], ignore_edge_H=edge[0],
        ignore_edge_W=edge[1], sample_with_color_grad=False, depth_limit=False, use_dynamic_radius=True,
        dynamic_r_query=_t(K.full_radius(g['r_query_win']), torch.float64), renderer=ren, decoders=dec,
        npc_geo_feats=npc.get_geo_feats().detach().clone(), npc_col_feats=npc.get_col_feats().detach().clone(),
        cloud_pos=npc.cloud_pos_tensor(), exposure_feat=None, handle_dynamic=True, use_color_in_tracking=True, w_color_loss=float(g['w_color']))
    gt_color, gt_depth = _t(K.full_image(g['color_win'])), _t(K.full_image(g['depth_win']))
    it = [0]
    _rand(dec, g, it)
    ref_common.torch = K.ReplayTorch([g[f'pix{k}'] for k in range(3)])
    try:
        for k in range(3):
            it[0] = k
            if k:
                with torch.no_grad():                # same evaluation point as the golden run (see the fused-tracker test)
                    quad.copy_(_t(g[f'cam_after{k - 1}'][:4])); T.copy_(_t(g[f'cam_after{k - 1}'][4:]))
            cam = torch.cat([quad, T], 0)
            loss, _, _ = Tracker.optimize_cam_in_batch(me, cam, gt_color, gt_depth, int(g['n_pixels']), opt)
            snap = opt.snapshots[-1]
            E.check('swap_tracker', f'loss it{k}', torch.tensor(loss), g[f'loss{k}'], 1e-4)
            _pose_grad('swap_tracker', g, k, torch.cat([snap[1][0], snap[0][0]]))
            E.check('swap_tracker', f'pose after Adam it{k}', torch.cat([quad, T]), g[f'cam_after{k}'], 5e-6)
    finally:
        ref_common.torch = torch


@need_ref
def test_reference_mapper_runs_on_the_drop_in():
    """Unmodified src/Mapper.py:optimize_map (oracle/_ref): add_neural_points, get_mask_from_c2w (the reference's numpy / cv2
    code on the drop-in's cloud_pos()), four joint iterations with the stage switch -- on the drop-in modules on the B200."""
    _, Mapper, ref_common, ref_mapper = K.install_module_swap()
    from point_slam_b200.default_config import make_cfg
    g = K.load('caller_mapper')
    cfg, dec, npc, ren, frames = _mapper_setup(g)
    cur = frames[2]
    n0 = npc.pts_num()
    orig_add = npc.add_neural_points

    def add_and_pin(*a, **kw):                       # the reference's rows for the appended points (device RNG differs from the CPU's)
        ret = orig_add(*a, **kw)
        assert npc.pts_num() - n0 == g['added_pos'].shape[0]
        npc.get_geo_feats()[n0:] = _t(g['added_geo'])
        npc.get_col_feats()[n0:] = _t(g['added_col'])
        return ret
    npc.add_neural_points = add_and_pin
    mcfg = make_cfg('replica', DEV)
    kf_dict = [dict(color=f['color'], depth=f['depth'], est_c2w=f['c2w'], gt_c2w=f['c2w'], dynamic_r_query=f['dyn_r_query']) for f in frames[:2]]
    me = types.SimpleNamespace(
        H=INTR['H'], W=INTR['W'], fx=INTR['fx'], fy=INTR['fy'], cx=INTR['cx'], cy=INTR['cy'], npc=npc, cfg=mcfg, device=DEV,
        keyframe_selection_method='global', mapping_window_size=3, keyframe_dict=kf_dict, save_selected_keyframes_info=False,
        mapping_pixels=int(g['n_pixels']), pixels_adding=int(g['pix_add'].shape[0]), pixels_based_on_color_grad=0, use_dynamic_radius=True,
        dynamic_r_add=_t(K.full_radius(g['r_add_win'], fill=0.08), torch.float64), dynamic_r_query=cur['dyn_r_query'], encode_exposure=False,
        frustum_feature_selection=True, frustum_edge=-4, fix_geo_decoder=True, fix_color_decoder=False, decoders=dec, BA=False,
        min_iter_ratio=0.95, geo_iter_first=400, geo_iter_ratio=0.4, n_img=10 ** 6, color_refine=False, vis_inside=False, renderer=ren,
        w_color_loss=float(g['w_color']), wandb=False, num_joint_iters=5, visualizer=types.SimpleNamespace(vis=lambda *a, **k: None),
        exposure_feat=None, gt_camera=False, save_rendered_image=False)
    me.get_mask_from_c2w = types.MethodType(Mapper.get_mask_from_c2w, me)
    n_it = int(g['n_iters'])
    draws = [g['pix_add']] + [g[f'pix{k}'][f] for k in range(n_it) for f in range(3)]
    ref_common.torch = K.ReplayTorch(draws)
    tw = K.TorchWithAdam(K.recording_adam())
    ref_mapper.torch = tw
    calls = [0]
    orig_render = ren.render_batch_ray

    def counted(*a, **kw):
        calls[0] += 1
        return orig_render(*a, **kw)
    ren.render_batch_ray = counted
    dec.draw_no_neighbor_vectors = lambda stage, device: (_t(g[f'rand_geo{calls[0] - 1}']),
                                                          _t(g[f'rand_col{calls[0] - 1}']) if stage == 'color' else None)
    np.random.seed(77)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            Mapper.optimize_map(me, 5, torch.tensor(5), cur['color'].cpu(), cur['depth'].cpu(), cur['c2w'], kf_dict, [0, 1], cur['c2w'])
    finally:
        ref_common.torch = torch
        ref_mapper.torch = torch
    opt = tw.made[-1]
    assert len(opt.snapshots) == n_it and calls[0] == n_it
    idx = torch.from_numpy(g['indices'])
    U = idx.shape[0]
    for k in range(n_it):
        snap = opt.snapshots[k]
        lim = 1e-4 if k == 0 else 2e-2                 # see test_fused_mapper_matches_reference_optimize_map
        E.check('swap_mapper', f'geo feature grad it{k}', snap[1][0], K.dense_rows(g[f'grad_geo_rows{k}'], g[f'grad_geo_vals{k}'], U), lim, noise=1.7e-4)
        if str(g['stages'][k]) == 'color':
            E.check('swap_mapper', f'col feature grad it{k}', snap[2][0], K.dense_rows(g[f'grad_col_rows{k}'], g[f'grad_col_vals{k}'], U), lim,
                    noise=1.7e-4)
        else:
            assert snap[2][0] is None
    scene = C.load_scene()
    geo0 = torch.cat([scene['geo_feats'], torch.from_numpy(g['added_geo'])])[idx]
    want = geo0.clone(); want[torch.from_numpy(g['geo_after_rows'])] = torch.from_numpy(g['geo_after_vals'])
    _end_state('swap_mapper', 'geometry features after optimize_map', npc.get_geo_feats()[idx.to(DEV)].cpu(), want, geo0)
    col0 = torch.cat([scene['col_feats'], torch.from_numpy(g['added_col'])])[idx]
    want = col0.clone(); want[torch.from_numpy(g['col_after_rows'])] = torch.from_numpy(g['col_after_vals'])
    _end_state('swap_mapper', 'colour features after optimize_map', npc.get_col_feats()[idx.to(DEV)].cpu(), want, col0)
