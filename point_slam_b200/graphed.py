"""Launch-bound inner loops as CUDA graphs (SURVEY.md section 8f, "next #2").

The reference's optimisation iterations (Tracker.optimize_cam_in_batch, the joint loop of Mapper.optimize_map) issue ~450
tiny ATen kernels and ~10 stream synchronisations each, because rays are compacted with boolean masks (data-dependent
shapes).  Here the same iteration is written with STATIC shapes -- every sampled pixel stays in the batch, rays that the
reference would have dropped (no depth, depth outlier) carry depth 0 and zero loss weight -- so that one whole iteration
(pixel sampling on the device RNG, ray generation, fused render forward, loss, backward, Adam) is captured once into a
CUDA graph and replayed with a single launch.  Sums over the kept rays are identical to the reference's sums over the
compacted rays; the dropped rays cost a few percent of extra render work.
"""
import ctypes as C

import torch

from . import _lib as L
from . import ops
from .src import common


import os as _os
# composite + ray mask + loss + composite backward as one launch (psl_render_tail).  Mapping: one thread per ray over many CTAs.
# Tracking needs the batch mean of the gate first -> single-CTA kernel, which measured SLOWER than the four small kernels (39 vs
# ~25 us per iteration at 1500 rays): off by default.
FUSED_TAIL = _os.environ.get('PSL_FUSED_TAIL', '1') != '0'
FUSED_TAIL_TRACKER = _os.environ.get('PSL_FUSED_TAIL_TRACKER', '0') != '0'

def _masked_stats(depth, valid):
    """10*median and 1.2*max of the valid depths (Tracker.py:142-143 / Mapper.py:507-509) without compaction."""
    nan = torch.full_like(depth, float('nan'))
    med = torch.nanmedian(torch.where(valid, depth, nan))
    mx = torch.max(torch.where(valid, depth, torch.full_like(depth, -float('inf'))))
    return torch.minimum(10 * med, 1.2 * mx)


def _msum(x, mask):
    return torch.where(mask, x, torch.zeros_like(x)).sum()


def sample_uv_device(H0, H1, W0, W1, n, depth, color, device):
    """common.get_sample_uv (common.py:77-89) without host-side meshgrids: the same single torch.randint draw over the
    flattened window, pixel coordinates recovered arithmetically (identical values: the meshgrid holds exact integers)."""
    ww = W1 - W0
    idx = torch.randint((H1 - H0) * ww, (n,), device=device)
    jj = torch.div(idx, ww, rounding_mode='floor') + H0
    ii = idx - (jj - H0) * ww + W0
    return ii.float(), jj.float(), depth[jj, ii], color[jj, ii]


def tracker_iteration_static(renderer, npc, decoders, cam, gt_color, gt_depth, dyn_r_query, intr, n_pixels, device,
                             geo_feats, col_feats, cloud_pos, edge, w_color=0.5):
    """One tracking iteration, static shapes, no host synchronisation.  Returns the loss (backward already run)."""
    H, W = intr['H'], intr['W']
    c2w = common.get_camera_from_tensor(cam)
    i, j, b_depth, b_color = sample_uv_device(edge[0], H - edge[0], edge[1], W - edge[1], n_pixels, gt_depth, gt_color, device)
    rays_o, rays_d = common.get_rays_from_uv(i, j, c2w, intr['fx'], intr['fy'], intr['cx'], intr['cy'], device)
    b_rq = dyn_r_query[j.long(), i.long()] if dyn_r_query is not None else None
    with torch.no_grad():
        valid = b_depth > 0
        inside = valid & (b_depth <= _masked_stats(b_depth, valid))
        depth_in = torch.where(inside, b_depth, torch.zeros_like(b_depth))
    depth, unc, color, _ = renderer.render_batch_ray(npc, decoders, rays_d, rays_o.contiguous(), device, stage='color',
                                                     gt_depth=depth_in, npc_geo_feats=geo_feats, npc_col_feats=col_feats,
                                                     is_tracker=True, cloud_pos=cloud_pos, dynamic_r_query=b_rq,
                                                     _zero_depth=(None, None))
    unc = unc.detach()
    tmp = torch.abs(depth_in - depth) / torch.sqrt(unc + 1e-10)
    with torch.no_grad():
        ok = inside & (~torch.isnan(depth)) & (~torch.isnan(unc))
        mean_tmp = _msum(tmp, inside) / inside.sum().clamp_min(1)
        mask = ok & (tmp < 10 * mean_tmp)
    loss = _msum(torch.clamp(tmp, min=0.0, max=1e3), mask) + w_color * _msum(torch.abs(b_color - color), mask[:, None].expand(-1, 3))
    loss.backward()
    return loss.detach()


def stack_keyframes(keyframes):
    """list of keyframe dicts -> one dict of stacked device tensors (done once per mapped frame)."""
    out = dict(color=torch.stack([k['color'] for k in keyframes]), depth=torch.stack([k['depth'] for k in keyframes]),
               c2w=torch.stack([k['c2w'][:3, :4] for k in keyframes]), dyn_r_query=None)
    if keyframes[0].get('dyn_r_query') is not None:
        out['dyn_r_query'] = torch.stack([k['dyn_r_query'] for k in keyframes])
    return out


def mapper_iteration_static(renderer, npc, decoders, state, kfs, intr, n_pixels, device, stage, cloud_pos, w_color=0.1):
    """One mapping iteration over the stacked keyframes `kfs` (see stack_keyframes): static shapes, no host sync.
    All keyframes are sampled with one batched draw (the reference loops over them, Mapper.py:459-500)."""
    H, W = intr['H'], intr['W']
    idx = state.indices
    npc_geo, npc_col = state.npc_geo, state.npc_col
    npc_geo[idx] = state.geo
    npc_col[idx] = state.col
    K = kfs['depth'].shape[0]
    per = n_pixels // K
    pix = torch.randint(H * W, (K, per), device=device)
    jj = torch.div(pix, W, rounding_mode='floor')
    ii = pix - jj * W
    kk = torch.arange(K, device=device)[:, None].expand(K, per)
    b_depth = kfs['depth'][kk, jj, ii].reshape(-1)
    b_color = kfs['color'][kk, jj, ii].reshape(-1, 3)
    b_rq = kfs['dyn_r_query'][kk, jj, ii].reshape(-1) if kfs['dyn_r_query'] is not None else None
    dirs = torch.stack([(ii.float() - intr['cx']) / intr['fx'], -(jj.float() - intr['cy']) / intr['fy'],
                        -torch.ones(K, per, device=device)], -1)                       # common.py:49-50
    c2w = kfs['c2w']
    rays_d = torch.sum(dirs[..., None, :] * c2w[:, None, :3, :3], -1).reshape(-1, 3)   # common.py:53
    rays_o = c2w[:, None, :3, 3].expand(K, per, 3).reshape(-1, 3)
    with torch.no_grad():
        valid = b_depth > 0
        inside = valid & (b_depth <= _masked_stats(b_depth, valid))
        depth_in = torch.where(inside, b_depth, torch.zeros_like(b_depth))
    depth, unc, color, vmask = renderer.render_batch_ray(npc, decoders, rays_d, rays_o, device, stage, gt_depth=depth_in,
                                                         npc_geo_feats=npc_geo, npc_col_feats=npc_col, is_tracker=False,
                                                         cloud_pos=cloud_pos, dynamic_r_query=b_rq, _zero_depth=(None, None))
    m = inside & vmask & (~torch.isnan(depth))
    loss = _msum(torch.abs(depth_in - depth), m)
    if stage == 'color':
        loss = loss + w_color * _msum(torch.abs(b_color - color), m[:, None].expand(-1, 3))
    loss.backward()
    return loss.detach()


# ---------------------------------------------------------------------------------------------------------------------
# fused shells: the same iterations with the glue (sampling, gate, loss + its gradient, pose chain rule, Adam on the pose /
# the feature rows) done by the library's shell kernels (csrc/psl_shell.cu) and the render called without autograd.
# One tracking iteration is ~17 kernel launches (was ~290), one colour-stage mapping iteration ~40 (was ~145).
# ---------------------------------------------------------------------------------------------------------------------
def require_supported(cfg, who, tracker):
    """The graph shells implement the branch of Tracker.optimize_cam_in_batch / Mapper.optimize_map that the Replica and TUM
    configurations take.  Anything else must go through the autograd Renderer path (module swap, INTEGRATION.md section 1),
    which covers every branch -- refuse loudly instead of optimising a different loss."""
    bad = []
    if cfg['model']['encode_exposure']:
        bad.append('model.encode_exposure (per-frame exposure affine: Tracker.py:151-157, Mapper.py:531-548)')
    t, m = cfg.get('tracking', {}), cfg.get('mapping', {})
    if tracker:
        if not t.get('use_color_in_tracking', True):
            bad.append('tracking.use_color_in_tracking = False')
        if not t.get('handle_dynamic', True):
            bad.append('tracking.handle_dynamic = False (median gate, Tracker.py:167-169)')
        if t.get('depth_limit', False):
            bad.append('tracking.depth_limit')
    elif m.get('BA', False):
        bad.append('mapping.BA (pose optimisation inside the mapper, Mapper.py:377-392)')
    if bad:
        raise NotImplementedError(f'{who}: configuration not covered by the fused iteration shells: ' + '; '.join(bad) +
                                  ' -- use the Renderer / autograd path for this configuration')


def _render_settings(renderer, npc, decoders, stage, is_tracker):
    return decoders.settings(stage, renderer.N_surface, is_tracker, coef=renderer.sigmoid_coefficient,
                             near_surface=renderer.near_end_surface, far_surface=renderer.far_end_surface,
                             exposure_feat=None, radius_query=npc.get_radius_query())


def _sample(lib, pix, K, per, H, W, H0, W0, ww, cam, c2w, color, depth, dyn, intr, device):
    n = K * per
    rays_o = torch.empty(n, 3, device=device); rays_d = torch.empty(n, 3, device=device)
    b_depth = torch.empty(n, device=device); b_color = torch.empty(n, 3, device=device)
    r2 = torch.empty(n, dtype=torch.float64, device=device) if dyn is not None else None
    L.check(lib.psl_sample_rays(L.ptr(pix), K, per, H, W, H0, W0, ww, L.ptr(cam), L.ptr(c2w), L.ptr(color), L.ptr(depth),
                                L.ptr(dyn), intr['fx'], intr['fy'], intr['cx'], intr['cy'], L.ptr(rays_o), L.ptr(rays_d),
                                L.ptr(b_depth), L.ptr(b_color), L.ptr(r2), L.stream()), 'psl_sample_rays')
    depth_in = torch.empty(n, device=device)
    inside = torch.empty(n, dtype=torch.uint8, device=device)
    L.check(lib.psl_depth_gate(L.ptr(b_depth), n, L.ptr(depth_in), L.ptr(inside), L.stream()), 'psl_depth_gate')
    return rays_o, rays_d, b_color, r2, depth_in, inside


def _draw_beside(decoders, stage, device):
    """decoders.draw_no_neighbor_vectors on the forked stream (same position in the host's RNG call order: the Philox offsets are
    assigned at call time)."""
    if not ops.OVERLAP_BRANCHES:
        return decoders.draw_no_neighbor_vectors(stage, device)
    main, side = torch.cuda.current_stream(device), ops._side_stream(device)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        return decoders.draw_no_neighbor_vectors(stage, device)


_ZEROS32 = {}


def _zeros32(device):
    z = _ZEROS32.get(str(device))
    if z is None:
        z = _ZEROS32[str(device)] = torch.zeros(32, device=device)
    return z


def _join_side(device):
    if ops.OVERLAP_BRANCHES:
        torch.cuda.current_stream(device).wait_stream(ops._side_stream(device))


def tracker_iteration_fused(renderer, npc, decoders, cam, d_cam, gt_color, gt_depth, dyn_r_query, intr, n_pixels, device,
                            geo_feats, col_feats, cloud_pos, edge, loss_out, w_color=0.5, pack=None, prepacked=False, pix=None):
    """tracker_iteration_static on the shell kernels.  cam (7) plain device tensor; writes d_cam (7) and loss_out ().
    pix: the window-relative flat pixel indices select_uv would draw (common.py:66); None = drawn here from the device RNG."""
    lib = L.load()
    H, W = intr['H'], intr['W']
    H0, W0, ww = edge[0], edge[1], W - 2 * edge[1]
    n = n_pixels
    if pix is None:
        pix = torch.randint((H - 2 * H0) * ww, (n,), device=device)
    dyn = dyn_r_query if renderer.use_dynamic_radius else None
    rg, rc = _draw_beside(decoders, 'color', device)           # four tiny RNG kernels: on the forked stream, beside the sampling kernels
    rays_o, rays_d, b_color, r2, depth_in, inside = _sample(lib, pix, 1, n, H, W, H0, W0, ww, cam, None, gt_color, gt_depth, dyn,
                                                            intr, device)
    _join_side(device)
    st = _render_settings(renderer, npc, decoders, 'color', True)
    params = [ops._f32c(p) for p in decoders.kernel_params()]
    depth, var, rgb, _, sv = ops.render_forward(st, npc.spatial_hash(), params, rays_o, rays_d, depth_in, None, r2, rg, rc,
                                                cloud_pos, geo_feats, col_feats, None, True, colour_param_grads=False,
                                                geo_param_grads=False, pack=pack, prepacked=prepacked,
                                                tail=dict(mode=0, depth_in=depth_in, inside=inside, b_color=b_color, w_color=w_color,
                                                          loss_out=loss_out) if FUSED_TAIL_TRACKER else None)
    d_depth = d_rgb = None
    if not FUSED_TAIL_TRACKER:
        d_depth = torch.empty(n, device=device); d_rgb = torch.empty(n, 3, device=device)
        L.check(lib.psl_shell_loss(0, n, L.ptr(depth_in), L.ptr(inside), None, L.ptr(depth), L.ptr(var), L.ptr(rgb), L.ptr(b_color),
                                   w_color, L.ptr(loss_out), L.ptr(d_depth), L.ptr(d_rgb), L.stream()), 'psl_shell_loss')
    d_o, d_d, _, _, _, _ = ops.render_backward(sv, d_depth, None, d_rgb, True, True, False, False, False, [False] * L.N_PARAMS,
                                               pack=pack, repack=False if prepacked else True)
    L.check(lib.psl_pose_bwd(L.ptr(pix), n, H0, W0, ww, intr['fx'], intr['fy'], intr['cx'], intr['cy'], L.ptr(cam), L.ptr(d_o),
                             L.ptr(d_d), L.ptr(d_cam), L.stream()), 'psl_pose_bwd')


class AdamRows:
    """torch.optim.Adam state for `n_slots` rows of width `width` (psl_adam_rows)."""

    def __init__(self, n_slots, width, device, lr, betas=(0.9, 0.999), eps=1e-8):
        self.n, self.w, self.lr, self.betas, self.eps = int(n_slots), int(width), float(lr), betas, float(eps)
        self.grad = torch.zeros(n_slots, width, device=device)
        self.m = torch.zeros(n_slots, width, device=device)
        self.v = torch.zeros(n_slots, width, device=device)
        self.t = torch.zeros(1, dtype=torch.int32, device=device)

    def reset(self):
        self.grad.zero_(); self.m.zero_(); self.v.zero_(); self.t.zero_()

    def step(self, param, rows=None, zero_grad=True):
        L.check(L.load().psl_adam_rows(L.ptr(param), L.ptr(self.grad), L.ptr(self.m), L.ptr(self.v), L.ptr(rows), self.n, self.w,
                                       L.ptr(self.t), self.lr, self.betas[0], self.betas[1], self.eps, int(zero_grad), L.stream()),
                'psl_adam_rows')


def mapper_iteration_fused(renderer, npc, decoders, fs, kfs, intr, n_pixels, device, stage, cloud_pos, loss_out, w_color=0.1,
                           apply_adam=True, pix=None):
    """mapper_iteration_static on the shell kernels.  fs: FusedMapper state (full feature tensors updated in place by
    AdamRows through the row list, compact gradients through row_map).  apply_adam=False leaves the gradients in
    fs.adam_geo.grad / fs.adam_col.grad / fs.flat (tests)."""
    lib = L.load()
    H, W = intr['H'], intr['W']
    K = kfs['depth'].shape[0]
    per = n_pixels // K
    n = K * per
    color = stage == 'color'
    if pix is None:
        pix = torch.randint(H * W, (K, per), device=device)
    dyn = kfs['dyn_r_query'] if renderer.use_dynamic_radius else None
    rg, rc = _draw_beside(decoders, stage, device)
    rays_o, rays_d, b_color, r2, depth_in, inside = _sample(lib, pix, K, per, H, W, 0, 0, W, None, kfs['c2w'], kfs['color'],
                                                            kfs['depth'], dyn, intr, device)
    _join_side(device)
    st = _render_settings(renderer, npc, decoders, stage, False)
    params = [ops._f32c(p) for p in decoders.kernel_params()]
    depth, var, rgb, ray_mask, sv = ops.render_forward(st, npc.spatial_hash(), params, rays_o, rays_d, depth_in, None, r2, rg,
                                                       rc if rc is not None else _zeros32(device), cloud_pos,
                                                       fs.npc_geo, fs.npc_col if color else None, None, True,
                                                       colour_param_grads=color, geo_param_grads=False, pack=fs.pack,
                                                       prepacked='geometry', pack_backward=True,
                                                       tail=dict(mode=1, depth_in=depth_in, inside=inside, b_color=b_color if color else None,
                                                                 w_color=w_color, loss_out=loss_out) if FUSED_TAIL else None)
    d_depth = d_rgb = None
    if not FUSED_TAIL:
        d_depth = torch.empty(n, device=device)
        d_rgb = torch.empty(n, 3, device=device) if color else None
        L.check(lib.psl_shell_loss(1, n, L.ptr(depth_in), L.ptr(inside), L.ptr(ray_mask), L.ptr(depth), None, L.ptr(rgb),
                                   L.ptr(b_color), w_color, L.ptr(loss_out), L.ptr(d_depth), L.ptr(d_rgb), L.stream()), 'psl_shell_loss')
    needs = fs.needs if color else [False] * L.N_PARAMS
    ops.render_backward(sv, d_depth, None, d_rgb, False, False, True, color, False, needs, pack=fs.pack, repack=False,
                        flat_out=fs.flat if color else None,
                        scatter_to=(fs.row_map, fs.u_max, fs.adam_geo.grad, fs.adam_col.grad))
    if not apply_adam:
        return
    fs.adam_geo.step(fs.npc_geo, fs.rows)
    if color:
        fs.adam_col.step(fs.npc_col, fs.rows)
        fs.dec_opt.step()


def _reset_adam(opt):
    """Fresh-optimizer semantics (the reference builds a new Adam per frame) without reallocating capturable state."""
    for st in opt.state.values():
        for k, v in st.items():
            if torch.is_tensor(v):
                v.zero_()


class GraphedTracker:
    """Tracker.optimize_cam_in_batch x n_iters as replays of one captured CUDA graph."""

    def __init__(self, renderer, npc, decoders, intr, n_pixels, device, edge=(20, 20), lr=0.002, w_color=0.5):
        require_supported(npc.cfg, 'GraphedTracker', tracker=True)
        self.r, self.npc, self.dec, self.intr, self.n, self.dev, self.edge, self.w = renderer, npc, decoders, intr, n_pixels, device, edge, w_color
        H, W = intr['H'], intr['W']
        self.color = torch.zeros(H, W, 3, device=device)
        self.depth = torch.zeros(H, W, device=device)
        self.dyn = torch.zeros(H, W, dtype=torch.float64, device=device)
        self.cam = torch.zeros(7, device=device, requires_grad=True)
        self.opt = torch.optim.Adam([self.cam], lr=lr, capturable=True, fused=True)
        self.loss = torch.zeros((), device=device)
        self.graph = None

    def _iter(self):
        # the pose is the only optimised quantity: decoder/feature gradients (which the reference's autograd computes and
        # throws away) are not requested, so the backward kernel skips every weight-gradient phase
        self.opt.zero_grad(set_to_none=True)
        loss = tracker_iteration_static(self.r, self.npc, self.dec, self.cam, self.color, self.depth, self.dyn, self.intr, self.n,
                                        self.dev, self.npc.get_geo_feats(), self.npc.get_col_feats(), self.npc.cloud_pos_tensor(),
                                        self.edge, self.w)
        self.opt.step()
        self.loss.copy_(loss)

    def load_frame(self, color, depth, dyn, cam_init):
        self.color.copy_(color, non_blocking=True); self.depth.copy_(depth, non_blocking=True); self.dyn.copy_(dyn, non_blocking=True)
        with torch.no_grad():
            self.cam.copy_(cam_init)
        _reset_adam(self.opt)

    def capture(self):
        flags = [(p, p.requires_grad) for p in self.dec.parameters()]
        for p, _ in flags:
            p.requires_grad_(False)
        try:
            self._capture()
        finally:
            for p, f in flags:
                p.requires_grad_(f)

    def _capture(self):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        cam0 = self.cam.detach().clone()
        with torch.cuda.stream(s):
            for _ in range(2):
                self._iter()
        torch.cuda.current_stream().wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._iter()
        with torch.no_grad():
            self.cam.copy_(cam0)
        _reset_adam(self.opt)

    def run(self, n_iters):
        if self.graph is None:
            self.capture()
        for _ in range(n_iters):
            self.graph.replay()
        return self.loss


class _MapState:
    pass


class GraphedMapper:
    """The joint loop of Mapper.optimize_map as replays of ONE captured graph per stage for the whole run.

    The frustum-selected feature slices change size from frame to frame; to keep every shape static the index list is
    padded to a fixed capacity `u_max` with the index of a dummy extra feature row (row N of (N+1)-row copies of the feature
    tensors): padded slots scatter into / gather from that row, which no kNN index ever references, so they receive zero
    gradient and Adam leaves them at zero.  Graphs are re-captured only when the cloud size, the capacity or the spatial
    hash changes (e.g. after add_neural_points)."""

    def __init__(self, renderer, npc, decoders, intr, n_pixels, device, w_color=0.1, lr_dec=0.005, lr_geo=0.005, lr_col=0.005,
                 u_max=1 << 17):
        self.r, self.npc, self.dec, self.intr, self.n, self.dev, self.w = renderer, npc, decoders, intr, n_pixels, device, w_color
        require_supported(npc.cfg, 'GraphedMapper', tracker=False)
        self.lrs = (lr_dec, lr_geo, lr_col)
        self.loss = torch.zeros((), device=device)
        self.u_max = int(u_max)
        self.graphs = {}
        self.state = None
        self.key = None
        self.warm = False

    def _alloc(self, N, n_kf):
        H, W = self.intr['H'], self.intr['W']
        d = self.dev
        st = _MapState()
        st.indices = torch.full((self.u_max,), N, dtype=torch.int64, device=d)
        st.npc_geo = torch.zeros(N + 1, 32, device=d)
        st.npc_col = torch.zeros(N + 1, 32, device=d)
        st.geo = torch.zeros(self.u_max, 32, device=d, requires_grad=True)
        st.col = torch.zeros(self.u_max, 32, device=d, requires_grad=True)
        st.optimizer = torch.optim.Adam([{'params': list(self.dec.color_decoder.parameters()), 'lr': self.lrs[0]},
                                         {'params': [st.geo], 'lr': self.lrs[1]}, {'params': [st.col], 'lr': self.lrs[2]}],
                                        capturable=True, fused=True)
        self.state = st
        self.keyframes = dict(color=torch.zeros(n_kf, H, W, 3, device=d), depth=torch.zeros(n_kf, H, W, device=d),
                              c2w=torch.zeros(n_kf, 3, 4, device=d), dyn_r_query=torch.zeros(n_kf, H, W, dtype=torch.float64, device=d))
        self.graphs = {}

    def begin_frame(self, indices, keyframes):
        """indices: (U,) int64 rows of the feature tensors to optimise; keyframes: list of dicts (color, depth, c2w, dyn_r_query)."""
        N, U = self.npc.pts_num(), int(indices.shape[0])
        while U > self.u_max:
            self.u_max *= 2
        key = (N, self.u_max, len(keyframes), self.npc.storage_gen(), self.npc.spatial_hash().build_gen)
        if key != self.key:
            self._alloc(N, len(keyframes))
            self.key = key
        st = self.state
        self.n_used = U
        with torch.no_grad():
            st.indices.fill_(N)
            st.indices[:U] = indices
            st.npc_geo[:N] = self.npc.get_geo_feats()
            st.npc_col[:N] = self.npc.get_col_feats()
            st.geo.copy_(st.npc_geo[st.indices])
            st.col.copy_(st.npc_col[st.indices])
            for i, kf in enumerate(keyframes):
                self.keyframes['color'][i].copy_(kf['color']); self.keyframes['depth'][i].copy_(kf['depth'])
                self.keyframes['c2w'][i].copy_(kf['c2w'][:3, :4]); self.keyframes['dyn_r_query'][i].copy_(kf['dyn_r_query'])
        _reset_adam(st.optimizer)

    def _iter(self, stage):
        st = self.state
        st.optimizer.zero_grad(set_to_none=True)
        loss = mapper_iteration_static(self.r, self.npc, self.dec, st, self.keyframes, self.intr, self.n, self.dev, stage,
                                       self.npc.cloud_pos_tensor(), self.w)
        st.optimizer.step()
        st.npc_geo, st.npc_col = st.npc_geo.detach(), st.npc_col.detach()
        self.loss.copy_(loss)

    def run(self, stage, n_iters):
        done = 0
        if stage not in self.graphs:
            # lazy initialisation (optimizer state, kernel attributes, allocator) must happen OUTSIDE of the capture -- a
            # state tensor created while capturing would be re-zeroed by every replay.  This executes one real iteration.
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._iter(stage)
            torch.cuda.current_stream().wait_stream(s)
            done = 1
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):                      # capture records the iteration, it does not execute it
                self._iter(stage)
            self.graphs[stage] = g
        for _ in range(n_iters - done):
            self.graphs[stage].replay()
        return self.loss

    def write_back(self):
        """Optimised slices -> the neural point cloud (Mapper.py:605-610)."""
        st, U = self.state, self.n_used
        self.npc.update_geo_feats(st.geo.detach()[:U], st.indices[:U])
        self.npc.update_col_feats(st.col.detach()[:U], st.indices[:U])


class FusedTracker:
    """Tracker.optimize_cam_in_batch x n_iters (Tracker.py:89-186, loop of :332-349): every iteration is one replay of a graph
    of ~17 library kernels (tracker_iteration_fused + psl_pose_adam).  The decoder is frozen while tracking, so its operand
    images are packed once per frame.  separate_LR: the quaternion steps with lr/5 (Tracker.py:291-299); `best_cam` is the
    pose of the iteration with the smallest loss, which is what the reference keeps (candidate_cam_tensor, :340-343).
    sample_with_color_grad (tracking.sample_with_color_grad, Tracker.py:117-129): load_frame builds the frame's candidate set --
    the grad_ratio * n_pixels pixels of largest colour gradient, kept if inside the edge window with depth > 0
    (ops.grad_candidates) -- and every iteration draws its n_pixels distinct pixels from it (ops.pick_candidates, without
    replacement like the reference's np.random.choice); `picked` holds the last draw.  The candidate buffer has a fixed
    capacity, so one captured graph serves every frame.  Off: uniform pixels of the window (torch.randint, common.py:77-89)."""

    def __init__(self, renderer, npc, decoders, intr, n_pixels, device, edge=(20, 20), lr=0.002, w_color=0.5, separate_lr=True,
                 sample_with_color_grad=False, grad_ratio=ops.GRAD_RATIO):
        require_supported(npc.cfg, 'FusedTracker', tracker=True)
        self.r, self.npc, self.dec, self.intr, self.n, self.dev, self.edge, self.w = renderer, npc, decoders, intr, n_pixels, device, edge, w_color
        H, W = intr['H'], intr['W']
        self.sample_with_color_grad = bool(sample_with_color_grad)
        if self.sample_with_color_grad:
            lib = L.load()
            cap = ops.grad_capacity(n_pixels, H, W, grad_ratio)
            self.grad_ratio = int(grad_ratio)
            self.mag = torch.zeros(H, W, dtype=torch.float64, device=device)
            self.cand = torch.zeros(cap, dtype=torch.int64, device=device)
            self.cand_count = torch.zeros(1, dtype=torch.int32, device=device)
            self.cand_ws = torch.empty(lib.psl_grad_candidates_ws_bytes(H * W), dtype=torch.uint8, device=device)
            self.pick_ws = torch.empty(lib.psl_pick_candidates_ws_bytes(cap), dtype=torch.uint8, device=device)
            self.picked = torch.zeros(n_pixels, dtype=torch.int64, device=device)
        self.color = torch.zeros(H, W, 3, device=device)
        self.depth = torch.zeros(H, W, device=device)
        self.dyn = torch.zeros(H, W, dtype=torch.float64, device=device)
        self.cam = torch.zeros(7, device=device)
        self.lr, self.separate_lr = float(lr), bool(separate_lr)
        self.adam = AdamRows(1, 7, device, lr)
        self.loss = torch.zeros((), device=device)
        self.best_loss = torch.full((1,), 1e20, device=device)
        self.best_cam = torch.zeros(7, device=device)
        self.pack = ops.PackedDecoder(device)
        self.pix = None                       # fixed pixel batch (tests); None = device RNG per iteration
        self.graph = None
        self.key = None
        self.captures = 0

    def _window(self):
        H, W = self.intr['H'], self.intr['W']
        return (self.edge[0], H - self.edge[0], self.edge[1], W - self.edge[1])

    def _iter(self):
        pix = self.pix
        if pix is None and self.sample_with_color_grad:
            pix = ops.pick_candidates(self.cand, self.cand_count, self.n, self.intr['W'], window=self._window(), pix=self.picked,
                                      ws=self.pick_ws)
        tracker_iteration_fused(self.r, self.npc, self.dec, self.cam, self.adam.grad, self.color, self.depth, self.dyn, self.intr,
                                self.n, self.dev, self.npc.get_geo_feats(), self.npc.get_col_feats(), self.npc.cloud_pos_tensor(),
                                self.edge, self.loss, self.w, pack=self.pack, prepacked=True, pix=pix)
        a = self.adam
        L.check(L.load().psl_pose_adam(L.ptr(self.cam), L.ptr(a.grad), L.ptr(a.m), L.ptr(a.v), L.ptr(a.t),
                                       self.lr * (0.2 if self.separate_lr else 1.0), self.lr, a.betas[0], a.betas[1], a.eps,
                                       L.ptr(self.loss.reshape(1)), L.ptr(self.best_loss), L.ptr(self.best_cam),
                                       int(self.separate_lr), L.stream()), 'psl_pose_adam')

    def load_frame(self, color, depth, dyn, cam_init):
        self.color.copy_(color, non_blocking=True); self.depth.copy_(depth, non_blocking=True); self.dyn.copy_(dyn, non_blocking=True)
        if self.sample_with_color_grad:                     # the frame's candidate set (Tracker.py:117-129), once per frame
            ops.frame_grad(self.color, self.npc.cfg, maps=False, mag_out=self.mag)
            ops.grad_candidates(self.mag, self.depth, self.n, self.grad_ratio, window=self._window(), cand=self.cand,
                                count=self.cand_count, ws=self.cand_ws)
        self.cam.copy_(cam_init)
        self.adam.reset()
        self.best_loss.fill_(1e20)
        self.best_cam.copy_(self.cam)
        self.pack.pack(self.dec.kernel_params())           # the mapper may have updated the colour decoder since the last frame

    def _graph_key(self):
        # device buffers the captured kernels point at; the cloud may GROW without invalidating the graph (capacity buffers,
        # sizes read from device memory: ops.SpatialHash), only a re-allocation forces a re-capture
        return (self.npc.storage_gen(), self.npc.cloud_pos_tensor().data_ptr(), self.npc.get_geo_feats().data_ptr(),
                self.npc.get_col_feats().data_ptr())

    def capture(self):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        keep = [t.clone() for t in (self.cam, self.best_loss, self.best_cam)]
        with torch.cuda.stream(s):
            self._iter()                                   # lazy initialisation (caches, allocator) outside of the capture
        torch.cuda.current_stream().wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._iter()
        self.key = self._graph_key()
        self.captures += 1
        ops.warm_allocator(self.dev)                       # torch.cuda.graph emptied the allocator's cache on entry: refill it
        for t, k in zip((self.cam, self.best_loss, self.best_cam), keep):
            t.copy_(k)
        self.adam.reset()

    def run(self, n_iters):
        """-> loss of the last iteration (device scalar); the frame's pose estimate is `best_cam` (Tracker.py:340-349)."""
        if self.graph is None or self.key != self._graph_key():    # a buffer was re-allocated (capacity doubling): re-capture
            self.capture()
        for _ in range(n_iters):
            self.graph.replay()
        return self.loss


class FusedMapper:
    """The joint loop of Mapper.optimize_map (Mapper.py:408-568) on the shell kernels, one graph replay per iteration.

    Instead of the reference's slice tensors + index_put / gather round trip, the cloud's feature tensors are optimised IN
    PLACE: `rows` (u_max, padded with -1) lists the frustum-selected points, `row_map` is its inverse; the render backward
    scatters feature gradients straight into compact (u_max,32) buffers and psl_adam_rows applies torch.optim.Adam's update to
    exactly those rows of `npc.get_geo_feats()` / `get_col_feats()` (the reference writes its optimised slices back with
    update_geo_feats(feats, indices) at the end, Mapper.py:605-610 -- the same end state; tracker and mapper never overlap,
    Tracker.py:264-266).  The colour decoder keeps a torch fused Adam whose .grad tensors are views of one flat buffer that
    the weight-gradient kernels write.  Graphs are captured once per stage and survive new frusta AND cloud growth: every
    captured pointer is a capacity buffer (NeuralPointCloud.reserve, ops.SpatialHash), sizes that change are read from device
    memory; only a re-allocation (capacity doubling) forces a re-capture."""

    def __init__(self, renderer, npc, decoders, intr, n_pixels, device, w_color=0.1, lr_dec=0.005, lr_geo=0.005, lr_col=0.005,
                 u_max=1 << 17, stage_lrs=None):
        self.r, self.npc, self.dec, self.intr, self.n, self.dev, self.w = renderer, npc, decoders, intr, n_pixels, device, w_color
        self.lrs = (lr_dec, lr_geo, lr_col)
        # per-stage learning rates of the ONE Adam the reference builds per mapped frame (Mapper.py:394-402, 425-432):
        # {'geometry': (decoders_lr, geometry_lr, color_lr), 'color': (...)}; cfg['mapping']['stage'] (point_slam.yaml:76-84)
        ms = npc.cfg.get('mapping', {}).get('stage') if stage_lrs is None else stage_lrs
        self.stage_lrs = ({k: (ms[k]['decoders_lr'], ms[k]['geometry_lr'], ms[k]['color_lr']) for k in ('geometry', 'color')}
                          if isinstance(ms, dict) and isinstance(ms.get('color'), dict) else
                          (ms or {'geometry': self.lrs, 'color': self.lrs}))
        self.loss = torch.zeros((), device=device)
        require_supported(npc.cfg, 'FusedMapper', tracker=False)
        self.pack = ops.PackedDecoder(device)              # geometry images packed once per frame (frozen), colour images per iteration
        self.u_max = int(u_max)
        self.graphs = {}
        self.key = None
        self.warm = False
        self.n_used = 0
        self.captures = 0
        self.pix = None

    def _alloc(self, cap_rows, n_kf):
        H, W = self.intr['H'], self.intr['W']
        d = self.dev
        self.rows = torch.full((self.u_max,), -1, dtype=torch.int64, device=d)
        self.row_map = torch.full((cap_rows,), -1, dtype=torch.int32, device=d)
        self.adam_geo = AdamRows(self.u_max, 32, d, self.lrs[1])
        self.adam_col = AdamRows(self.u_max, 32, d, self.lrs[2])
        plist = self.dec.kernel_params()
        self.dec_params = [(nm, p) for nm, p in zip(ops.PARAM_ORDER, plist) if nm.startswith('c_') and p.requires_grad]
        self.flat = torch.zeros(sum(p.numel() for _, p in self.dec_params), device=d)
        off = 0
        for _, p in self.dec_params:
            p.grad = self.flat[off:off + p.numel()].view(p.shape)
            off += p.numel()
        self.dec_opt = torch.optim.Adam([p for _, p in self.dec_params], lr=self.lrs[0], capturable=True, fused=True)
        self.dec_opt.step()                                # zero gradients: creates the state tensors OUTSIDE of any capture
        _reset_adam(self.dec_opt)
        self.keyframes = dict(color=torch.zeros(n_kf, H, W, 3, device=d), depth=torch.zeros(n_kf, H, W, device=d),
                              c2w=torch.zeros(n_kf, 3, 4, device=d), dyn_r_query=torch.zeros(n_kf, H, W, dtype=torch.float64, device=d))
        self.graphs = {}
        self.warm = False

    def begin_frame(self, indices, keyframes):
        """indices: (U,) int64 rows of the feature tensors to optimise; keyframes: list of dicts (color, depth, c2w, dyn_r_query)."""
        N, U = self.npc.pts_num(), int(indices.shape[0])
        u_max = self.u_max
        while U > u_max:
            u_max *= 2
        self.npc_geo, self.npc_col = self.npc.get_geo_feats(), self.npc.get_col_feats()
        cap_rows = self.npc.feature_capacity()
        key = (self.npc.storage_gen(), cap_rows, u_max, len(keyframes), self.npc_geo.data_ptr(), self.npc_col.data_ptr(),
               self.npc.cloud_pos_tensor().data_ptr())
        if key != self.key:
            self.u_max = u_max
            self._alloc(cap_rows, len(keyframes))
            self.key = key
        self.n_used = U
        with torch.no_grad():
            self.rows.fill_(-1)
            self.rows[:U] = indices
            self.row_map.fill_(-1)
            self.row_map[indices] = torch.arange(U, dtype=torch.int32, device=self.dev)
            for i, kf in enumerate(keyframes):
                self.keyframes['color'][i].copy_(kf['color']); self.keyframes['depth'][i].copy_(kf['depth'])
                self.keyframes['c2w'][i].copy_(kf['c2w'][:3, :4]); self.keyframes['dyn_r_query'][i].copy_(kf['dyn_r_query'])
            self.pack.pack_geometry(self.dec.kernel_params())
        self.adam_geo.reset(); self.adam_col.reset()
        _reset_adam(self.dec_opt)
        off = 0
        for _, p in self.dec_params:                       # another optimizer's zero_grad(set_to_none) may have dropped the views
            p.grad = self.flat[off:off + p.numel()].view(p.shape)
            off += p.numel()

    @property
    def needs(self):
        want = {nm for nm, _ in self.dec_params}
        return [nm in want for nm in ops.PARAM_ORDER]

    def _iter(self, stage):
        lr_dec, lr_geo, lr_col = self.stage_lrs[stage]      # launch constants of this stage's graph
        self.adam_geo.lr, self.adam_col.lr = float(lr_geo), float(lr_col)
        for g in self.dec_opt.param_groups:
            g['lr'] = float(lr_dec)
        mapper_iteration_fused(self.r, self.npc, self.dec, self, self.keyframes, self.intr, self.n, self.dev, stage,
                               self.npc.cloud_pos_tensor(), self.loss, self.w, pix=self.pix)

    def run(self, stage, n_iters):
        done = 0
        if stage not in self.graphs:
            # lazy initialisation (optimizer state, kernel attributes, allocator) must happen OUTSIDE of the capture -- a
            # state tensor created while capturing would be re-zeroed by every replay.  This executes one real iteration.
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._iter(stage)
            torch.cuda.current_stream().wait_stream(s)
            done = 1
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):                      # capture records the iteration, it does not execute it
                self._iter(stage)
            self.graphs[stage] = g
            self.captures += 1
            ops.warm_allocator(self.dev)
        for _ in range(n_iters - done):
            self.graphs[stage].replay()
        return self.loss

    def write_back(self):
        """Mapper.py:605-610 (update_geo_feats / update_col_feats of the optimised rows): nothing to copy, the rows were
        optimised in place in the cloud's own feature tensors."""
        return self.rows[:self.n_used]
