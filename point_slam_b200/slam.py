"""Single-process tracker / mapper scheduling (SURVEY.md section 8f rank 3).

The reference runs tracking and mapping as two OS processes plus a manager process hosting the neural point cloud
(`src/Point_SLAM.py:93-97,189-207`), but the Pipe hand-shake serialises them: the tracker blocks until the mapper has finished the
frame it waits for (`Tracker.py:264-266,379-380`, `Mapper.py:670-675,783`), every `npc.*` call is a pickled RPC and every map
update ships the whole cloud as a Python list (`Tracker.py:188-201`).  On one GPU the same schedule is a plain loop in ONE
process: for every frame, track (if the frame is not one of the first two), then -- every `mapping.every_frame` frames -- map.
The cloud, the features and the decoders are shared by reference; the tracker sees a map update the moment the mapper's kernels
have run (same stream), which is what `update_para_from_mapping` achieves with clones.

    slam = PointSLAM(cfg, renderer, npc, decoders, intr, device)
    for idx, color, depth, gt_c2w in frames:        # tensors on the device; gt_c2w (4,4) is used for frames 0 and 1 like the reference
        est_c2w = slam.process_frame(idx, color, depth, gt_c2w)

What is kept from the callers (cited lines) and what is not:
  * per frame: the dynamic radius maps from the colour gradient (`Tracker.py:237-248`, `Mapper.py:686-704`) and the gradient
    magnitude behind them, in one device pass (ops.frame_grad, the values synth.sobel_radius_map computes on the host);
  * tracking: constant-speed initialisation (`Tracker.py:279-286`), separate learning rates and the smallest-loss candidate
    (`:289-349`, inside graphed.FusedTracker), gt pose for idx <= 1 (`:275-276`), `sample_with_color_grad`: pixels drawn
    without replacement from the frame's gradient candidates (`:117-129`, `common.py:92-159`);
  * mapping: `add_neural_points` on `pixels_adding` random pixels + `pixels_based_on_color_grad` pixels drawn from the
    gradient candidates of the whole image with 0 < depth <= 5 m (ratio 15), added with the small radius, iteration count scaled
    by the number of added locations (`:404-406`), frustum feature selection (`:345`), keyframe selection 'global' or 'overlap'
    (`:170-235`), geometry -> colour stage switch (`:420-423`), keyframe insertion every `keyframe_every` frames (`:741-751`);
  * not reproduced: BA, exposure latents, colour refinement at the end of the run, visualiser / wandb / checkpoints (the
    checkpoint writer is `src/utils/Logger.py`), lazy_start.
"""
import numpy as np
import torch

from . import graphed as G
from . import ops
from .src import common


MAPPER_DEPTH_LIMIT = 5.0      # depth bound of the mapper's gradient pixels (DESIGN.md section 1, stated assumptions)


class PointSLAM:
    def __init__(self, cfg, renderer, npc, decoders, intr, device, mapping_iters=None, first_iters=None, max_keyframes=None):
        self.cfg, self.r, self.npc, self.dec, self.intr, self.dev = cfg, renderer, npc, decoders, intr, device
        t, m = cfg['tracking'], cfg['mapping']
        self.t, self.m = t, m
        self.every_frame = m['every_frame']
        self.keyframe_every = m['keyframe_every']
        self.window = m['mapping_window_size']
        self.n_kf_slots = max(self.window - 1, 1) if max_keyframes is None else max_keyframes     # selected keyframes + last keyframe
        self.iters = m['iters'] if mapping_iters is None else mapping_iters
        self.iters_first = m['iters_first'] if first_iters is None else first_iters
        self.tracker = G.FusedTracker(renderer, npc, decoders, intr, t['pixels'], device, edge=(t['ignore_edge_H'], t['ignore_edge_W']),
                                      lr=t['lr'], w_color=t['w_color_loss'], separate_lr=t['separate_LR'],
                                      sample_with_color_grad=t.get('sample_with_color_grad', False))
        self.mapper = None                     # built on the first mapped frame (needs a non-empty cloud for its capacity buffers)
        self.keyframes = []                    # dicts: idx, color, depth, c2w (est), dyn_r_query
        self.est = {}                          # idx -> (4,4) float32 device pose
        self.gen = torch.Generator(device=device).manual_seed(cfg.get('setup_seed', 1219))
        self.rng = np.random.default_rng(cfg.get('setup_seed', 1219))
        self.log = []

    # ---- helpers ------------------------------------------------------------------------------------------------------------
    def _radius_maps(self, color):
        """-> (r_add, r_query, mag) float64 (H,W) device maps of the frame (no host round trip)."""
        return ops.frame_grad(color, self.cfg)

    def _grad_pixels(self, mag, depth, n):
        """get_samples_with_pixel_grad of the mapper (common.py:92-159): n distinct pixels (flat indices) of the gradient candidates
        of the whole image with 0 < depth <= 5 m -- fewer when there are fewer candidates."""
        I = self.intr
        cand, count = ops.grad_candidates(mag, depth, n, ops.GRAD_RATIO, depth_max=MAPPER_DEPTH_LIMIT)
        pix = ops.pick_candidates(cand, count, n, I['W'], generator=self.gen)
        return pix[pix >= 0]

    def _cam_tensor(self, c2w):
        return common.get_tensor_from_camera(c2w.detach().cpu()).to(self.dev).float()

    def _c2w_from_cam(self, cam):
        c = common.get_camera_from_tensor(cam.detach())
        return torch.cat([c, torch.tensor([[0., 0., 0., 1.]], device=self.dev)], 0)

    # ---- tracking (Tracker.run, Tracker.py:222-382) ----------------------------------------------------------------------
    def track(self, idx, color, depth, r_query, gt_c2w):
        if idx <= 1 or self.t.get('gt_camera', False):
            return gt_c2w.to(self.dev).float()
        pre = self.est[idx - 1]
        if self.t.get('const_speed_assumption', True) and idx - 2 in self.est:
            init = (pre @ torch.linalg.inv(self.est[idx - 2])) @ pre                # :279-284
        else:
            init = pre
        cam = self._cam_tensor(init)
        gt_cam = self._cam_tensor(gt_c2w)
        if float(torch.dot(cam[:4], gt_cam[:4])) < 0:                               # :287-288
            cam[:4] *= -1
        tr = self.tracker
        tr.load_frame(color, depth, r_query, cam)
        tr.run(self.t['iters'])
        return self._c2w_from_cam(tr.best_cam)

    # ---- mapping (Mapper.run / optimize_map, Mapper.py:237-640, 642-790) ----------------------------------------------------
    def _select_keyframes(self, c2w, depth):
        n = len(self.keyframes)
        if n == 0:
            return []
        k = self.window - 2
        cand = list(range(n - 1))
        if self.m.get('keyframe_selection_method', 'overlap') == 'overlap' and cand:
            cand = self._overlap(c2w, depth, cand)
        sel = [int(v) for v in self.rng.permutation(np.array(cand, dtype=np.int64))[:max(min(len(cand), k), 0)]] if cand else []
        return sel + [n - 1]                                                       # + the last keyframe (:275-277)

    def _overlap(self, c2w, depth, cand, n_samples=8, pixels=200):
        """keyframe_selection_overlap (Mapper.py:170-235): keyframes into whose image points along 200 rays of the current
        frame project (device tensors instead of the per-keyframe numpy loop)."""
        I = self.intr
        pix = torch.randint(0, I['H'] * I['W'], (pixels,), device=self.dev, generator=self.gen)
        j, i = pix // I['W'], pix % I['W']
        ro, rd = common.get_rays_from_uv(i.float(), j.float(), c2w[:3, :4], I['fx'], I['fy'], I['cx'], I['cy'], self.dev)
        d = depth[j, i]
        keep = d > 0
        ro, rd, d = ro[keep], rd[keep], d[keep]
        if d.numel() == 0:
            return cand
        t = torch.linspace(0., 1., n_samples, device=self.dev)
        z = (d[:, None] * 0.8) * (1. - t) + (d[:, None] + 0.5) * t
        pts = (ro[:, None, :] + rd[:, None, :] * z[..., None]).reshape(-1, 3)
        out = []
        for kf in cand:
            w2c = torch.linalg.inv(self.keyframes[kf]['c2w'])
            pc = pts @ w2c[:3, :3].T + w2c[:3, 3]
            u = I['fx'] * (-pc[:, 0]) / (pc[:, 2] + 1e-5) + I['cx']
            v = I['fy'] * pc[:, 1] / (pc[:, 2] + 1e-5) + I['cy']
            inside = (u < I['W'] - 20) & (u > 20) & (v < I['H'] - 20) & (v > 20) & (pc[:, 2] < 0)
            if float(inside.float().mean()) > 0.0:
                out.append(kf)
        return out

    def map(self, idx, color, depth, c2w, r_add, r_query, mag):
        I, m, npc = self.intr, self.m, self.npc
        init = idx == 0
        n_add = m['pixels_adding']
        if init:                                                                   # Mapper.py:306-310
            n_add = int(torch.clamp(n_add * ((depth.median() / 2.5) ** 2), min=n_add, max=n_add * 3))
        added = 0
        for n_pix, grad in ((n_add, False), (m.get('pixels_based_on_color_grad', 0), True)):
            if n_pix <= 0:
                continue
            if grad:
                pix = self._grad_pixels(mag, depth, n_pix)
            else:
                pix = torch.randint(0, I['H'] * I['W'], (n_pix,), device=self.dev, generator=self.gen)
            j, i = pix // I['W'], pix % I['W']
            ro, rd = common.get_rays_from_uv(i.float(), j.float(), c2w[:3, :4], I['fx'], I['fy'], I['cx'], I['cy'], self.dev)
            gd = depth[j, i]
            keep = gd > 0
            added += int(npc.add_neural_points(ro[keep], rd[keep], gd[keep], color[j, i][keep], is_pts_grad=grad,
                                               dynamic_radius=r_add[j, i][keep] if self.r.use_dynamic_radius else None))
        iters = self.iters_first if init else int(np.clip(int(self.iters * added / 300), int(m['min_iter_ratio'] * self.iters), 2 * self.iters))
        sel = self._select_keyframes(c2w, depth)
        frames = [self.keyframes[k] for k in sel][-self.n_kf_slots:]
        cur = dict(color=color, depth=depth, c2w=c2w, dyn_r_query=r_query)
        # fixed number of frame slots (static shapes of the iteration graph): missing keyframes are filled with the current frame
        kfl = frames + [cur] * (self.n_kf_slots + 1 - len(frames))
        idxs = ops.frustum_select(npc.cloud_pos_tensor(), c2w, depth, I['H'], I['W'], I['fx'], I['fy'], I['cx'], I['cy'],
                                  edge=m['frustum_edge'], reuse=True)
        if self.mapper is None:
            lr = m['init' if init else 'stage']
            self.mapper = G.FusedMapper(self.r, npc, self.dec, I, m['pixels'], self.dev, w_color=m['w_color_loss'])
        # per-stage learning rates of this call: the first frame uses mapping.init, later ones mapping.stage (Mapper.py:424-432)
        ms = m['init' if init else 'stage']
        lrs = {k: (ms[k]['decoders_lr'], ms[k]['geometry_lr'], ms[k]['color_lr']) for k in ('geometry', 'color')}
        if lrs != self.mapper.stage_lrs:
            self.mapper.stage_lrs = lrs
            self.mapper.graphs = {}                       # learning rates are launch constants of the captured iterations
        self.mapper.begin_frame(idxs, kfl)
        n_geo = min((m['geo_iter_first'] if init else int(iters * m['geo_iter_ratio'])) + 1, iters)      # joint_iter <= ... (:420)
        self.mapper.run('geometry', n_geo)
        loss = self.mapper.run('color', iters - n_geo) if iters > n_geo else self.mapper.loss
        self.mapper.write_back()
        if idx % self.keyframe_every == 0:                                         # :741-751
            self.keyframes.append(dict(idx=idx, color=color, depth=depth, c2w=c2w.clone(), dyn_r_query=r_query))
        return added, iters, loss

    # ---- one frame of the sequence ------------------------------------------------------------------------------------------
    def process_frame(self, idx, color, depth, gt_c2w):
        """-> estimated (4,4) camera-to-world pose of frame idx.  Order of the reference's hand-shake: frame 0 is mapped before
        anything is tracked; a frame is tracked, then (every `every_frame` frames) mapped with the tracked pose."""
        r_add, r_query, mag = self._radius_maps(color)
        c2w = self.track(idx, color, depth, r_query, gt_c2w)
        self.est[idx] = c2w
        info = dict(idx=idx, mapped=False)
        if idx == 0 or idx % self.every_frame == 0:
            added, iters, loss = self.map(idx, color, depth, c2w, r_add, r_query, mag)
            info.update(mapped=True, added=added, iters=iters, points=self.npc.pts_num())
        self.log.append(info)
        return c2w
