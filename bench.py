#!/usr/bin/env python
"""bench.py -- Point-SLAM render hot path on B200: ray-samples/sec (render + kNN + MLP), frames/sec.

    python bench.py --gpus 1 --steps 5 --warmup 3                    # CUDA path (this repo), workload C2
    python bench.py --config c3                                      # other BASELINE.json configs: c1, c3, c4
    python bench.py --impl reference --steps 3 --warmup 1            # the reference algorithm on the host cores (CPU oracle port)
    python bench.py --dump-outputs /tmp/out                          # + the outputs of the last timed step as /tmp/out/<name>.npy

Workloads (BASELINE.json `configs`; shapes from the reference's YAML files, see SURVEY.md section 8):
  c2 (default, the configuration `metric` is quoted on): one STEP = the hot-path work of one Replica-config frame:
     40 tracking iterations x 1500 rays (render fwd + loss + bwd to the 7-d pose + Adam, Tracker.py:89-186), then the map update
     of a mapped frame -- add_neural_points on 6000 + 1000 pixels (Mapper.py:306-331), frustum feature selection
     (Mapper.py:345) -- and the per-frame share of mapping, 300/5 = 60 iterations x 5000 rays over the current frame + 4
     keyframes (25 geometry-stage then 35 colour-stage iterations: `joint_iter <= int(n * 0.4)`, Mapper.py:420; bwd to the
     frustum-selected feature rows and the colour decoder + Adam), S = 5, 500k-point cloud, 640x480 synthetic RGB-D frames.
     The map update runs EVERY step (the reference maps every 5th frame), so its cost is over-weighted five-fold.
  c4: TUM-fr1_desk-like tracking only: 200 iterations x 5000 rays, noisy depth + 5 % holes, rel-pos encoding off (tum.yaml).
  c1 / c3: forward render of one ray batch (1000 rays x 5 samples vs 50k points; 5000 rays x 32 samples vs 2M points).
`value` = ray-samples per second with the inputs already in HBM; `e2e` = the same step fed from pinned HOST memory (frame /
ray batch H2D, pose + loss / rendered pixels D2H inside the timed region).
Multi-GPU (`--gpus N`, torchrun): one independent scene per GPU (BASELINE config C5, the reference's SLURM array), no
data-path collective -> weak scaling; `--share-map` adds the design's one collective (NCCL broadcast of the map delta from
rank 0 after its map update, point_slam_b200/parallel.py) to every step.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from point_slam_b200 import synth                                    # noqa: E402
from point_slam_b200.default_config import make_cfg                  # noqa: E402
from point_slam_b200 import iteration as IT                          # noqa: E402

INTR = synth.TUM_INTRINSICS
N_KEYFRAMES = 4
FLOP_FWD = {True: 397894, False: 225382}     # SURVEY.md section 8d: forward FLOP per sample with / without the rel-pos neighbour MLP
TC_MAC = {True: 182956, False: 96700}        # colour-branch MACs per sample on the tensor cores (trunk + neighbour MLP / trunk)

CONFIGS = {
    # mode, dataset cfg, points, S, (track iters, rays), (map iters, rays), edge, noise, holes
    'c2': dict(mode='slam', dataset='replica', points=500000, S=5, track=(40, 1500), map=(60, 5000), edge=100, noise=False, holes=0.0,
               name='C2 Replica-office0-like frame'),
    'c4': dict(mode='track', dataset='tum', points=500000, S=5, track=(200, 5000), map=None, edge=20, noise=True, holes=0.05,
               name='C4 TUM-fr1_desk-like tracking only'),
    'c1': dict(mode='render', dataset='replica', points=50000, S=5, rays=1000, name='C1 single-batch render'),
    'c3': dict(mode='render', dataset='replica', points=2000000, S=32, rays=5000, name='C3 2M-point cloud, MLP-decode roofline'),
    # end-of-run re-render (Mapper.py:826-876): one step = FRAMES_PER_STEP full 640x480 images from their poses, frames sharded over the
    # ranks (frame r, r + N, ...) against the replicated cloud -> STRONG scaling (fixed total work); one all_reduce of the metrics per step
    'rerender': dict(mode='rerender', dataset='replica', points=500000, S=5, frames=8, name='frame-parallel re-render of 8 full 640x480 frames'),
}


def geo_iters(n_map):
    """Geometry-stage iterations of a mapping call of n_map iterations: joint_iter <= int(n * geo_iter_ratio), Mapper.py:420."""
    return min(int(n_map * 0.4) + 1, n_map)


def workload_config(name, points):
    """The `config` object of the JSON line -- identical for the CUDA arm and the reference arm."""
    c = CONFIGS[name]
    if c['mode'] == 'render':
        return {'workload': f"{c['name']}: {c['rays']} rays x {c['S']} samples, {points} pts, forward render (kNN + decode + composite)",
                'points': points, 'rays': c['rays'], 'S': c['S'], 'parallelism': 'scene-per-gpu'}
    if c['mode'] == 'rerender':
        return {'workload': f"{c['name']} (render_img: 307200 rays x {c['S']} samples each), {points} pts, frames sharded over the GPUs",
                'points': points, 'frames_per_step': c['frames'], 'S': c['S'], 'parallelism': 'frame-parallel'}
    w = f"{c['name']}: {c['track'][0]} track it x {c['track'][1]} rays"
    mix = {'track_iters': c['track'][0], 'track_rays': c['track'][1]}
    if c['map']:
        g = geo_iters(c['map'][0])
        w += (f" + map update (add_neural_points 6000+1000 px, frustum selection) + {c['map'][0]} map it x {c['map'][1]} rays "
              f"({g} geometry-stage, {c['map'][0] - g} colour-stage)")
        mix.update({'map_iters': c['map'][0], 'map_rays': c['map'][1], 'geometry_stage_iters': g})
    w += f", S={c['S']}, {points} pts, 640x480"
    return {'workload': w, 'points': points, 'iteration_mix': mix, 'parallelism': 'scene-per-gpu'}


DUMP_ROWS = 1 << 16          # --dump-outputs: a longer output is stored as a fixed seeded sample of this many rows
DUMP_LIMIT = 64 << 20        # bytes of all dumped arrays together


def sample_rows(t, seed=0):
    """t, or a fixed seeded sample of DUMP_ROWS of its rows (kept in row order) when it has more."""
    if t.shape[0] <= DUMP_ROWS:
        return t
    sel = np.sort(np.random.default_rng(seed).choice(t.shape[0], DUMP_ROWS, replace=False))
    return t[torch.from_numpy(sel).to(t.device)]


def dump_outputs(path, arrays):
    """One path/<name>.npy per array: float64 arrays and integer ones (row indices) as float64, everything else as float32."""
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        host[name] = a.astype(np.float64 if a.dtype == np.float64 or np.issubdtype(a.dtype, np.integer) else np.float32)
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_LIMIT, f'--dump-outputs: {total} bytes, more than {DUMP_LIMIT}'
    os.makedirs(path, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(path, f'{name}.npy'), a)


def load_decoder_state():
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'decoders_base.npz'))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def make_frames(n, seed, noise=False, holes=0.0):
    poses = synth.trajectory(n, seed=seed)
    frames = []
    for k in range(n):
        depth, color = synth.make_frame(poses[k], INTR, noise=noise, holes=holes, seed=k)
        r_add, rq = synth.sobel_radius_map(color)
        frames.append(dict(c2w=poses[k], depth=depth, color=color, dyn_r_query=rq, dyn_r_add=r_add))
    return frames


def cam_tensor_from_c2w(c2w, jitter, rng):
    from scipy.spatial.transform import Rotation
    q = np.roll(Rotation.from_matrix(c2w[:3, :3]).as_quat(), 1)
    t = c2w[:3, 3] + rng.normal(0, jitter, 3)
    return torch.tensor(np.concatenate([q, t]), dtype=torch.float32)


class Clocks:
    """nvidia-smi clock / throttle-reason sampler running during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        try:
            ms = os.environ.get('PSL_CLOCKS_MS', '100')
            self.p = None if ms == '0' else subprocess.Popen(['nvidia-smi', '-i', str(index), f'--query-gpu={self.Q}',
                                                             '--format=csv,noheader,nounits', '-lms', ms], stdout=self.f,
                                                            stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(',') for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[2:6]):
                if 'Active' in v and 'Not' not in v:
                    reasons.add(name)
        hi = sorted(sm)[len(sm) // 2:] if sm else []          # upper half == samples taken under load
        return {'sm_mhz': float(np.median(hi)) if hi else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def build_decoders(cfg, device):
    from point_slam_b200.src.conv_onet import config as model_config
    torch.manual_seed(1219)
    decoders = model_config.get_model(cfg)
    sd = load_decoder_state()
    emb = sd.pop('color_decoder.embedder._B')
    decoders.load_state_dict(sd, strict=True)
    decoders.color_decoder.embedder._B = emb
    return decoders.to(device)


def build_cloud(cfg, device, n_points, seed, reserve=None):
    from point_slam_b200.src.neural_point import NeuralPointCloud
    cloud = synth.make_cloud(n_points, seed=seed)
    gf, cf = synth.make_features(n_points, seed=seed)
    npc = NeuralPointCloud(cfg)
    npc._cloud_pos = torch.from_numpy(cloud)
    npc._pts_num = n_points
    npc.geo_feats = torch.from_numpy(gf).to(device)
    npc.col_feats = torch.from_numpy(cf).to(device)
    if reserve:
        npc.reserve(reserve)
    npc.index.add(npc._pos)
    return npc


# ---------------------------------------------------------------------------------------------------------------------
# CUDA arm, tracking / mapping workloads (c2, c4)
# ---------------------------------------------------------------------------------------------------------------------
class GpuScene:
    def __init__(self, rank, device, wl, n_points, n_frames, share_map=False, dist=None):
        from point_slam_b200.src.utils.Renderer import Renderer
        from point_slam_b200 import graphed as G, ops
        import types
        self.device, self.wl, self.rank, self.dist, self.share_map = device, wl, rank, dist, share_map
        self.S = wl['S']
        self.cfg = make_cfg(wl['dataset'], device)
        self.decoders = build_decoders(self.cfg, device)
        seed = 1219 + (0 if share_map else rank)
        # capacity for everything the timed steps may append (<= 7000 pixels x 3 points per step): no re-allocation, so the
        # captured iteration graphs stay valid while the cloud grows
        self.npc = build_cloud(self.cfg, device, n_points, seed, reserve=n_points + (n_frames + 2) * 21000 + 4096)
        self.renderer = Renderer(self.cfg, None, types.SimpleNamespace(**{k: INTR[k] for k in ('H', 'W', 'fx', 'fy', 'cx', 'cy')}))
        self.renderer.sigmoid_coefficient = 0.1
        self.frames_host = make_frames(n_frames + N_KEYFRAMES, seed=seed, noise=wl['noise'], holes=wl['holes'])
        self.rng = np.random.default_rng(7 + rank)
        self.gen = torch.Generator(device=device).manual_seed(11 + rank)
        # keyframes are resident (they were mapped earlier); incoming frames live in pinned host memory
        self.keyframes = [self._to_device(f) for f in self.frames_host[:N_KEYFRAMES]]
        keys = ('color', 'depth', 'dyn_r_query', 'dyn_r_add')
        self.pinned = [{k: torch.from_numpy(np.ascontiguousarray(f[k])).pin_memory() for k in keys} for f in self.frames_host[N_KEYFRAMES:]]
        self.resident = [self._to_device(f) for f in self.frames_host[N_KEYFRAMES:]]
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.pinned[0].values())
        self.out_host = torch.empty(8, dtype=torch.float32).pin_memory()
        self.r_add = torch.zeros(INTR['H'], INTR['W'], dtype=torch.float64, device=device)
        self.G, self.ops = G, ops
        tc = self.cfg['tracking']
        self.tracker = G.FusedTracker(self.renderer, self.npc, self.decoders, INTR, wl['track'][1], device, edge=(wl['edge'], wl['edge']),
                                      lr=tc['lr'], w_color=tc['w_color_loss'], separate_lr=tc['separate_LR'])
        self.mapper = G.FusedMapper(self.renderer, self.npc, self.decoders, INTR, wl['map'][1], device) if wl['map'] else None
        self.map_ev = []
        self.map_host = []                # host wall time of the same section (it holds the step's host syncs)
        self.map_parts = []               # ... split into (add_neural_points x2, frustum selection, mapper.begin_frame)
        self.added = 0
        self.channel = None
        self.delta_ev = []

    def _to_device(self, f):
        d = self.device
        return dict(color=torch.from_numpy(f['color']).to(d), depth=torch.from_numpy(f['depth']).to(d),
                    dyn_r_query=torch.from_numpy(f['dyn_r_query']).to(d), dyn_r_add=torch.from_numpy(f['dyn_r_add']).to(d),
                    c2w=torch.from_numpy(f['c2w'][:3, :4].astype(np.float32)).to(d))

    def map_update(self, c2w, depth, color):
        """The per-mapped-frame map update (Mapper.py:306-345): add_neural_points on 6000 random pixels with the per-pixel add
        radius and on 1000 more with the small radius (the reference picks those by colour gradient on the host -- out of scope,
        SURVEY.md section 2 row 4 -- here they are random pixels), then the frustum feature selection.  Rank 0 of a shared map
        broadcasts the delta (new points + their feature rows) to the replicas."""
        from point_slam_b200.src import common
        d, npc = self.device, self.npc
        n0 = npc.pts_num()
        for n_pix, grad in ((6000, False), (1000, True)):
            pix = torch.randint(0, INTR['H'] * INTR['W'], (n_pix,), device=d, generator=self.gen)
            j, i = pix // INTR['W'], pix % INTR['W']
            ro, rd = common.get_rays_from_uv(i.float(), j.float(), c2w, INTR['fx'], INTR['fy'], INTR['cx'], INTR['cy'], d)
            gd, gc = depth[j, i], color[j, i]
            keep = gd > 0                                          # get_samples(depth_filter=True), common.py:173-179
            if self.share_map and self.rank != 0:
                continue
            npc.add_neural_points(ro[keep], rd[keep], gd[keep], gc[keep], is_pts_grad=grad, dynamic_radius=self.r_add[j, i][keep])
        self.added += npc.pts_num() - n0
        return n0

    def share_delta(self, n0, rows):
        """Shared-map mode: rank 0's map delta of this frame (appended points + their feature rows, the feature rows its mapper
        optimised, the colour decoder) reaches every replica with ONE NCCL broadcast (parallel.DeltaChannel)."""
        from point_slam_b200 import parallel as PAR
        if self.channel is None:
            self.channel = PAR.DeltaChannel(self.device, PAR.n_decoder_floats(self.decoders))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if self.rank == 0:
            self.channel.pack_from(self.npc, self.decoders, n0, rows)
        PAR.apply_delta(self.npc, self.decoders, self.channel.broadcast(None, 0))
        e1.record()
        self.delta_ev.append((e0, e1))

    def step(self, k, from_host, graphs=True):
        """Process frame k.  graphs=True: each iteration is one CUDA-graph replay of the static-shape shell
        (point_slam_b200/graphed.py); graphs=False: the same iterations launched eagerly (per-kernel timing pass).
        Returns the number of ray-samples rendered (fwd+bwd)."""
        d, wl = self.device, self.wl
        fh = self.frames_host[N_KEYFRAMES + k]
        src = self.pinned[k] if from_host else self.resident[k]
        cam0 = cam_tensor_from_c2w(fh['c2w'], 0.01, self.rng).to(d, non_blocking=True)
        tr = self.tracker
        tr.load_frame(src['color'], src['depth'], src['dyn_r_query'], cam0)        # H2D from pinned memory in the e2e pass
        self.r_add.copy_(src['dyn_r_add'], non_blocking=True)
        t_it, t_rays = wl['track']
        if graphs:
            loss = tr.run(t_it)
        else:
            for _ in range(t_it):
                tr._iter()
            loss = tr.loss
        samples = t_it * t_rays * self.S
        if self.mapper is not None:
            m_it, m_rays = wl['map']
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            h0 = time.perf_counter()
            c2w = torch.from_numpy(fh['c2w'][:3, :4].astype(np.float32)).to(d, non_blocking=True)
            n0 = self.map_update(c2w, tr.depth, tr.color)
            h1 = time.perf_counter()
            cur = dict(color=tr.color, depth=tr.depth, dyn_r_query=tr.dyn, c2w=c2w)
            # frustum feature selection with the sensor-depth test, Mapper.get_mask_from_c2w (library kernel, one 4-byte D2H)
            idx = self.ops.frustum_select(self.npc.cloud_pos_tensor(), fh['c2w'], tr.depth, INTR['H'], INTR['W'], INTR['fx'], INTR['fy'],
                                          INTR['cx'], INTR['cy'], edge=-4, reuse=True)
            h2 = time.perf_counter()
            self.mapper.begin_frame(idx, [cur] + self.keyframes)
            e1.record()
            self.map_ev.append((e0, e1))
            h3 = time.perf_counter()
            self.map_host.append((h3 - h0) * 1e3)
            self.map_parts.append((round((h1 - h0) * 1e3, 2), round((h2 - h1) * 1e3, 2), round((h3 - h2) * 1e3, 2)))
            g = geo_iters(m_it)
            if graphs:
                self.mapper.run('geometry', g)
                loss = self.mapper.run('color', m_it - g)
            else:
                for it in range(m_it):
                    self.mapper._iter('geometry' if it < g else 'color')
                loss = self.mapper.loss
            rows = self.mapper.write_back()
            self.last_n0, self.last_rows = n0, rows
            if self.share_map:
                self.share_delta(n0, rows)
            samples += m_it * (m_rays // (1 + N_KEYFRAMES)) * (1 + N_KEYFRAMES) * self.S
        if from_host:
            self.out_host[:7].copy_(tr.best_cam, non_blocking=True)
            self.out_host[7:8].copy_(loss.reshape(1), non_blocking=True)
        return samples

    def captures(self):
        return self.tracker.captures + (self.mapper.captures if self.mapper else 0)

    def outputs(self):
        """What the last step hands its caller: the frame's pose estimate and its last tracking loss; with mapping also the mapping
        loss, the points the map update appended, the feature rows the mapper optimised (row indices + geometry and colour
        features, a fixed sample of DUMP_ROWS rows) and the colour decoder's parameters."""
        out = dict(pose=self.tracker.best_cam, tracking_loss=self.tracker.loss)
        if self.mapper is not None:
            rows = sample_rows(self.last_rows)
            out.update(mapping_loss=self.mapper.loss, added_points=self.npc.cloud_pos_tensor()[self.last_n0:], feature_rows=rows,
                       geo_feats=self.npc.get_geo_feats()[rows], col_feats=self.npc.get_col_feats()[rows],
                       color_decoder=torch.cat([p.detach().reshape(-1) for p in self.decoders.color_decoder.parameters()]))
        return out


# ---------------------------------------------------------------------------------------------------------------------
# CUDA arm, forward-render workloads (c1, c3)
# ---------------------------------------------------------------------------------------------------------------------
class RenderScene:
    def __init__(self, rank, device, wl, n_points, n_frames):
        from point_slam_b200.src.utils.Renderer import Renderer
        from point_slam_b200 import ops
        import types
        self.device, self.wl, self.ops = device, wl, ops
        self.S, self.R = wl['S'], wl['rays']
        self.cfg = make_cfg(wl['dataset'], device, **{'rendering.N_surface': self.S})
        self.decoders = build_decoders(self.cfg, device)
        self.npc = build_cloud(self.cfg, device, n_points, 1219 + rank)
        self.renderer = Renderer(self.cfg, None, types.SimpleNamespace(**{k: INTR[k] for k in ('H', 'W', 'fx', 'fy', 'cx', 'cy')}))
        self.renderer.sigmoid_coefficient = 0.1
        frames = make_frames(n_frames, seed=1219 + rank)
        rng = np.random.default_rng(3 + rank)
        self.batches = []
        for f in frames:
            pix = rng.integers(0, INTR['H'] * INTR['W'], self.R)
            j, i = pix // INTR['W'], pix % INTR['W']
            o, dd = synth.pixel_rays(f['c2w'], INTR['H'], INTR['W'], INTR['fx'], INTR['fy'], INTR['cx'], INTR['cy'])
            b = dict(rays_o=np.broadcast_to(o, (self.R, 3)).astype(np.float32).copy(), rays_d=dd[j, i].astype(np.float32),
                     depth=f['depth'][j, i].copy(), r_query=f['dyn_r_query'][j, i].copy())
            self.batches.append(b)
        self.pinned = [{k: torch.from_numpy(v).pin_memory() for k, v in b.items()} for b in self.batches]
        self.resident = [{k: torch.from_numpy(v).to(device) for k, v in b.items()} for b in self.batches]
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.pinned[0].values())
        self.out_host = torch.empty(self.R, 5, dtype=torch.float32).pin_memory()
        self.stage = {k: torch.empty_like(v) for k, v in self.resident[0].items()}
        self.tracker = self.mapper = None

    def step(self, k, from_host, graphs=True):
        b = self.resident[k]
        if from_host:
            for key, t in self.pinned[k].items():
                self.stage[key].copy_(t, non_blocking=True)
            b = self.stage
        with torch.no_grad():
            depth, unc, color, _ = self.renderer.render_batch_ray(
                self.npc, self.decoders, b['rays_d'], b['rays_o'], self.device, 'color', gt_depth=b['depth'],
                npc_geo_feats=self.npc.get_geo_feats(), npc_col_feats=self.npc.get_col_feats(), cloud_pos=self.npc.cloud_pos_tensor(),
                dynamic_r_query=b['r_query'], _zero_depth=(None, None))
        self.last = dict(depth=depth, uncertainty=unc, color=color)
        if from_host:
            self.out_host[:, 0].copy_(depth, non_blocking=True); self.out_host[:, 1].copy_(unc, non_blocking=True)
            self.out_host[:, 2:].copy_(color, non_blocking=True)
        return self.R * self.S

    def captures(self):
        return 0

    def outputs(self):
        """Depth, uncertainty and colour of every ray of the last batch."""
        return self.last

    def knn_stats(self):
        """Mean number of candidate points the kNN kernel stages per query (SURVEY.md section 8d asks for C-bar)."""
        b = self.resident[0]
        return self.ops.raymarch_knn_stats(self.npc.spatial_hash(), b['rays_o'], b['rays_d'], b['depth'], self.S,
                                           (b['r_query'] ** 2).contiguous())


class RerenderScene:
    """Frame-parallel re-render: the cloud / features / decoders are replicated (same seed on every rank), the frames of a step
    are sharded over the ranks by parallel.rerender_frames."""

    def __init__(self, rank, world, device, wl, n_points, n_frames):
        from point_slam_b200.src.utils.Renderer import Renderer
        import types
        self.device, self.wl, self.S, self.world = device, wl, wl['S'], world
        self.cfg = make_cfg(wl['dataset'], device)
        self.decoders = build_decoders(self.cfg, device)
        self.npc = build_cloud(self.cfg, device, n_points, 1219)
        self.renderer = Renderer(self.cfg, None, types.SimpleNamespace(**{k: INTR[k] for k in ('H', 'W', 'fx', 'fy', 'cx', 'cy')}))
        self.renderer.sigmoid_coefficient = 0.1
        F = wl['frames']
        host = make_frames(F, seed=1219)
        self.pinned = [{k: torch.from_numpy(np.ascontiguousarray(f[k])).pin_memory() for k in ('color', 'depth', 'dyn_r_query')} for f in host]
        self.c2w = [torch.from_numpy(f['c2w']).float().to(device) for f in host]
        self.resident = [dict(color=p['color'].to(device), depth=p['depth'].to(device), dyn_r_query=p['dyn_r_query'].to(device), c2w=c)
                         for p, c in zip(self.pinned, self.c2w)]
        self.stage = [{k: torch.empty_like(v) for k, v in f.items()} for f in self.resident]
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.pinned[0].values()) * F
        self.out_host = torch.empty(4, dtype=torch.float64).pin_memory()
        self.tracker = self.mapper = None
        self.metrics = None

    def step(self, k, from_host, graphs=True):
        from point_slam_b200 import parallel as PAR
        frames = self.resident
        if from_host:
            import torch.distributed as dist
            rank = dist.get_rank() if dist.is_initialized() else 0
            for i in PAR.shard_strided(len(self.stage), rank, self.world):        # only this rank's frames cross the bus
                for key, t in self.pinned[i].items():
                    self.stage[i][key].copy_(t, non_blocking=True)
                self.stage[i]['c2w'] = self.c2w[i]
            frames = self.stage
        self.metrics = PAR.rerender_frames(self.renderer, self.npc, self.decoders, frames, self.device)
        n_local = len(self.metrics['rendered'])
        return n_local * INTR['H'] * INTR['W'] * self.S

    def captures(self):
        return 0

    def outputs(self):
        """The image metrics and, of every frame this rank rendered, depth and colour at a fixed sample of DUMP_ROWS pixels."""
        m = self.metrics
        out = dict(psnr=m['psnr'], depth_l1=m['depth_l1'])
        for k, (d, c) in sorted(m['rendered'].items()):
            out[f'depth_frame{k}'] = sample_rows(d.reshape(-1), seed=k)
            out[f'color_frame{k}'] = sample_rows(c.reshape(-1, 3), seed=k)
        return out


class HostSampler:
    """Diagnostics (PSL_HOST_SAMPLER=1): a thread notes every 4 ms which Python line the main thread is executing (or blocked in, when
    the callee released the GIL); runs of identical samples longer than 20 ms that are not one of the step's known device syncs
    are reported in timing.host_stalls."""

    def __init__(self):
        import threading
        self.tid = threading.get_ident()
        self.samples = []
        self.stop = False
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        while not self.stop:
            f = sys._current_frames().get(self.tid)
            chain = []
            while f is not None and len(chain) < 5:
                chain.append(f'{os.path.basename(f.f_code.co_filename)}:{f.f_lineno}:{f.f_code.co_name}')
                f = f.f_back
            self.samples.append((time.perf_counter(), ' < '.join(chain)))
            time.sleep(0.004)

    def report(self):
        self.stop = True
        self.th.join()
        out, i, s = [], 0, self.samples
        while i < len(s):
            j = i
            while j + 1 < len(s) and s[j + 1][1] == s[i][1]:
                j += 1
            dt = (s[j][0] - s[i][0]) * 1e3
            if dt > 20.0:
                out.append((round(dt, 1), s[i][1]))
            gap = (s[j + 1][0] - s[j][0]) * 1e3 if j + 1 < len(s) else 0.0
            if gap > 20.0:
                out.append((round(gap, 1), 'GIL held after: ' + s[j][1]))
            i = j + 1
        return out


def timed_steps(scene, steps, first, from_host, dist):
    gc.collect()
    gc.disable()          # a generation-2 collection inside a step stalls the host between two device syncs of the map update (seen
    try:                  # as one 20 ms step per run, always at the same step index); both arms time with the collector off
        return _timed_steps(scene, steps, first, from_host, dist)
    finally:
        gc.enable()


def _timed_steps(scene, steps, first, from_host, dist):
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    samples = 0
    for k in range(steps):
        samples += scene.step(first + k, from_host)
        ev[k + 1].record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    per_step = [ev[k].elapsed_time(ev[k + 1]) for k in range(steps)]
    return ev[0].elapsed_time(ev[steps]), samples, per_step


def run_ours(args):
    from point_slam_b200 import _lib
    # keep stdout clean for the ONE JSON line: libraries that printf to fd 1 (e.g. the NCCL version banner) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    dist = None
    torch.cuda.set_device(local)
    device = f'cuda:{local}'
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device(device))
    lib = _lib.load()
    wl = CONFIGS[args.config]
    points = args.points or wl['points']
    render_mode = wl['mode'] in ('render', 'rerender')
    n_frames = args.steps + args.warmup
    if wl['mode'] == 'rerender':
        scene = RerenderScene(rank, world, device, wl, points, n_frames)
    elif render_mode:
        scene = RenderScene(rank, device, wl, points, n_frames)
    else:
        scene = GpuScene(rank, device, wl, points, n_frames, share_map=args.share_map and world > 1, dist=dist)
    # the CUDA arm has no CPU-parallel work after the scene is built: keep the intra-op pool small so that N ranks on one host do not
    # spin 128 OpenMP workers each between the few tiny ATen CPU ops of a step (the cpu_baseline leg calibrates its own count later)
    torch.set_num_threads(max(1, min(8, (os.cpu_count() or 8) // max(world, 1))))
    for k in range(args.warmup):
        scene.step(k, False)
    cap0 = scene.captures()
    ms0 = torch.cuda.memory_stats(device)
    sampler = HostSampler() if os.environ.get('PSL_HOST_SAMPLER') else None
    clocks = Clocks(local) if rank == 0 else None
    ms, samples, per_step = timed_steps(scene, args.steps, args.warmup, False, dist)
    ms_e2e, samples_e2e, per_step_e2e = timed_steps(scene, args.steps, args.warmup, True, dist)
    clk = clocks.stop() if clocks else None
    recaptures = scene.captures() - cap0
    host_stalls = sampler.report() if sampler else None
    ms1 = torch.cuda.memory_stats(device)
    if args.dump_outputs and rank == 0:
        # the last step of the second timed pass (inputs from pinned host memory): it replays the frames of the first pass on the
        # map that pass has grown; with --gpus N only rank 0's scene is written
        dump_outputs(args.dump_outputs, scene.outputs())
    alloc_diag = {k: ms1.get(k, 0) - ms0.get(k, 0) for k in ('num_device_alloc', 'num_device_free', 'num_alloc_retries', 'num_sync_all_streams')}
    alloc_diag['reserved_GB'] = round(ms1.get('reserved_bytes.all.current', 0) / 1e9, 2)
    map_ms = None
    if getattr(scene, 'map_ev', None):
        map_each = [round(a.elapsed_time(b), 2) for a, b in scene.map_ev[-2 * args.steps:]]
        map_ms = float(np.median(map_each))
        map_host_each = [round(v, 2) for v in scene.map_host[-2 * args.steps:]]
    # per-kernel device time of one more step (CUDA events on the launching stream inside the library): the same static-shape
    # iterations launched eagerly (graph replays bypass the host-side event hooks), geometry kernels in-line (no stream fork:
    # a forked kernel's slot would include the time it waits for free SMs and could be mistaken for the dominant kernel)
    from point_slam_b200 import ops as _ops
    l0 = lib.psl_launch_count()
    overlap, _ops.OVERLAP_BRANCHES = _ops.OVERLAP_BRANCHES, False
    _lib.timing_enable(True)
    n_prof = scene.step(min(args.warmup, n_frames - 1), False, graphs=False)
    prof = _lib.timing_collect()
    _lib.timing_enable(False)
    _ops.OVERLAP_BRANCHES = overlap
    launches = (lib.psl_launch_count() - l0) * args.steps           # kernels of this library per step x timed steps
    per_rank = [ms / args.steps]
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=device)
        gathered = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        per_rank = [float(g[0]) / args.steps for g in gathered]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        s = torch.tensor([samples, samples_e2e], device=device, dtype=torch.float64)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        ms, ms_e2e = float(t[0]), float(t[1])
        samples, samples_e2e = float(s[0]), float(s[1])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    value = samples / (ms * 1e-3)
    e2e = samples_e2e / (ms_e2e * 1e-3)
    peaks = {}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    bf16_peak = float(peaks.get('bf16_tflops', 1590.0))
    peak_src = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)'
    rel = bool(scene.cfg['model']['encode_rel_pos_in_col'])
    S = wl['S']
    bytes_fwd, bytes_bwd = 2144 + 49.0 / S, 2144 + 2048 + 49.0 / S       # SURVEY.md section 8d (gathered bytes per sample)
    tot_kernel_ms = sum(v[0] for v in prof.values())
    top = max(prof, key=lambda k: prof[k][0])
    top_ms, top_n = prof[top]
    # samples one launch of the dominant kernel processes (tracker launches see track_rays*S, the mapper's map_rays*S)
    if render_mode:
        samples_top = n_prof
    else:
        t_it, t_rays = wl['track']
        m_it, m_rays = wl['map'] if wl['map'] else (0, 0)
        col_it = m_it - geo_iters(m_it) if m_it else 0
        per_kernel = {'wgrad_tc': col_it * m_rays * S, 'color_fwd_tc': t_it * t_rays * S + col_it * m_rays * S,
                      'color_bwd_tc': t_it * t_rays * S + col_it * m_rays * S}
        samples_top = per_kernel.get(top, n_prof)
    per_launch_samples = samples_top / max(top_n, 1)
    avg_launch_s = top_ms / max(top_n, 1) * 1e-3
    bytes_per_sample = bytes_bwd if top in ('decode_bwd', 'color_bwd_tc', 'wgrad_tc') else bytes_fwd
    hbm_achieved = per_launch_samples * bytes_per_sample / avg_launch_s / 1e9
    traffic = None
    tj = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tj):
        t = json.load(open(tj)).get(top)
        if t:
            traffic = t['bytes_per_sample'] * per_launch_samples          # scaled to this launch size; source in profiles/traffic.json
    hbm_view = {'achieved': hbm_achieved, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': hbm_achieved / hbm_peak,
                'algorithmic_bytes_per_sample': bytes_per_sample}
    if top in ('color_fwd_tc', 'color_bwd_tc', 'wgrad_tc'):
        # ALGORITHMIC FLOPs of the launch (2 x MACs of the colour branch, SURVEY.md section 8d) over its duration against the
        # measured dense-bf16 peak; the MMA work actually issued (error-compensated split products) is a second field
        tf = per_launch_samples * 2 * TC_MAC[rel] / avg_launch_s / 1e12
        roof = {'bound': 'tensor', 'kernel': top, 'achieved': tf, 'peak': bf16_peak, 'unit': 'TFLOP/s', 'frac': tf / bf16_peak,
                'traffic': traffic, 'peak_source': peak_src, 'issued_mma_tflops': 3 * tf,
                'note': 'achieved = algorithmic FLOP/s of the colour branch (no x3 for the split-operand products); issued_mma_tflops counts the 3 MMAs per fp32-accurate product',
                'hbm': hbm_view}
    else:
        roof = {'bound': 'hbm', 'kernel': top, 'traffic': traffic, 'peak_source': peak_src, **hbm_view}
    fwd_bwd = 1 if render_mode else 3
    roof.update({'samples_per_launch': per_launch_samples, 'avg_launch_ms': avg_launch_s * 1e3,
                 'kernel_share_of_device_time': top_ms / max(tot_kernel_ms, 1e-9),
                 'algorithmic_tflops_all_kernels': fwd_bwd * FLOP_FWD[rel] * n_prof / max(tot_kernel_ms * 1e-3, 1e-9) / 1e12})
    cfg_out = workload_config(args.config, points)
    cfg_out['parallelism'] = f'scene-per-gpu x{world}' + (' + NCCL map-delta broadcast from rank 0' if args.share_map and world > 1 else '')
    out = {
        'metric': 'ray-samples/sec (render+kNN+MLP' + (' forward' if render_mode else ' fwd+bwd, frame step') + ')', 'value': value,
        'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps,
        'frames_per_sec': (wl['frames'] if wl['mode'] == 'rerender' else world) * args.steps / (ms * 1e-3), 'higher_is_better': True,
        'scaling': 'strong' if wl['mode'] == 'rerender' else 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'config': cfg_out,
        'timing': {'l2': 'inputs larger than L2 (cloud + features 134 MB at 500k points; saved activations ~290 MB per mapper iteration)',
                   'per_rank_ms_per_step': [round(x, 3) for x in per_rank],
                   'graph_recaptures_in_timed_region': recaptures, 'allocator_in_timed_region': alloc_diag, 'host_stalls': host_stalls, 'map_update_ms_per_step': map_ms, 'map_update_ms_each': map_each if map_ms is not None else None,
                   'map_update_host_ms_each': map_host_each if map_ms is not None else None,
                   'map_update_host_parts_ms': scene.map_parts[-2 * args.steps:] if map_ms is not None else None,
                   'points_at_end': scene.npc.pts_num(), 'points_added': getattr(scene, 'added', 0),
                   'map_delta_ms_per_step': (float(np.mean([a.elapsed_time(b) for a, b in scene.delta_ev[-2 * args.steps:]]))
                                             if getattr(scene, 'delta_ev', None) else None)},
        'e2e': {'value': e2e, 'unit': 'samples/s', 'h2d_bytes_per_step': scene.h2d_bytes,
                'd2h_bytes_per_step': 32 if not render_mode else scene.out_host.numel() * scene.out_host.element_size(),
                'ms_per_step': ms_e2e / args.steps},
        'gpu_launches': int(launches),
        'clocks': clk,
        'roofline': roof,
        'step_ms': [round(x, 2) for x in per_step], 'step_ms_e2e': [round(x, 2) for x in per_step_e2e],
        'kernel_ms_per_step': {k: round(v[0], 3) for k, v in prof.items()},
        'kernel_launches_per_step': {k: v[1] for k, v in prof.items()},
    }
    if wl['mode'] == 'rerender':
        out['rerender'] = {k: v for k, v in scene.metrics.items() if k != 'rendered'}
        cfg_out['parallelism'] = f'frame-parallel x{world} (cloud replicated; one all_reduce of the image metrics per step)'
    if wl['mode'] == 'render':
        out['knn'] = scene.knn_stats()
        knn_ms = prof['knn'][0]
        out['value_knn_excluded'] = n_prof / max((tot_kernel_ms - knn_ms) * 1e-3, 1e-9)
        out['roofline']['hbm_whole_forward'] = {'achieved': n_prof * bytes_fwd / (tot_kernel_ms * 1e-3) / 1e9, 'peak': hbm_peak,
                                                 'frac': n_prof * bytes_fwd / (tot_kernel_ms * 1e-3) / 1e9 / hbm_peak, 'unit': 'GB/s'}
    if world == 1 and not args.no_cpu_baseline:
        out['cpu_baseline'] = cpu_baseline_sample(args.config, points)
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(out) + '\n').encode())
    if dist is not None:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# reference arm: the reference algorithm (CPU oracle port) on the host cores, same iteration shells, same iteration mix
# ---------------------------------------------------------------------------------------------------------------------
class CpuScene:
    def __init__(self, wl, n_points, n_frames):
        from scipy.spatial import cKDTree
        from point_slam_b200.src.conv_onet import config as model_config
        self.wl, self.S = wl, wl['S']
        self.cfg = make_cfg(wl['dataset'], 'cpu', **{'rendering.N_surface': wl['S']})
        torch.manual_seed(1219)
        self.decoders = model_config.get_model(self.cfg)
        sd = load_decoder_state()
        emb = sd.pop('color_decoder.embedder._B')
        self.decoders.load_state_dict(sd, strict=True)
        self.decoders.color_decoder.embedder._B = emb
        self.rel = bool(self.cfg['model']['encode_rel_pos_in_col'])
        cloud = synth.make_cloud(n_points, seed=1219)
        gf, cf = synth.make_features(n_points, seed=1219)
        self.cloud = torch.from_numpy(cloud)
        self.geo, self.col = torch.from_numpy(gf), torch.from_numpy(cf)
        self.tree = cKDTree(cloud.astype(np.float64))
        self.frames = []
        for f in make_frames(n_frames + 1, seed=1219, noise=wl.get('noise', False), holes=wl.get('holes', 0.0)):
            self.frames.append(dict(color=torch.from_numpy(f['color']), depth=torch.from_numpy(f['depth']),
                                    dyn_r_query=torch.from_numpy(f['dyn_r_query']), dyn_r_add=torch.from_numpy(f['dyn_r_add']),
                                    c2w=torch.from_numpy(f['c2w'][:3, :4].astype(np.float32)), c2w64=f['c2w']))
        self.rng = np.random.default_rng(7)

    # duck-typed npc for the iteration shells
    def get_geo_feats(self):
        return self.geo

    def get_col_feats(self):
        return self.col

    def render(self, npc, decoders, rays_d, rays_o, device, stage, gt_depth=None, npc_geo_feats=None, npc_col_feats=None,
               is_tracker=False, cloud_pos=None, dynamic_r_query=None, exposure_feat=None):
        from oracle import point_slam_oracle as O
        P = dict(decoders.named_parameters())
        P['color_decoder.embedder._B'] = decoders.color_decoder.embedder._B
        rg = torch.zeros([32]).normal_(mean=0, std=0.01)
        rc = torch.zeros([32]).normal_(mean=0, std=0.01)
        return O.render_batch_ray(P, rays_d, rays_o, gt_depth, stage, self.cloud, npc_geo_feats, npc_col_feats, S=self.S,
                                  is_tracker=is_tracker, radius_query=0.08, dynamic_r_query=dynamic_r_query, rand_geo=rg,
                                  rand_col=rc, coef=0.1, encode_rel_pos=self.rel, tree=self.tree)

    def map_update(self, cur):
        """add_neural_points on 6000 + 1000 pixels (kept-location test only: the appended points are not indexed, like a frame
        that adds nothing) and the frustum feature selection -- the CPU restatements of oracle/point_slam_oracle.py."""
        from oracle import point_slam_oracle as O
        from point_slam_b200.src import common
        for n_pix, grad in ((6000, False), (1000, True)):
            pix = torch.from_numpy(self.rng.integers(0, INTR['H'] * INTR['W'], n_pix))
            j, i = pix // INTR['W'], pix % INTR['W']
            ro, rd = common.get_rays_from_uv(i.float(), j.float(), cur['c2w'], INTR['fx'], INTR['fy'], INTR['cx'], INTR['cy'], 'cpu')
            gd = cur['depth'][j, i]
            keep = gd > 0
            O.add_points(self.cloud, ro[keep], rd[keep], gd[keep], dynamic_radius=cur['dyn_r_add'][j, i][keep], is_pts_grad=grad,
                         tree=self.tree)
        return torch.from_numpy(O.frustum_indices(self.cloud.numpy(), cur['c2w64'].astype(np.float32), cur['depth'].numpy(), INTR['H'],
                                                  INTR['W'], INTR['fx'], INTR['fy'], INTR['cx'], INTR['cy'], edge=-4))

    def step(self, k, track_iters, map_iters, map_pix):
        """Frame k with `track_iters` tracking and `map_iters` mapping iterations (first geo_iters(map_iters) geometry-stage)."""
        wl = self.wl
        cur = self.frames[1 + k]
        samples = 0
        tc = self.cfg['tracking']
        cam = cam_tensor_from_c2w(cur['c2w64'], 0.01, self.rng).requires_grad_(True)
        opt = torch.optim.Adam([cam], lr=tc['lr'])
        for _ in range(track_iters):
            _, n = IT.tracker_iteration(self.render, self, self.decoders, cam, opt, cur['color'], cur['depth'],
                                        cur['dyn_r_query'], INTR, wl['track'][1], 'cpu', self.geo, self.col, self.cloud,
                                        edge=(wl['edge'], wl['edge']))
            samples += n * self.S
        if map_iters:
            idx = self.map_update(cur)
            state = IT.MapperState(self, self.decoders, idx)
            g = geo_iters(map_iters)
            for it in range(map_iters):
                _, n = IT.mapper_iteration(self.render, self, self.decoders, state, [cur, self.frames[0]], INTR, map_pix, 'cpu',
                                           'geometry' if it < g else 'color', self.cloud)
                samples += n * self.S
        return samples


class CpuRenderScene:
    def __init__(self, wl, n_points, n_frames):
        self.inner = CpuScene(dict(wl, track=None, map=None, edge=0), n_points, n_frames)
        self.wl = wl
        rng = np.random.default_rng(3)
        self.batches = []
        for f in self.inner.frames:
            pix = rng.integers(0, INTR['H'] * INTR['W'], wl['rays'])
            j, i = pix // INTR['W'], pix % INTR['W']
            o, dd = synth.pixel_rays(f['c2w64'], INTR['H'], INTR['W'], INTR['fx'], INTR['fy'], INTR['cx'], INTR['cy'])
            self.batches.append(dict(rays_o=torch.from_numpy(np.broadcast_to(o, (wl['rays'], 3)).astype(np.float32).copy()),
                                     rays_d=torch.from_numpy(dd[j, i].astype(np.float32)), depth=f['depth'][j, i],
                                     r_query=f['dyn_r_query'][j, i]))

    def step(self, k, n_rays):
        b = self.batches[k % len(self.batches)]
        with torch.no_grad():
            self.inner.render(None, self.inner.decoders, b['rays_d'][:n_rays], b['rays_o'][:n_rays], 'cpu', 'color',
                              gt_depth=b['depth'][:n_rays], npc_geo_feats=self.inner.geo, npc_col_feats=self.inner.col,
                              dynamic_r_query=b['r_query'][:n_rays])
        return n_rays * self.wl['S']


def cpu_sample_sizes(name):
    """Bounded CPU sample of one step with the SAME iteration mix as the CUDA arm (track : map iterations and the geometry
    share of the mapping iterations), sized for ~10-20 s on the host cores."""
    wl = CONFIGS[name]
    if wl['mode'] in ('render', 'rerender'):
        return None
    if wl['map']:
        f = 2                                               # c2: 40 : 60 (25 geometry) -> 20 : 30 (13 geometry), ~10 s per sample
        return max(wl['track'][0] // f, 1), max(wl['map'][0] // f, 1)
    return max(wl['track'][0] // 3, 1), 0                   # c4: 200 -> 66 tracking iterations (~11 s)


def pick_threads(step_fn):
    """The faster of {all host threads, 32} torch threads on a small untimed step each (tiny ATen ops oversubscribe a
    128-thread box: 32 threads were 7x faster there)."""
    times = {}
    for k, th in enumerate([os.cpu_count()] + ([32] if os.cpu_count() > 32 else [])):
        torch.set_num_threads(th)
        step_fn(k)                                          # first touch (allocator, thread pool)
        t0 = time.perf_counter()
        step_fn(k)
        times[th] = time.perf_counter() - t0
    threads = min(times, key=times.get)
    torch.set_num_threads(threads)
    return threads


def cpu_run(name, n_points, steps, warmup):
    """-> (samples/s, threads, seconds, description of the per-step sample)"""
    wl = CONFIGS[name]
    if wl['mode'] in ('render', 'rerender'):
        wl = dict(wl, rays=wl.get('rays', 2000))           # re-render: a 2000-ray sample of the image
        sc = CpuRenderScene(wl, n_points, steps + warmup + 2)
        n_rays = min(wl['rays'], 5000)
        reps = max(1, int(np.ceil(1.2e6 / (n_rays * wl['S']))))      # ~10 s of host work per step at ~1.2e5 samples/s
        threads = pick_threads(lambda k: sc.step(k, 200))
        for k in range(warmup):
            sc.step(k, 200)
        gc.collect(); gc.disable()
        t0 = time.perf_counter()
        n = sum(sc.step(2 + warmup + k, n_rays) for k in range(steps) for _ in range(reps))
        dt = time.perf_counter() - t0
        gc.enable()
        what = f'{n_rays} of the {wl["rays"]} rays' if CONFIGS[name]['mode'] == 'render' else f'{n_rays} rays of a 640x480 frame'
        return n / dt, threads, dt, f'{reps} x ({what} x {wl["S"]} samples, forward render)'
    r_track, r_map = cpu_sample_sizes(name)
    sc = CpuScene(wl, n_points, steps + warmup + 2)
    m_pix = wl['map'][1] if wl['map'] else 0
    threads = pick_threads(lambda k: sc.step(k, 1, 1 if r_map else 0, 500))
    for k in range(warmup):
        sc.step(2 + k, 1, 1 if r_map else 0, 500)
    gc.collect(); gc.disable()
    t0 = time.perf_counter()
    n = sum(sc.step(2 + warmup + k, r_track, r_map, m_pix) for k in range(steps))
    dt = time.perf_counter() - t0
    gc.enable()
    desc = f'{r_track} of the {wl["track"][0]} tracking iterations x {wl["track"][1]} rays'
    if r_map:
        desc += (f' + map update + {r_map} of the {wl["map"][0]} mapping iterations x {m_pix} rays ({geo_iters(r_map)} geometry-stage): '
                 'same track : map : geometry-stage proportions as the full step')
    return n / dt, threads, dt, desc


def cpu_baseline_sample(name, n_points):
    v, threads, dt, desc = cpu_run(name, n_points, 1, 0)
    return {'value': v, 'unit': 'samples/s', 'cores': threads, 'kind': 'port',
            'sample': f'{desc}; fwd+loss+bwd+Adam through the oracle port of the reference (oracle/point_slam_oracle.py, iteration '
                      f'shells of point_slam_b200/iteration.py), {n_points}-point cloud, torch {torch.__version__} CPU ({threads} of '
                      f'{os.cpu_count()} threads) + scipy cKDTree exact kNN; {dt:.1f} s', 'seconds': dt}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if rank != 0:
        return
    wl = CONFIGS[args.config]
    points = args.points or wl['points']
    v, threads, dt, desc = cpu_run(args.config, points, args.steps, args.warmup)
    sample = f'per step: {desc}; host cores ({threads} torch threads of {os.cpu_count()}; oracle port of the reference, exact cKDTree kNN)'
    render_mode = wl['mode'] in ('render', 'rerender')
    out = {'impl': 'reference', 'metric': 'ray-samples/sec (render+kNN+MLP' + (' forward' if render_mode else ' fwd+bwd, frame step') + ')',
           'value': v, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
           'ms_per_step': dt * 1e3 / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
           'dtype': 'f32', 'data': 'synthetic', 'config': dict(workload_config(args.config, points), parallelism=f'scene-per-gpu x{world}'),
           'sample': sample,
           'cpu_baseline': {'value': v, 'unit': 'samples/s', 'cores': threads, 'kind': 'port', 'sample': sample},
           'e2e': {'value': v, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps (default: 20 for the c2 frame step of the CUDA arm, else 5)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='c2', choices=sorted(CONFIGS))
    ap.add_argument('--points', type=int, default=0, help='override the cloud size of the configuration')
    ap.add_argument('--share-map', action='store_true', help='N > 1: one scene replicated on every GPU, rank 0 maps and broadcasts the map delta (NCCL) every step')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last timed step computed as '
                    'DIR/<name>.npy (float32 / float64, at most 64 MiB; the inputs are seeded, so two builds compare output for output). '
                    'That step is the last of the second timed pass (inputs from pinned host memory), which replays the frames of the '
                    'first pass on the map the first pass has grown; with --gpus N only rank 0 writes its scene')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs dumps the CUDA arm (--impl ours)')
    if args.steps is None:
        # one host hiccup inside the map update's sync window costs a whole step (~45 ms: see DESIGN.md section 5), so the default
        # averages over 20 frame steps (1 s of device time) instead of 5
        args.steps = 20 if (args.impl == 'ours' and args.config == 'c2') else 5
    if args.impl == 'reference':
        run_reference(args)
    else:
        assert torch.cuda.is_available(), 'bench.py (CUDA arm) needs a GPU; there is no CPU fallback'
        run_ours(args)


if __name__ == '__main__':
    main()
