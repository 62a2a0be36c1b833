"""Per-frame colour-gradient pass: host path against device path, and the C4 tracking step with uniform against
gradient-selected pixels (DESIGN.md section 5).

    python profiles/prof_frame_grad.py [--frames 20] [--reps 3] [--out FILE.json]

1. Radius maps of one 640x480 frame: the host path PointSLAM used before (device colour -> host, synth.sobel_radius_map in
   float64 numpy, both maps back to the device) against psl_frame_grad + psl_grad_candidates (tracker window, 5000 x 15).
   Host clock around work that ends in a device synchronise, and CUDA events for the device path.
2. The C4-shaped tracking step (TUM configuration, 500 k points, 200 iterations x 5000 rays, noisy depth with holes): one
   load_frame + run(200) of FusedTracker with uniform pixels and with sample_with_color_grad=True, alternated `--reps` times
   over the same frames.  Edge pixels have other neighbourhoods, so the kNN and colour kernels may take another time.
The card name and power limit are printed beside the numbers.  Needs a GPU; there is no fallback.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                                  # the numbers still name the device below
        q = f'nvidia-smi unavailable ({e})'
    return {'device': torch.cuda.get_device_name(0), 'nvidia_smi': q}


def host_vs_device(frames, dev):
    from point_slam_b200 import ops, synth
    from point_slam_b200.default_config import make_cfg
    cfg = make_cfg('tum', dev)
    pc = cfg['pointcloud']
    cols = [torch.from_numpy(f['color']).to(dev) for f in frames]
    deps = [torch.from_numpy(f['depth']).to(dev) for f in frames]
    H, W = deps[0].shape
    win = (20, H - 20, 20, W - 20)

    def host(c):
        r_add, r_q = synth.sobel_radius_map(c.cpu().numpy(), pc['radius_add_max'], pc['radius_add_min'], pc['radius_query_ratio'],
                                            pc['color_grad_threshold'])
        return torch.from_numpy(r_add).to(dev), torch.from_numpy(r_q).to(dev)

    def device(c, d):
        r_add, r_q, mag = ops.frame_grad(c, cfg)
        ops.grad_candidates(mag, d, 5000, 15, window=win)
        return r_add, r_q

    for c, d in zip(cols[:2], deps[:2]):                                   # warm-up (module load, cub tuning, allocator)
        host(c); device(c, d)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for c in cols:
        host(c)
    torch.cuda.synchronize()
    host_ms = (time.perf_counter() - t0) * 1e3 / len(cols)
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for c, d in zip(cols, deps):
            device(c, d)
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / (reps * len(cols))
    # the two kernels alone (no allocation): psl_frame_grad with every output, then the candidate list
    mag = torch.empty(H, W, dtype=torch.float64, device=dev)
    ra, rq = torch.empty_like(mag), torch.empty_like(mag)
    cand = torch.empty(75000, dtype=torch.int64, device=dev); cnt = torch.empty(1, dtype=torch.int32, device=dev)
    from point_slam_b200 import _lib as L
    ws = torch.empty(L.load().psl_grad_candidates_ws_bytes(H * W), dtype=torch.uint8, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    for _ in range(reps):
        for c in cols:
            ops.frame_grad(c, cfg, mag_out=mag)
    ev[1].record()
    for _ in range(reps):
        for d in deps:
            ops.grad_candidates(mag, d, 5000, 15, window=win, cand=cand, count=cnt, ws=ws)
    ev[2].record()
    torch.cuda.synchronize()
    n = reps * len(cols)
    return {'host_sobel_with_copies_ms': host_ms, 'device_frame_grad_plus_candidates_ms': dev_ms,
            'frame_grad_ms': ev[0].elapsed_time(ev[1]) / n, 'grad_candidates_ms': ev[1].elapsed_time(ev[2]) / n,
            'frames': len(cols)}


def tracking(dev, n_frames, reps):
    import bench
    from point_slam_b200 import graphed as G
    wl = bench.CONFIGS['c4']
    scene = bench.GpuScene(0, dev, wl, wl['points'], n_frames)
    it, rays = wl['track']
    tc = scene.cfg['tracking']
    mk = lambda grad: G.FusedTracker(scene.renderer, scene.npc, scene.decoders, bench.INTR, rays, dev, edge=(wl['edge'], wl['edge']),
                                     lr=tc['lr'], w_color=tc['w_color_loss'], separate_lr=tc['separate_LR'], sample_with_color_grad=grad)
    trackers = {'uniform': mk(False), 'color_grad': mk(True)}
    cams = [bench.cam_tensor_from_c2w(scene.frames_host[bench.N_KEYFRAMES + k]['c2w'], 0.01, scene.rng).to(dev) for k in range(n_frames)]

    def step(tr, k):
        f = scene.resident[k]
        tr.load_frame(f['color'], f['depth'], f['dyn_r_query'], cams[k])
        tr.run(it)

    for tr in trackers.values():                                           # capture + warm-up
        step(tr, 0)
    torch.cuda.synchronize()
    # the per-iteration draw alone (key draw + psl_pick_candidates), to split the step difference into drawing and rendering
    from point_slam_b200 import ops
    g = trackers['color_grad']
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(it):
        ops.pick_candidates(g.cand, g.cand_count, rays, bench.INTR['W'], window=g._window(), pix=g.picked, ws=g.pick_ws)
    e1.record()
    torch.cuda.synchronize()
    pick_ms = e0.elapsed_time(e1) / it
    times = {k: [] for k in trackers}
    for _ in range(reps):
        for name, tr in trackers.items():                                 # alternated, same frames
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(n_frames):
                step(tr, k)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / n_frames)
    out = {f'{k}_ms_per_step': float(np.median(v)) for k, v in times.items()}
    out.update({f'{k}_ms_all': v for k, v in times.items()})
    out['pick_candidates_ms_per_iteration'] = pick_ms
    out['candidate_capacity'] = int(g.cand.numel())
    out['captures'] = {k: tr.captures for k, tr in trackers.items()}
    out['workload'] = f'C4: {it} iterations x {rays} rays, {wl["points"]} points, TUM configuration, noisy depth with 5 % holes'
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=20)
    ap.add_argument('--track-frames', type=int, default=4)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'prof_frame_grad.py measures on a GPU'
    import bench
    dev = 'cuda:0'
    frames = bench.make_frames(args.frames, seed=1219, noise=True, holes=0.05)
    res = {'card': card(), 'radius_maps': host_vs_device(frames, dev), 'tracking': tracking(dev, args.track_frames, args.reps)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
