"""Helpers shared by the CPU and GPU tests that replay the reference's own callers of the render path
(tests/golden/caller_*.npz, render_img_*.npz -- frozen from the unmodified reference by oracle/make_golden_callers.py)."""
import contextlib
import os

import numpy as np
import torch

from tests import cases as C

WIN = (150, 330, 220, 420)          # pixel window (j0, j1, i0, i1) of the golden scene
INTR = C.INTR


def load(name):
    z = np.load(os.path.join(C.GOLDEN, f'{name}.npz'))
    return {k: z[k] for k in z.files}


def full_image(win, channels_last=False, dtype=None):
    """Window crop -> full 480x640 image, zero outside the window (what the generator fed the reference)."""
    j0, j1, i0, i1 = WIN
    shape = (INTR['H'], INTR['W']) + tuple(win.shape[2:])
    out = np.zeros(shape, dtype or win.dtype)
    out[j0:j1, i0:i1] = win
    return out


def full_radius(win, fill=0.16):
    """The per-pixel radius maps are only read where the depth is > 0 (inside the window); outside any finite value does."""
    j0, j1, i0, i1 = WIN
    out = np.full((INTR['H'], INTR['W']), fill, np.float64)
    out[j0:j1, i0:i1] = win
    return out


def dense_rows(rows, vals, n, width=32):
    out = np.zeros((n, width), np.float32)
    out[rows] = vals
    return out


@contextlib.contextmanager
def replay_randint(draws, device=None):
    """torch.randint returns the recorded draws, in order (select_uv's only RNG use, common.py:66)."""
    it = iter(draws)
    orig = torch.randint

    def fake(*a, **kw):
        d = torch.as_tensor(next(it))
        assert d.shape[0] == a[1][0], 'recorded draw has another size than the one requested'
        return d.to(kw.get('device', device) or 'cpu')
    torch.randint = fake
    try:
        yield
    finally:
        torch.randint = orig


class Errors:
    """Collects (case, quantity, achieved error, limit) rows; the GPU session writes them to $PSL_PARITY_JSON (tests/conftest.py)."""
    rows = []

    @classmethod
    def check(cls, case, quantity, got, want, limit, noise=None):
        """err = max|got - want| / max|want| (the tensor-scale relative error the north-star's 1e-4 is read with).
        `noise`: error of the fp32 oracle against fp64 for the same quantity, when known -- the limit may not be tighter than
        the reference's own rounding noise."""
        err = C.rel_err(torch.as_tensor(got).detach().cpu(), torch.as_tensor(want))
        lim = limit if noise is None else max(limit, 3 * noise)
        cls.rows.append(dict(case=case, quantity=quantity, err=float(err), limit=float(lim), flat_limit=float(limit),
                             fp32_noise=None if noise is None else float(noise), ok=bool(err <= lim)))
        assert err <= lim, f'{case} {quantity}: rel err {err:.3e} > {lim:.1e}'
        return err

    @classmethod
    def dump(cls, path):
        import json
        os.makedirs(os.path.dirname(path), exist_ok=True)
        prev = []
        if os.path.exists(path):
            try:
                prev = json.load(open(path))['rows']
            except Exception:
                prev = []
        keys = {(r['case'], r['quantity']) for r in cls.rows}
        rows = [r for r in prev if (r['case'], r['quantity']) not in keys] + cls.rows
        json.dump({'note': 'achieved parity per case x quantity: err = max|a-b|/max|b| against the stated reference '
                           '(golden = unmodified reference on the CPU, oracle64 = float64 oracle); limit = the bound the test applied',
                   'rows': sorted(rows, key=lambda r: (r['case'], r['quantity']))}, open(path, 'w'), indent=1)


# ---------------------------------------------------------------------------------------------------------------------
# running the reference's own callers (oracle/_ref, a git-ignored copy of the reference's src/ + configs/ made by
# __graft_entry__.build() where it finds the reference) on top of the drop-in modules: INTEGRATION.md section 1, executed
# ---------------------------------------------------------------------------------------------------------------------
REF_COPY = os.path.join(C.ROOT, 'oracle', '_ref')


def have_reference_copy():
    return os.path.exists(os.path.join(REF_COPY, 'src', 'Tracker.py'))


def install_module_swap():
    """Register the drop-in modules under the reference's module paths and import the reference's Tracker / Mapper from
    oracle/_ref.  -> (Tracker class, Mapper class, reference `src.common` module, reference `src.Mapper` module)."""
    import sys
    import types
    import point_slam_b200.src as b
    import point_slam_b200.src.neural_point
    import point_slam_b200.src.conv_onet.models.decoder
    import point_slam_b200.src.utils.Renderer

    def stub(name, **attrs):
        if name not in sys.modules:
            m = types.ModuleType(name)
            for k, v in attrs.items():
                setattr(m, k, v)
            sys.modules[name] = m
    # import-time-only dependencies of the reference callers that this image lacks (never reached by the methods under test)
    sk = types.ModuleType('skimage'); skc = types.ModuleType('skimage.color'); skf = types.ModuleType('skimage.filters')
    skc.rgb2gray = lambda x: x
    skf.sobel_h = skf.sobel_v = None
    sk.color, sk.filters = skc, skf
    for n, m in (('skimage', sk), ('skimage.color', skc), ('skimage.filters', skf)):
        sys.modules.setdefault(n, m)
    stub('open3d'); stub('colorama', Fore=types.SimpleNamespace(), Style=types.SimpleNamespace())
    stub('matplotlib'); stub('matplotlib.pyplot'); stub('torchmetrics'); stub('torchmetrics.image')
    stub('torchmetrics.image.lpip', LearnedPerceptualImagePatchSimilarity=object)
    stub('pytorch_msssim', ms_ssim=None); stub('wandb')
    for k in [k for k in sys.modules if k == 'src' or k.startswith('src.')]:
        del sys.modules[k]
    if REF_COPY not in sys.path:
        sys.path.insert(0, REF_COPY)
    import src                                                   # the reference package (oracle/_ref/src)
    assert os.path.realpath(os.path.dirname(src.__file__)).startswith(os.path.realpath(REF_COPY))
    sys.modules['src.neural_point'] = b.neural_point             # the swap of INTEGRATION.md section 1
    sys.modules['src.conv_onet'] = b.conv_onet
    sys.modules['src.conv_onet.models'] = b.conv_onet.models
    sys.modules['src.conv_onet.models.decoder'] = b.conv_onet.models.decoder
    sys.modules['src.utils.Renderer'] = b.utils.Renderer
    cwd = os.getcwd()
    os.chdir(REF_COPY)
    try:
        import src.common as ref_common
        import src.Tracker as ref_tracker
        import src.Mapper as ref_mapper
    finally:
        os.chdir(cwd)
    return ref_tracker.Tracker, ref_mapper.Mapper, ref_common, ref_mapper


class ReplayTorch:
    """`torch` as seen by the reference's src/common.py: randint replays the recorded pixel draws (on the requested device)."""

    def __init__(self, draws):
        self.it = iter(draws)

    def __getattr__(self, name):
        return getattr(torch, name)

    def randint(self, high, size, device=None, **kw):
        d = torch.as_tensor(next(self.it))
        assert d.shape[0] == size[0]
        return d.to(device or 'cpu')


def recording_adam():
    class RecordingAdam(torch.optim.Adam):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            self.snapshots = []

        def step(self, closure=None):
            self.snapshots.append([[None if p.grad is None else p.grad.detach().clone() for p in g['params']]
                                   for g in self.param_groups])
            return super().step(closure)
    return RecordingAdam


class TorchWithAdam:
    def __init__(self, adam_cls):
        self.made = []

        def make(*a, **kw):
            o = adam_cls(*a, **kw)
            self.made.append(o)
            return o
        import types
        self.optim = types.SimpleNamespace(Adam=make)

    def __getattr__(self, name):
        return getattr(torch, name)


# ---------------------------------------------------------------------------------------------------------------------
# float64 truth for the caller goldens: the oracle port of the callers' iterations (pinned to the goldens by
# tests/test_oracle_callers.py) evaluated in float64 at the SAME state -- gives the fp32 rounding noise of the reference itself,
# below which no fp32 implementation can be asked to agree (same rule as tests/test_gpu_parity.py)
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_render(P, cloud, S, rg, rc, encode_rel_pos=True):
    from oracle import point_slam_oracle as O

    def render(npc, decoders, rays_d, rays_o, device, stage, gt_depth=None, npc_geo_feats=None, npc_col_feats=None,
               is_tracker=False, cloud_pos=None, dynamic_r_query=None, exposure_feat=None):
        return O.render_batch_ray(P, rays_d, rays_o, gt_depth, stage, cloud, npc_geo_feats, npc_col_feats, S=S, is_tracker=is_tracker,
                                  radius_query=0.08, dynamic_r_query=dynamic_r_query, rand_geo=rg, rand_col=rc, coef=0.1,
                                  encode_rel_pos=encode_rel_pos)
    return render


def tracker_truth(g, k, dtype=torch.float64):
    """Loss and d loss / d [quat, T] of tracking iteration k of caller_tracker.npz at the pose the reference evaluated it at."""
    from point_slam_b200 import iteration as IT
    scene = C.load_scene(dtype)
    P = C.load_params(False, dtype)
    cam = torch.from_numpy(g['cam0'] if k == 0 else g[f'cam_after{k - 1}']).to(dtype).requires_grad_(True)
    depth = torch.from_numpy(full_image(g['depth_win'])).to(dtype)
    color = torch.from_numpy(full_image(g['color_win'])).to(dtype)
    rq = torch.from_numpy(full_radius(g['r_query_win']))
    opt = torch.optim.SGD([cam], lr=0.0)
    grads = {}
    orig = opt.step

    def step():
        grads['cam'] = cam.grad.clone()
        return orig()
    opt.step = step
    render = _oracle_render(P, scene['cloud'], 5, torch.from_numpy(g[f'rand_geo{k}']), torch.from_numpy(g[f'rand_col{k}']))
    with replay_randint([g[f'pix{k}']]):
        loss, _ = IT.tracker_iteration(render, None, None, cam, opt, color, depth, rq, INTR, int(g['n_pixels']), 'cpu', scene['geo_feats'],
                                       scene['col_feats'], scene['cloud'], edge=tuple(int(v) for v in g['edge']), w_color=float(g['w_color']))
    return loss.detach(), grads['cam']
