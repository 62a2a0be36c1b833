"""GPU parity tests (B200): the CUDA path, called through the drop-in API -> ctypes -> C ABI, against the CPU oracle.

Tolerances.  kNN: bit-exact (indices, distances, counts).  Floating point: the north-star bar is 1e-4 relative.
The reference itself is fp32; evaluating the SAME algorithm in fp64 (oracle, dtype=float64) shows that fp32
rounding alone moves some gradients by up to ~2.6e-4 (tests/test_oracle_vs_golden.py::test_fp64_noise_floor).
A quantity therefore passes when  err(gpu, fp64 truth) <= max(1e-4, 3 * err(fp32 oracle, fp64 truth)),
err = max|a-b| / max|b|.
"""
import numpy as np
import pytest
import torch

from tests import cases as C

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


_CASE = ['']
_WORST = {}


def _tol(name, got, o32, o64, floor=1e-4, param=False):
    """Checks one quantity and records the achieved error ($PSL_PARITY_JSON, written by tests/conftest.py).  The ~50
    decoder-parameter gradients of a case are recorded as ONE row (the worst), the other quantities one row each."""
    from tests.callers import Errors
    e_gpu = C.rel_err(got.detach().cpu(), o64)
    e_ref = C.rel_err(o32, o64)
    lim = max(floor, 3 * e_ref)
    if param:
        w = _WORST.setdefault(_CASE[0], dict(case=_CASE[0], quantity='worst decoder-parameter gradient (vs oracle64)', err=0.0, limit=0.0,
                                             flat_limit=floor, fp32_noise=0.0, ok=True, which=''))
        if e_gpu / lim >= w['err'] / max(w['limit'], 1e-30):
            w.update(err=float(e_gpu), limit=float(lim), fp32_noise=float(e_ref), which=name)
        w['ok'] = w['ok'] and e_gpu <= lim
    else:
        Errors.rows.append(dict(case=_CASE[0], quantity=name + ' (vs oracle64)', err=float(e_gpu), limit=float(lim), flat_limit=floor,
                                fp32_noise=float(e_ref), ok=bool(e_gpu <= lim)))
    assert e_gpu <= lim, f'{name}: gpu-vs-fp64 {e_gpu:.3e} > {lim:.3e} (fp32 oracle-vs-fp64 {e_ref:.3e})'
    return e_gpu


@pytest.fixture(scope='module')
def oracle_cache():
    return {}


def _oracles(name, cache):
    if name not in cache:
        c = C.load_case(name)
        cache[name] = (c, C.run_oracle(c, torch.float32), C.run_oracle(c, torch.float64))
    return cache[name]


def test_knn_bit_exact_golden_scene():
    from point_slam_b200 import ops
    from oracle import point_slam_oracle as O
    scene = C.load_scene()
    cloud = scene['cloud']
    grid = ops.SpatialHash(0.08).build(cloud.to(DEV))
    g = torch.Generator().manual_seed(3)
    # queries: near the surface (cloud points + jitter), exact duplicates of cloud points (ties at D=0), far points
    q = torch.cat([cloud[torch.randint(0, cloud.shape[0], (3000,), generator=g)] + 0.03 * torch.randn(3000, 3, generator=g),
                   cloud[:200], cloud.mean(0) + 5.0 + torch.randn(50, 3, generator=g)], 0)
    for radius, dyn in ((0.08, None), (0.04, None), (None, 0.04 + 0.12 * torch.rand(q.shape[0], generator=g, dtype=torch.float64))):
        D, I, n = ops.knn_query(grid, q.to(DEV), radius=radius or 0.08, dynamic_radius=None if dyn is None else dyn.to(DEV))
        Do, Io, no = O.find_neighbors(cloud, q, radius or 0.08, dyn)
        r2 = O.radius_sq_f64(q.shape[0], radius, dyn)
        inr = Do.double() <= r2[:, None]
        Ie = torch.where(inr, Io, torch.full_like(Io, -1))
        De = torch.where(inr, Do, torch.full_like(Do, torch.finfo(torch.float32).max))
        assert torch.equal(I.cpu().long(), Ie)
        assert torch.equal(D.cpu(), De)
        assert torch.equal(n.cpu(), no)


def test_knn_bit_exact_large_cloud():
    from point_slam_b200 import ops, synth
    from oracle import point_slam_oracle as O
    from scipy.spatial import cKDTree
    cloud = torch.from_numpy(synth.make_cloud(300000, seed=5))
    grid = ops.SpatialHash(0.08).build(cloud.to(DEV))
    poses = synth.trajectory(3, seed=5)
    depth, color = synth.make_frame(poses[1])
    o, d = synth.pixel_rays(poses[1], 480, 640, 517.3, 516.5, 318.6, 255.3)
    rng = np.random.default_rng(0)
    pix = rng.integers(0, 480 * 640, 3000)
    dep = depth.reshape(-1)[pix]
    z = dep[:, None] * np.linspace(0.98, 1.02, 5)[None, :]
    q = torch.from_numpy((o[None, None, :] + d.reshape(-1, 3)[pix][:, None, :] * z[..., None]).reshape(-1, 3).astype(np.float32))
    _, rq = synth.sobel_radius_map(color)
    dyn = torch.from_numpy(rq.reshape(-1)[pix])
    D, I, n = ops.knn_query(grid, q.to(DEV), dynamic_radius=dyn.to(DEV), group=5)
    tree = cKDTree(cloud.double().numpy())
    Do, Io, no = O.find_neighbors(cloud, q, 0.08, dyn.repeat_interleave(5), tree=tree)
    r2 = (dyn.repeat_interleave(5) ** 2)
    inr = Do.double() <= r2[:, None]
    assert torch.equal(I.cpu().long(), torch.where(inr, Io, torch.full_like(Io, -1)))
    assert torch.equal(D.cpu(), torch.where(inr, Do, torch.full_like(Do, torch.finfo(torch.float32).max)))
    assert torch.equal(n.cpu(), no)


def test_knn_distance_ties_resolve_to_the_smaller_index():
    """Exact distance ties (duplicated cloud points, and points mirrored around the query): the list merge compares the 32-bit
    distance first and falls back to the index only on equality -- the reported order must be (distance, index) ascending like
    the oracle's stable sort, for every query."""
    from point_slam_b200 import ops
    g = torch.Generator().manual_seed(11)
    base = torch.rand(4000, 3, generator=g) * 0.5
    cloud = torch.cat([base, base[:1500], base[200:900]], 0)                  # duplicates at higher indices
    q = base[::3][:1200].clone()
    q[::2] += 0.004                                                           # half of the queries sit exactly on cloud points
    grid = ops.SpatialHash(0.08).build(cloud.to(DEV))
    D, I, n = ops.knn_query(grid, q.to(DEV), radius=0.08)
    qf, cf = q.float(), cloud.float()                                         # reference order: canonical fp32 distance, then index
    dx, dy, dz = (qf[:, None, 0] - cf[None, :, 0]), (qf[:, None, 1] - cf[None, :, 1]), (qf[:, None, 2] - cf[None, :, 2])
    dist = (dx * dx + dy * dy) + dz * dz
    order = torch.argsort(dist, dim=1, stable=True)[:, :8]                    # stable: equal distances stay in index order
    dref = torch.gather(dist, 1, order)
    inr = dref <= torch.tensor(0.08, dtype=torch.float32) ** 2
    assert int((dref[:, 1:] == dref[:, :-1]).sum()) > 500                     # the case really has ties
    assert torch.equal(I.cpu().long(), torch.where(inr, order, torch.full_like(order, -1)))
    assert torch.equal(D.cpu(), torch.where(inr, dref, torch.full_like(dref, torch.finfo(torch.float32).max)))


def test_incremental_hash_append_is_bit_identical_to_full_rebuild():
    """psl_grid_append (sort the new points + stable merge) == psl_grid_sort on the whole cloud: same sorted copy, same keys, same
    neighbours; several appends in a row, including points that fall into already occupied cells (duplicates of old positions)."""
    from point_slam_b200 import ops, synth
    cloud = torch.from_numpy(synth.make_cloud(120000, seed=9)).to(DEV)
    extra = cloud[torch.randperm(120000, device=DEV)[:3000]] + 1e-3            # same cells as existing points, mostly
    buf = torch.empty((200000, 3), device=DEV)
    buf[:120000] = cloud
    inc = ops.SpatialHash(0.08)
    inc.reserve(200000, DEV)
    n = 90000
    inc.build(buf[:n])
    assert inc.incremental_builds == 0
    q = cloud[::7][:20000].contiguous() + 0.01
    for step, k in enumerate((1, 777, 20000, 9222, 3000)):
        if step == 4:
            buf[n:n + k] = extra
        inc.build(buf[:n + k], appended_from=n)
        n += k
        full = ops.SpatialHash(0.08).build(buf[:n].clone())
        assert inc.incremental_builds == step + 1
        assert torch.equal(inc.sorted_pts[:n].view(torch.int32), full.sorted_pts[:n].view(torch.int32))
        assert torch.equal(inc._keys[:n], full._keys[:n])
        assert (inc.struct.n, inc.struct.capacity) == (full.struct.n, full.struct.capacity)
        a = ops.knn_query(inc, q, radius=0.08)
        b = ops.knn_query(full, q, radius=0.08)
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    # a caller that does NOT vouch for the old rows gets the full sort
    inc.build(buf[:n])
    assert inc.incremental_builds == 5


def test_composite_matches_reference_vectors():
    from point_slam_b200 import ops
    z = np.load(C.GOLDEN + '/aux.npz')
    raw = torch.from_numpy(z['comp_raw']).to(DEV).requires_grad_(True)
    zv = torch.from_numpy(z['comp_z']).to(DEV)
    d, v, rgb, w = ops.composite(raw, zv, None, 0.1)
    for a, b in ((d, 'comp_depth'), (v, 'comp_var'), (rgb, 'comp_rgb'), (w, 'comp_w')):
        assert C.rel_err(a.detach().cpu(), z[b]) < 2e-6, b
    # backward against autograd of the oracle restatement
    from oracle import point_slam_oracle as O
    r2 = torch.from_numpy(z['comp_raw']).double().requires_grad_(True)
    do, vo, co, _ = O.composite(r2, torch.from_numpy(z['comp_z']).double())
    g = torch.Generator().manual_seed(1)
    gd, gv, gc = torch.randn(64, generator=g), torch.randn(64, generator=g), torch.randn(64, 3, generator=g)
    (do * gd.double()).sum().add((vo * gv.double()).sum()).add((co * gc.double()).sum()).backward()
    ((d * gd.to(DEV)).sum() + (v * gv.to(DEV)).sum() + (rgb * gc.to(DEV)).sum()).backward()
    assert C.rel_err(raw.grad.cpu(), r2.grad) < 1e-5


@pytest.mark.parametrize('name', C.CASES + C.EXPO_CASES)
def test_render_case_against_oracle(name, oracle_cache):
    from tests.gpu_harness import run_case_gpu
    c, o32, o64 = _oracles(name, oracle_cache)
    got = run_case_gpu(c)
    _CASE[0] = 'case_' + name
    assert torch.equal(got['valid'].cpu(), o32['valid'])
    _tol('depth', got['depth'], o32['depth'], o64['depth'])
    _tol('color', got['color'], o32['color'], o64['color'])
    _tol('var', got['var'], o32['var'], o64['var'])
    _tol('loss', got['loss'], o32['loss'], o64['loss'])
    if 'grad_cam' in o64:
        _tol('pose grad', got['grad_cam'], o32['grad_cam'], o64['grad_cam'])
    if 'grad_exposure_feat' in o64:
        _tol('exposure grad', got['grad_exposure_feat'], o32['grad_exposure_feat'], o64['grad_exposure_feat'])
    if not c['is_tracker'] or True:
        _tol('geo feature grad', got['grad_geo'], o32['grad_geo'], o64['grad_geo'])
        if c['stage'] == 'color':
            _tol('col feature grad', got['grad_col'], o32['grad_col'], o64['grad_col'])
    checked = 0
    for k, g64 in o64['grad_params'].items():
        if k == 'color_decoder.embedder._B' or k not in got['grad_params']:
            assert k == 'color_decoder.embedder._B' or float(g64.abs().max()) == 0.0, f'missing gradient for {k}'
            continue
        _tol(k, got['grad_params'][k], o32['grad_params'][k], o64['grad_params'][k], param=True)
        checked += 1
    if 'case_' + name in _WORST:
        from tests.callers import Errors
        Errors.rows.append(_WORST['case_' + name])
    assert checked >= (20 if c['stage'] == 'geometry' else 40)


def test_backward_is_bit_deterministic():
    from tests.gpu_harness import run_case_gpu, build_objects
    c = C.load_case('mapper_color')
    objs = build_objects(c)
    a = run_case_gpu(c, objs)
    b = run_case_gpu(c, objs)
    assert torch.equal(a['grad_geo'], b['grad_geo']) and torch.equal(a['grad_col'], b['grad_col'])
    for k in a['grad_params']:
        assert torch.equal(a['grad_params'][k], b['grad_params'][k]), k


def test_point_forward_matches_fused_render():
    """POINT.forward + raw2outputs (the un-fused API the reference Renderer would call) == fused render."""
    from tests.gpu_harness import build_objects
    from point_slam_b200.src import common
    c = C.load_case('mapper_color')
    cfg, decoders, npc, renderer = build_objects(c)
    t = lambda k, dt=torch.float32: torch.from_numpy(np.asarray(c[k])).to(device=DEV, dtype=dt)
    rg, rc = t('rand_geo'), t('rand_col')
    decoders.draw_no_neighbor_vectors = lambda stage, device: (rg, rc if stage == 'color' else None)
    rays_o, rays_d, gt_depth, dyn = t('rays_o'), t('rays_d'), t('gt_depth'), t('dynamic_r_query', torch.float64)
    with torch.no_grad():
        d1, v1, c1, m1 = renderer.render_batch_ray(npc, decoders, rays_d, rays_o, DEV, 'color', gt_depth=gt_depth,
                                                   npc_geo_feats=npc.get_geo_feats(), npc_col_feats=npc.get_col_feats(),
                                                   cloud_pos=npc.cloud_pos_tensor(), dynamic_r_query=dyn)
        S = c['S']
        tv = torch.linspace(0., 1., S, device=DEV)
        z = 0.98 * gt_depth[:, None] * (1. - tv) + 1.02 * gt_depth[:, None] * tv
        pts = (rays_o[:, None, :] + rays_d[:, None, :] * z[..., None]).reshape(-1, 3)
        raw, ray_mask, point_mask = renderer.eval_points(pts, decoders, npc, 'color', DEV, npc.get_geo_feats(),
                                                         npc.get_col_feats(), False, npc.cloud_pos_tensor(), None,
                                                         ray_pts_num=S, dynamic_r_query=dyn.repeat_interleave(S))
        raw[~point_mask, 3] = -100.0
        d2, v2, c2, _ = common.raw2outputs_nerf_color(raw.reshape(-1, S, 4), z, rays_d, device=DEV, coef=0.1)
    assert torch.equal(m1, ray_mask)
    assert torch.allclose(d1, d2, rtol=1e-6, atol=0) and torch.allclose(c1, c2, rtol=1e-6, atol=1e-7)


def test_add_neural_points_and_sample_near_pcl():
    from tests.gpu_harness import build_objects
    z = np.load(C.GOLDEN + '/aux.npz')
    c = C.load_case('mapper_color')
    cfg, decoders, npc, renderer = build_objects(c)
    ro, rd, gd = (torch.from_numpy(z[k]).to(DEV) for k in ('add_rays_o', 'add_rays_d', 'add_depth'))
    r_add = torch.from_numpy(z['add_r_add']).to(DEV)
    col = torch.zeros(ro.shape[0], 3, device=DEV)
    n0 = npc.pts_num()
    zz, inv = npc.sample_near_pcl(ro[:96].clone(), rd[:96].clone(), 0.3, torch.tensor(4.2), 5)
    assert np.array_equal(inv.cpu().numpy(), z['snp_invalid'])
    assert np.allclose(zz.cpu().numpy(), z['snp_z'], rtol=0, atol=1e-6)
    k1 = npc.add_neural_points(ro, rd, gd, col, dynamic_radius=r_add[gd > 0])
    n1 = npc.pts_num()
    k2 = npc.add_neural_points(ro, rd, gd, col, is_pts_grad=True)
    assert int(k1) == int(z['add_kept1']) and int(k2) == int(z['add_kept2'])
    cp = np.asarray(npc.cloud_pos(), dtype=np.float32)
    assert np.array_equal(cp[n0:n1], z['add_new1']) and np.array_equal(cp[n1:], z['add_new2'])
    assert npc.get_geo_feats().shape[0] == npc.pts_num() == npc.index_ntotal()
    assert np.array_equal(np.asarray(npc.input_pos(), np.float32), z['add_input_pos'])

