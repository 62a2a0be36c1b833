"""Host-side wrappers over the C ABI: spatial hash, kNN, fused render (autograd), decode (autograd), composite.

PyTorch is used for device memory, streams and the autograd graph only; every arithmetic step of the hot path runs
in libpointslam_b200.so.  There is no CPU / eager fallback.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math
import os
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib as L

PARAM_ORDER = (['g_B'] + [f'g_W{i}' for i in range(5)] + [f'g_b{i}' for i in range(5)] +
               [f'g_Wc{i}' for i in range(5)] + [f'g_bc{i}' for i in range(5)] + ['g_Wo', 'g_bo', 'c_B', 'c_Brel',
               'c_N1', 'c_n1b', 'c_N2', 'c_n2b'] + [f'c_W{i}' for i in range(5)] + [f'c_b{i}' for i in range(5)] +
               [f'c_Wc{i}' for i in range(5)] + [f'c_bc{i}' for i in range(5)] + ['c_Wo', 'c_bo'])
assert len(PARAM_ORDER) == L.N_PARAMS


def decoder_param_list(decoders) -> List[torch.Tensor]:
    """The 51 tensors of a POINT module in psl_decoder_params order (reference names in the comments of
    include/pointslam_b200.h)."""
    g, c = decoders.geo_decoder, decoders.color_decoder
    out = [g.embedder._B]
    out += [g.pts_linears[i].weight for i in range(5)] + [g.pts_linears[i].bias for i in range(5)]
    out += [g.fc_c[i].weight for i in range(5)] + [g.fc_c[i].bias for i in range(5)]
    out += [g.output_linear.weight, g.output_linear.bias]
    out += [c.embedder._B, c.embedder_rel_pos._B, c.mlp_col_neighbor.linear1.weight, c.mlp_col_neighbor.linear1.bias,
            c.mlp_col_neighbor.linear2.weight, c.mlp_col_neighbor.linear2.bias]
    out += [c.pts_linears[i].weight for i in range(5)] + [c.pts_linears[i].bias for i in range(5)]
    out += [c.fc_c[i].weight for i in range(5)] + [c.fc_c[i].bias for i in range(5)]
    out += [c.output_linear.weight, c.output_linear.bias]
    return out


def state_dict_param_list(P: dict, device) -> List[torch.Tensor]:
    """Same list from a flat dict keyed like the reference state_dict (+ 'color_decoder.embedder._B')."""
    g, c = 'geo_decoder.', 'color_decoder.'
    keys = [g + 'embedder._B'] + [g + f'pts_linears.{i}.weight' for i in range(5)] + \
        [g + f'pts_linears.{i}.bias' for i in range(5)] + [g + f'fc_c.{i}.weight' for i in range(5)] + \
        [g + f'fc_c.{i}.bias' for i in range(5)] + [g + 'output_linear.weight', g + 'output_linear.bias'] + \
        [c + 'embedder._B', c + 'embedder_rel_pos._B', c + 'mlp_col_neighbor.linear1.weight',
         c + 'mlp_col_neighbor.linear1.bias', c + 'mlp_col_neighbor.linear2.weight', c + 'mlp_col_neighbor.linear2.bias'] + \
        [c + f'pts_linears.{i}.weight' for i in range(5)] + [c + f'pts_linears.{i}.bias' for i in range(5)] + \
        [c + f'fc_c.{i}.weight' for i in range(5)] + [c + f'fc_c.{i}.bias' for i in range(5)] + \
        [c + 'output_linear.weight', c + 'output_linear.bias']
    return [P[k].to(device=device, dtype=torch.float32).contiguous() for k in keys]


def _param_struct(tensors: Sequence[Optional[torch.Tensor]]) -> L.DecoderParams:
    s = L.DecoderParams()
    flat = [None if t is None else t.data_ptr() for t in tensors]
    it = iter(flat)
    for name, ctype in L.DecoderParams._fields_:
        if ctype is L._vp:
            setattr(s, name, next(it))
        else:
            arr = getattr(s, name)
            for i in range(5):
                arr[i] = next(it)
    return s


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


# ------------------------------------------------------------------------------------------------------------------
# spatial hash
# ------------------------------------------------------------------------------------------------------------------
class SpatialHash:
    """GPU-resident hash grid over the neural point cloud (K0).  Rebuilt on every append (about 0.2 ms for 500 k points);
    point indices are stable (the grid stores a sorted copy carrying the original index).

    All device buffers (sorted copy, table, sort scratch) are allocated for a CAPACITY of points and re-used by every
    rebuild; the three numbers that change with a rebuild (table size in use, point count, first-pass radius) are also kept
    in a 16-byte device block (`psl_grid_meta`) that the kernels read at run time.  A CUDA graph captured over this hash
    therefore stays valid while the cloud grows: `alloc_gen` changes only when a rebuild had to re-allocate (capacity
    doubling), `build_gen` counts every rebuild (the reference re-trains / re-adds its faiss index the same way,
    neural_point.py:161-164)."""

    def __init__(self, cell: float = 0.08, two_pass: bool = True):
        self.cell = float(cell)
        self.two_pass = two_pass
        self.n = 0
        self.cap_points = 0
        self.sorted_pts = self.table_keys = self.table_vals = self._keys = self._ws = self.meta = None
        self._meta_host = None
        self.capacity = 0                 # table entries in use (power of two)
        self.table_alloc = 0              # table entries allocated
        self.n_cells = 0
        self.r_small = 0.0
        self.alloc_gen = 0
        self.build_gen = 0
        self._covered, self._covered_ptr = 0, 0       # points (and their buffer) the sorted copy currently covers
        self.incremental_builds = 0
        self.struct = L.Grid(None, None, None, 0, 0, self.cell, 0.0, None)

    def reserve(self, n_points: int, device):
        """Buffers for up to `n_points` points (doubling growth).  Returns True when something was re-allocated."""
        if n_points <= self.cap_points and self.sorted_pts is not None:
            return False
        lib = L.load()
        cap = max(int(n_points), 2 * self.cap_points, 1024)
        self.cap_points = cap
        self.sorted_pts = torch.empty((cap, 4), dtype=torch.float32, device=device)
        self._keys = torch.empty(cap, dtype=torch.int64, device=device)
        self._ws_bytes = max(lib.psl_grid_sort_ws_bytes(cap), lib.psl_grid_append_ws_bytes(cap, max(cap // 4, 1)))
        self._covered = 0                              # the old sorted copy is not carried over
        self._ws = torch.empty(self._ws_bytes, dtype=torch.uint8, device=device)
        self.table_alloc = 1 << max(4, int(math.ceil(math.log2(2 * cap))))      # worst case: every point in its own cell
        self.table_keys = torch.empty(self.table_alloc, dtype=torch.int64, device=device)
        self.table_vals = torch.empty((self.table_alloc, 2), dtype=torch.int32, device=device)
        if self.meta is None:
            self.meta = torch.zeros(4, dtype=torch.int32, device=device)
            self._meta_host = torch.zeros(4, dtype=torch.int32).pin_memory() if torch.cuda.is_available() else torch.zeros(4, dtype=torch.int32)
        self.alloc_gen += 1
        return True

    def build(self, cloud_pos: torch.Tensor, appended_from: int = 0):
        """Cover `cloud_pos`.  `appended_from` = k > 0 is the caller's statement that rows [0, k) are exactly the rows of the previous
        build (same storage, unchanged): only rows [k, n) are sorted and merged in (psl_grid_append)."""
        lib = L.load()
        pos = _f32c(cloud_pos).reshape(-1, 3)
        n = pos.shape[0]
        dev = pos.device
        self.n = n
        self.build_gen += 1
        if n == 0:
            self.struct = L.Grid(None, None, None, 0, 0, self.cell, 0.0, None)
            self._covered = 0
            return self
        n_old = self._covered
        realloc = self.reserve(n, dev)
        n_cells = C.c_int64(0)
        if (INCREMENTAL_HASH and not realloc and 0 < n_old < n and appended_from == n_old and (n - n_old) * 4 <= n and
                self._covered_ptr == pos.data_ptr() and lib.psl_grid_append_ws_bytes(n, n - n_old) <= self._ws_bytes):
            # an append to the cloud this hash already covers: sort the new points only and merge (bit-identical to a full sort)
            L.check(lib.psl_grid_append(L.ptr(pos), n_old, n - n_old, self.cell, L.ptr(self.sorted_pts), L.ptr(self._keys), L.ptr(self._ws),
                                        self._ws_bytes, C.byref(n_cells), L.stream()), 'psl_grid_append')
            self.incremental_builds += 1
        else:
            L.check(lib.psl_grid_sort(L.ptr(pos), n, self.cell, L.ptr(self.sorted_pts), L.ptr(self._keys), L.ptr(self._ws),
                                      self._ws_bytes, C.byref(n_cells), L.stream()), 'psl_grid_sort')
        self._covered, self._covered_ptr = n, pos.data_ptr()
        cap = 1 << max(4, int(math.ceil(math.log2(max(2 * n_cells.value, 2)))))
        assert cap <= self.table_alloc
        self.capacity = cap
        L.check(lib.psl_grid_hash(L.ptr(self._keys), n, L.ptr(self.table_keys), L.ptr(self.table_vals), cap, L.stream()),
                'psl_grid_hash')
        self.n_cells = n_cells.value
        # first-pass radius: expect ~32 points inside it, estimated from the mean occupancy of the occupied cells
        # (a cell of edge h cuts ~1.5 h^2 of surface); clamped to [h/4, h]
        self.r_small = 0.0
        if self.two_pass:
            rs = math.sqrt(32.0 * 1.5 * self.cell ** 2 * max(self.n_cells, 1) / (math.pi * n))
            self.r_small = float(min(max(rs, self.cell / 4), self.cell))
        # device copy of (capacity, n, r_small): stream-ordered after the rebuild, before the next query
        self._meta_host[0] = cap if cap < (1 << 31) else cap - (1 << 32)
        self._meta_host[1] = n
        self._meta_host[2:3] = torch.tensor([self.r_small], dtype=torch.float32).view(torch.int32)
        self.meta.copy_(self._meta_host, non_blocking=True)
        self.struct = L.Grid(self.sorted_pts.data_ptr(), self.table_keys.data_ptr(), self.table_vals.data_ptr(),
                             cap, n, self.cell, self.r_small, self.meta.data_ptr())
        return self


def _r2_args(radius, dynamic_radius, M_groups, device):
    """(r2 tensor or None, r2_scalar) with the comparison semantics of neural_point.py:208-213."""
    if dynamic_radius is not None:
        # squared in the tensor's own dtype (the reference squares before the promoting comparison), then float64
        r2 = (dynamic_radius.detach().reshape(-1).to(device=device) ** 2).to(torch.float64).contiguous()
        assert r2.shape[0] == M_groups, 'shape mis-match for input points and dynamic radius'
        return r2, 0.0
    return None, float(np.float32(radius ** 2))


def knn_query(grid: SpatialHash, pos: torch.Tensor, radius: float = 0.08, dynamic_radius=None, group: int = 1):
    """find_neighbors_faiss kernel (a5): -> D (M,8) f32, I (M,8) i32, neighbor_num (M,) i32.
    `group`: consecutive queries that belong together (samples of one ray); dynamic_radius then has M/group rows."""
    lib = L.load()
    pos = _f32c(pos).reshape(-1, 3)
    M = pos.shape[0]
    dev = pos.device
    I = torch.empty((M, 8), dtype=torch.int32, device=dev)
    D = torch.empty((M, 8), dtype=torch.float32, device=dev)
    nn = torch.empty((M,), dtype=torch.int32, device=dev)
    if M == 0:
        return D, I, nn
    r2, r2s = _r2_args(radius, dynamic_radius, (M + group - 1) // group if dynamic_radius is not None else 0, dev)
    L.check(lib.psl_knn_query(C.byref(grid.struct), L.ptr(pos), M, L.ptr(r2), r2s, int(group), L.ptr(I), L.ptr(D),
                              L.ptr(nn), L.stream()), 'psl_knn_query')
    return D, I, nn


def raymarch_knn_stats(grid: SpatialHash, rays_o, rays_d, gt_depth, S, r2_ray=None, radius=0.08, near=0.98, far=1.02):
    """Work counters of one ray-march + kNN launch (bench.py): -> dict with the mean number of candidate points staged per query
    (C-bar of SURVEY.md section 8d), hash cells probed per query and the share of warps that needed the second search pass."""
    lib = L.load()
    ro, rd, dep = _f32c(rays_o).reshape(-1, 3), _f32c(rays_d).reshape(-1, 3), _f32c(gt_depth).reshape(-1)
    R = ro.shape[0]
    dev = ro.device
    M = R * S
    z = torch.empty((R, S), dtype=torch.float32, device=dev); pos = torch.empty((M, 3), dtype=torch.float32, device=dev)
    I = torch.empty((M, 8), dtype=torch.int32, device=dev); D = torch.empty((M, 8), dtype=torch.float32, device=dev)
    nn = torch.empty((M,), dtype=torch.int32, device=dev)
    stats = torch.zeros(4, dtype=torch.int64, device=dev)
    L.check(lib.psl_raymarch_knn_stats(C.byref(grid.struct), L.ptr(ro), L.ptr(rd), L.ptr(dep), R, S, L.ptr(surface_t_vals(S, dev)),
                                       near, far, None, L.ptr(r2_ray), float(np.float32(radius ** 2)), L.ptr(z), L.ptr(pos), L.ptr(I),
                                       L.ptr(D), L.ptr(nn), L.ptr(stats), L.stream()), 'psl_raymarch_knn_stats')
    c, passes, q, cells = (int(x) for x in stats.tolist())
    warps = (R * ((S + 31) // 32))
    return {'queries': q, 'candidates_per_query': c / max(q, 1), 'cells_probed_per_query': cells / max(q, 1),
            'second_pass_share_of_warps': max(passes - warps, 0) / max(warps, 1), 'candidate_bytes_per_query': 16.0 * c / max(q, 1)}


_T_VALS = {}


def surface_t_vals(S: int, device) -> torch.Tensor:
    """linspace(0,1,S) evaluated by torch on the CPU (bit-identical to the oracle), cached per device."""
    key = (S, str(device))
    if key not in _T_VALS:
        _T_VALS[key] = torch.linspace(0.0, 1.0, steps=S, dtype=torch.float32).to(device)
    return _T_VALS[key]


class RenderSettings:
    """Static (non-tensor) arguments of one render call."""

    def __init__(self, stage='color', S=5, near_surface=0.98, far_surface=1.02, radius_query=0.08, coef=0.1,
                 encode_rel_pos=True, rgb_mode=L.RGB_SIGMOID, weighting='distance', min_nn=2, is_tracker=False):
        self.stage, self.S = stage, int(S)
        self.near_surface, self.far_surface = float(near_surface), float(far_surface)
        self.radius_query, self.coef = float(radius_query), float(coef)
        self.encode_rel_pos, self.rgb_mode = bool(encode_rel_pos), int(rgb_mode)
        self.weighting, self.min_nn, self.is_tracker = weighting, int(min_nn), bool(is_tracker)
        self.grad_mode = True

    def cfg(self, r2_group, r2_scalar):
        return L.DecodeCfg(L.STAGE[self.stage], int(self.encode_rel_pos), self.rgb_mode, L.WEIGHTING[self.weighting],
                           self.min_nn, int(r2_group), int(self.is_tracker), 0, float(r2_scalar))


USE_TENSOR_CORES = os.environ.get('PSL_TC', '1') != '0'      # tcgen05 colour branch (forward)
USE_TC_BACKWARD = os.environ.get('PSL_TC_BWD', '1') != '0'    # tcgen05 colour-branch backward (data gradients)
USE_TC_WGRAD = os.environ.get('PSL_TC_WGRAD', '1') != '0'     # tcgen05 weight-gradient GEMMs of the colour branch
USE_GEO_MMA = os.environ.get('PSL_GEO_MMA', '1') != '0'           # geometry branch on mma.sync 3xTF32 when its parameters are frozen
WARM_ALLOCATOR = os.environ.get('PSL_WARM_ALLOC', '1') != '0'     # pre-fill the caching allocator's pools after a graph capture
INCREMENTAL_HASH = os.environ.get('PSL_HASH_APPEND', '1') != '0'   # add_neural_points: sort + merge the new points only (psl_grid_append)
USE_H2_BACKWARD = os.environ.get('PSL_H2_BWD', '1') != '0'     # f16-plane colour backward with per-row gradient scaling (psl_color_bwd_h2.cu)
USE_H2_FORWARD = os.environ.get('PSL_H2', '1') != '0'           # f16-plane, two-tiles-in-flight colour forward (psl_color_h2.cu)
OVERLAP_BRANCHES = os.environ.get('PSL_OVERLAP', '1') != '0'  # geometry kernel on a forked stream next to the colour kernel
_SIDE = {}


def _side_stream(device):
    key = str(device)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device)
    return _SIDE[key]


class PackedDecoder:
    """Device images of the decoder parameters in the kernels' operand layouts (FFMA blob, tcgen05 forward and backward
    blobs).  The render calls re-pack into the per-device default instance on every call; a caller that knows the
    parameters are frozen (tracking) packs ONCE into a private instance and passes it with prepacked=True."""

    def __init__(self, device):
        lib = L.load()
        self.packed = torch.empty(lib.psl_packed_params_floats(), dtype=torch.float32, device=device)
        self.blob = torch.empty(lib.psl_tc_blob_floats(), dtype=torch.float32, device=device)
        self.bblob = torch.empty(lib.psl_tc_bwd_blob_floats(), dtype=torch.float32, device=device)
        self.hblob = torch.empty(lib.psl_h2_blob_bytes(), dtype=torch.uint8, device=device)      # f16 hi/lo planes (psl_color_h2.cu)
        self.bhblob = torch.empty(lib.psl_h2_bwd_blob_bytes(), dtype=torch.uint8, device=device)  # ... of the backward (psl_color_bwd_h2.cu)

    def pack_geometry(self, params):
        """FFMA blob + geometry fragment images only (render calls then pass prepacked='geometry')."""
        pstruct = _param_struct([_f32c(p.detach()) for p in params])
        L.check(L.load().psl_pack_params(C.byref(pstruct), L.ptr(self.packed), L.stream()), 'psl_pack_params')
        return self

    def pack(self, params, backward=True):
        lib = L.load()
        pstruct = _param_struct([_f32c(p.detach()) for p in params])
        L.check(lib.psl_pack_params(C.byref(pstruct), L.ptr(self.packed), L.stream()), 'psl_pack_params')
        _tc_fold_or_pack(lib, pstruct, self.blob)
        if USE_H2_FORWARD:
            L.check(lib.psl_h2_pack_params(C.byref(pstruct), L.ptr(self.blob), L.ptr(self.hblob), L.stream()), 'psl_h2_pack_params')
        if backward:
            if USE_H2_BACKWARD:
                L.check(lib.psl_h2_bwd_pack_params(C.byref(pstruct), L.ptr(self.blob), L.ptr(self.bhblob), L.stream()), 'psl_h2_bwd_pack_params')
            else:
                L.check(lib.psl_tc_bwd_pack_params(C.byref(pstruct), L.ptr(self.blob), lib.psl_tc_fold_offset_floats(), L.ptr(self.bblob),
                                                   L.stream()), 'psl_tc_bwd_pack_params')
        return self


def _tc_fold_or_pack(lib, pstruct, blob):
    """Folded fp32 rows + small vectors (all the f16-plane kernels read), plus the tf32 chunk images only when a 3xTF32 kernel is
    still selected (PSL_H2=0 / PSL_H2_BWD=0 A/B runs)."""
    if USE_H2_FORWARD and USE_H2_BACKWARD and USE_TC_BACKWARD and USE_TC_WGRAD and USE_TENSOR_CORES:
        L.check(lib.psl_tc_fold_params(C.byref(pstruct), L.ptr(blob), L.stream()), 'psl_tc_fold_params')
    else:
        L.check(lib.psl_tc_pack_params(C.byref(pstruct), L.ptr(blob), L.stream()), 'psl_tc_pack_params')


_DEFAULT_PACK = {}


def _default_pack(device):
    key = str(device)
    if key not in _DEFAULT_PACK:
        _DEFAULT_PACK[key] = PackedDecoder(device)
    return _DEFAULT_PACK[key]


def _fwd_flags(st, need_grad, colour_param_grads):
    """(use_tc, tc_bwd, use_h2) of a decode call -- which kernels run, hence which operand images they need"""
    use_tc = USE_TENSOR_CORES and st.stage == 'color' and st.weighting == 'distance'
    tc_bwd = use_tc and need_grad and USE_TC_BACKWARD and (USE_TC_WGRAD or not colour_param_grads)
    use_h2 = use_tc and USE_H2_FORWARD and (tc_bwd or not need_grad)
    return use_tc, tc_bwd, use_h2


def _pack_images(st, params, pk, prepacked, need_grad, colour_param_grads, backward=False):
    """Rebuild the operand images a render call needs (on the current stream).  prepacked: False = everything, 'geometry' = the
    colour images only (the FFMA blob + geometry fragments are current), True = nothing.  backward=True also rebuilds the image of
    the tensor-core backward (the caller then passes repack=False to render_backward)."""
    if prepacked is True:
        return
    lib = L.load()
    pstruct = _param_struct(params)
    if prepacked is False:
        L.check(lib.psl_pack_params(C.byref(pstruct), L.ptr(pk.packed), L.stream()), 'psl_pack_params')
    use_tc, tc_bwd, use_h2 = _fwd_flags(st, need_grad, colour_param_grads)
    if use_tc:
        _tc_fold_or_pack(lib, pstruct, pk.blob)
        if use_h2:
            L.check(lib.psl_h2_pack_params(C.byref(pstruct), L.ptr(pk.blob), L.ptr(pk.hblob), L.stream()), 'psl_h2_pack_params')
        if backward and tc_bwd:
            if USE_H2_BACKWARD:
                L.check(lib.psl_h2_bwd_pack_params(C.byref(pstruct), L.ptr(pk.blob), L.ptr(pk.bhblob), L.stream()), 'psl_h2_bwd_pack_params')
            else:
                L.check(lib.psl_tc_bwd_pack_params(C.byref(pstruct), L.ptr(pk.blob), lib.psl_tc_fold_offset_floats(), L.ptr(pk.bblob),
                                                   L.stream()), 'psl_tc_bwd_pack_params')


def _decode_forward(st: RenderSettings, cfg, params, pos, I, D, nn, r2, cloud_pos, geo, col, rand_geo, rand_col,
                    affine, need_grad, colour_param_grads=True, geo_param_grads=True, pack=None, prepacked=False):
    """-> raw, has_nb, save (FFMA layout or None), tsave (tensor-core layout or None), param struct"""
    lib = L.load()
    dev = pos.device
    M = pos.shape[0]
    pk = pack if pack is not None else _default_pack(dev)
    packed = pk.packed
    pstruct = _param_struct(params)
    # prepacked: True = every operand image is current; 'geometry' = the FFMA blob + geometry fragment images are (frozen geometry
    # decoder: packed once per frame), the colour images are rebuilt here; False = rebuild everything
    _pack_images(st, params, pk, prepacked, need_grad, colour_param_grads)
    raw = torch.empty((M, 4), dtype=torch.float32, device=dev)
    has_nb = torch.empty((M,), dtype=torch.uint8, device=dev)
    save = tsave = None
    use_tc, tc_bwd, use_h2 = _fwd_flags(st, need_grad, colour_param_grads)
    # geometry branch without parameter gradients (frozen geometry decoder): warp-level tensor-core kernels (psl_geo_mma.cu), which
    # keep one ReLU mask word per layer for the backward.  The choice travels to the backward in bit 1 of cfg.reserved.
    if USE_GEO_MMA and not (need_grad and geo_param_grads) and (use_tc or st.stage == 'geometry'):
        cfg.reserved |= 2
    geo_bit = cfg.reserved & 2
    if need_grad:
        scfg = L.DecodeCfg(L.STAGE['geometry'], cfg.encode_rel_pos, L.RGB_SIGMOID, cfg.weighting, cfg.min_nn, cfg.r2_group,
                           cfg.is_tracker, geo_bit, cfg.r2_scalar) if tc_bwd else cfg
        per = lib.psl_decode_save_floats_per_sample(C.byref(scfg))
        save = torch.empty(max(M * per, 1), dtype=torch.float32, device=dev)
        if tc_bwd:
            tsave = torch.empty(lib.psl_tc_save_floats(M, cfg.encode_rel_pos), dtype=torch.float32, device=dev)
    if use_tc:
        # the colour branch on tcgen05 and the geometry branch (fp32 FFMA kernel: occupancy, has_nb, geometry activations) are
        # independent (they write different words of `raw`): the geometry kernel runs on a forked stream and fills the SMs
        # the colour kernel's partial last wave leaves idle (25 000 samples = 196 tiles on 148 SMs; tracking: 59 tiles)
        gcfg = L.DecodeCfg(L.STAGE['geometry'], cfg.encode_rel_pos, L.RGB_SIGMOID, cfg.weighting, cfg.min_nn, cfg.r2_group,
                           cfg.is_tracker, 1 | (geo_bit if (tc_bwd or not need_grad) else 0), cfg.r2_scalar)   # bit 0: occupancy only (rgb belongs to the colour kernel)
        blob = pk.blob
        main = torch.cuda.current_stream(dev)
        side = _side_stream(dev) if OVERLAP_BRANCHES else None
        if side is not None:
            side.wait_stream(main)                       # fork: everything issued so far (kNN, packing) is visible to the side stream
        if use_h2:
            L.check(lib.psl_color_fwd_h2(C.byref(cfg), L.ptr(pk.hblob), L.ptr(pos), M, L.ptr(I), L.ptr(D), L.ptr(nn), L.ptr(r2),
                                         L.ptr(cloud_pos), L.ptr(col), L.ptr(rand_col), L.ptr(affine), L.ptr(raw), L.ptr(tsave),
                                         L.stream()), 'psl_color_fwd_h2')
        else:
            L.check(lib.psl_color_fwd_tc(C.byref(cfg), L.ptr(blob), L.ptr(pos), M, L.ptr(I), L.ptr(D), L.ptr(nn), L.ptr(r2),
                           L.ptr(cloud_pos), L.ptr(col), L.ptr(rand_col), L.ptr(affine), L.ptr(raw),
                           None if tc_bwd else L.ptr(save), L.ptr(tsave), L.stream()), 'psl_color_fwd_tc')
        with torch.cuda.stream(side) if side is not None else contextlib.nullcontext():
            L.check(lib.psl_decode_fwd(C.byref(gcfg), L.ptr(packed), L.ptr(pos), M, L.ptr(I), L.ptr(D), L.ptr(nn), L.ptr(r2),
                                       L.ptr(cloud_pos), L.ptr(geo), None, L.ptr(rand_geo), None, None, L.ptr(raw),
                                       L.ptr(has_nb), L.ptr(save), L.stream()), 'psl_decode_fwd[geometry]')
        if side is not None:
            main.wait_stream(side)                       # join
        return raw, has_nb, save, tsave, pstruct
    L.check(lib.psl_decode_fwd(C.byref(cfg), L.ptr(packed), L.ptr(pos), M, L.ptr(I), L.ptr(D), L.ptr(nn), L.ptr(r2),
                               L.ptr(cloud_pos), L.ptr(geo), L.ptr(col), L.ptr(rand_geo), L.ptr(rand_col),
                               L.ptr(affine), L.ptr(raw), L.ptr(has_nb), L.ptr(save), L.stream()), 'psl_decode_fwd')
    return raw, has_nb, save, None, pstruct


def _decode_backward(st: RenderSettings, cfg, params, needs, pos, I, D, nn, r2, cloud_pos, geo, col, affine, raw, save,
                     d_raw, want_pos, want_geo, want_col, want_affine, tsave=None, pack=None, repack=True, flat_out=None,
                     scatter_to=None):
    """-> (d_pos, d_geo, d_col, param grads list, d_affine)
    pack / repack: operand images to use and whether to rebuild them from `params`: True = forward and backward images,
    'bwd' = backward image only (the forward of the same parameters has just packed the rest), False = the caller packed;
    flat_out: caller-owned flat buffer for the requested parameter gradients (else allocated);
    scatter_to = (row_map i32 (N), n_rows, d_geo (n_rows,32) or None, d_col (n_rows,32) or None): feature gradients go to these
    PRE-ZEROED compact buffers (psl_feat_scatter_mapped) instead of fresh dense (N,32) tensors."""
    lib = L.load()
    dev = pos.device
    M = pos.shape[0]
    color = st.stage == 'color'
    rel = color and st.encode_rel_pos
    d_pos = torch.empty((M, 3), dtype=torch.float32, device=dev) if want_pos else None
    want_col = want_col and color
    d_cg = torch.empty((M, 32), dtype=torch.float32, device=dev) if want_geo else None
    wn = torch.empty((M, 8), dtype=torch.float32, device=dev) if (want_geo or want_col) else None
    d_colpair = None
    if want_col:
        d_colpair = torch.empty((M, 8, 32) if rel else (M, 32), dtype=torch.float32, device=dev)
    # one flat buffer for all requested parameter gradients (k_reduce_partials writes every element: no memset needed)
    want = [bool(n and (color or name.startswith('g_')) and name != 'c_B') for n, name in zip(needs, L_PARAM_NAMES)]
    sizes = [p.numel() if w else 0 for p, w in zip(params, want)]
    flat = None
    if any(want):
        flat = flat_out if flat_out is not None else torch.empty(sum(sizes), dtype=torch.float32, device=dev)
        assert flat.numel() == sum(sizes), 'flat_out does not match the requested parameter gradients'
    grads, off = [], 0
    for p, w, n_el in zip(params, want, sizes):
        grads.append(flat[off:off + n_el].view(p.shape) if w else None)
        off += n_el
    gstruct = _param_struct(grads)
    pstruct = _param_struct(params)
    d_aff = torch.zeros(12, dtype=torch.float32, device=dev) if want_affine else None
    ws_bytes = lib.psl_decode_bwd_ws_bytes(M)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    pk = pack if pack is not None else _default_pack(dev)
    packed = pk.packed
    if tsave is not None:
        # colour branch on tensor cores (data gradients), then geometry branch + IDW weights + d_pos on the FFMA kernel
        blob, bblob = pk.blob, pk.bblob
        if repack is True:
            _tc_fold_or_pack(lib, pstruct, blob)
        if repack:
            if USE_H2_BACKWARD:
                L.check(lib.psl_h2_bwd_pack_params(C.byref(pstruct), L.ptr(blob), L.ptr(pk.bhblob), L.stream()), 'psl_h2_bwd_pack_params')
            else:
                L.check(lib.psl_tc_bwd_pack_params(C.byref(pstruct), L.ptr(blob), lib.psl_tc_fold_offset_floats(), L.ptr(bblob), L.stream()),
                        'psl_tc_bwd_pack_params')
        tbwd = torch.empty(lib.psl_tc_bwd_tmp_floats(M, cfg.encode_rel_pos), dtype=torch.float32, device=dev)
        if wn is None:
            wn = torch.empty((M, 8), dtype=torch.float32, device=dev)
        dwn_col = torch.empty((M, 8), dtype=torch.float32, device=dev)
        dpos_col = torch.empty((M, 3), dtype=torch.float32, device=dev) if want_pos else None
        want_cparams = any(w and name.startswith('c_') for w, name in zip(want, L_PARAM_NAMES))
        grid_a = C.c_int32(0)
        gcfg = L.DecodeCfg(L.STAGE['geometry'], cfg.encode_rel_pos, L.RGB_SIGMOID, cfg.weighting, cfg.min_nn, cfg.r2_group,
                           cfg.is_tracker, cfg.reserved & 2, cfg.r2_scalar)
        assert not ((cfg.reserved & 2) and any(w and name.startswith('g_') for w, name in zip(want, L_PARAM_NAMES))), \
            'the forward kept only ReLU masks of the geometry branch (geo_param_grads=False) but a geometry parameter gradient is requested'

        def geometry_backward(dwn_extra, dpos_extra):
            L.check(lib.psl_decode_bwd(C.byref(gcfg), C.byref(pstruct), L.ptr(packed), L.ptr(pos), M, L.ptr(I), L.ptr(D),
                                       L.ptr(nn), L.ptr(r2), L.ptr(cloud_pos), L.ptr(geo), None, None, L.ptr(raw),
                                       L.ptr(save), L.ptr(d_raw), L.ptr(d_pos), L.ptr(d_cg), None, None,
                                       C.byref(gstruct), None, L.ptr(dwn_extra), L.ptr(dpos_extra), L.ptr(ws), ws_bytes, L.stream()),
                    'psl_decode_bwd[geometry]')

        # The geometry branch needs nothing from the colour branch except, for d_pos, the colour branch's gradient on the IDW weights
        # -- which enters linearly and is added afterwards (psl_idw_chain) -- so it runs on a forked stream and fills the SMs that
        # the colour kernel's partial last wave leaves idle.
        main = torch.cuda.current_stream(dev)
        side = _side_stream(dev) if OVERLAP_BRANCHES else None
        # everything the side stream will touch is allocated here, on the main stream (the caching allocator ties a block to the
        # stream that was current when it was allocated)
        scatter_args = None
        if want_geo or want_col:
            ws2_bytes = lib.psl_feat_scatter_ws_bytes(M)
            ws2 = torch.empty(ws2_bytes, dtype=torch.uint8, device=dev)
            if scatter_to is not None:
                row_map, n_rows, d_geo, d_col = scatter_to
                d_geo = d_geo if want_geo else None
                d_col = d_col if want_col else None
            else:
                row_map, n_rows = None, geo.shape[0]
                d_geo = torch.zeros_like(geo) if want_geo else None
                d_col = torch.zeros_like(col) if want_col else None
            scatter_args = (row_map, n_rows, d_geo, d_col, ws2, ws2_bytes)

        def scatter():
            row_map, n_rows, d_geo, d_col, ws2, ws2_bytes = scatter_args
            L.check(lib.psl_feat_scatter_mapped(L.ptr(I), M, L.ptr(row_map), n_rows, L.ptr(wn), L.ptr(d_cg),
                                                L.ptr(d_colpair) if rel else None, None if rel else L.ptr(d_colpair),
                                                L.ptr(d_geo), L.ptr(d_col), L.ptr(ws2), ws2_bytes, L.stream()), 'psl_feat_scatter')

        if side is not None:
            side.wait_stream(main)
        bwd_tc = lib.psl_color_bwd_h2 if USE_H2_BACKWARD else lib.psl_color_bwd_tc
        L.check(bwd_tc(C.byref(cfg), L.ptr(pk.bhblob if USE_H2_BACKWARD else bblob), L.ptr(pos), M, L.ptr(I), L.ptr(D), L.ptr(nn), L.ptr(r2),
                       L.ptr(cloud_pos), L.ptr(col), L.ptr(affine), L.ptr(raw), L.ptr(d_raw), L.ptr(tsave),
                       L.ptr(tbwd), L.ptr(d_colpair), L.ptr(wn), L.ptr(dwn_col), L.ptr(dpos_col),
                       int(want_cparams or want_affine), C.byref(grid_a), L.stream()), 'psl_color_bwd_tc')
        if side is not None:
            colour_done = torch.cuda.Event()
            colour_done.record(main)
            with torch.cuda.stream(side):
                geometry_backward(None, None)
                if scatter_args is not None:
                    # the deterministic feature-gradient scatter (radix sort of the (point, pair) keys + segmented sums) needs the
                    # colour kernel's per-pair gradients but nothing from the weight-gradient kernel: it runs beside it, in the issue
                    # slots that latency-bound kernel leaves idle
                    side.wait_event(colour_done)
                    scatter()
        if want_cparams or want_affine:
            wsf = lib.psl_wgrad_tc_ws_floats(M)
            wws = torch.empty(wsf, dtype=torch.float32, device=dev)
            L.check(lib.psl_wgrad_tc(C.byref(cfg), C.byref(pstruct), L.ptr(pos), M, L.ptr(I), L.ptr(cloud_pos), L.ptr(col),
                                     L.ptr(tsave), L.ptr(tbwd), grid_a.value, C.byref(gstruct), L.ptr(d_aff), L.ptr(wws), wsf,
                                     L.stream()), 'psl_wgrad_tc')
        if side is not None:
            main.wait_stream(side)
            if want_pos:
                # tracking: the geometry backward applied the IDW chain rule to its own share of d(weights) while the colour kernel
                # ran; the chain is linear, so the colour branch's share (and its direct d_pos) is added by one small pass
                L.check(lib.psl_idw_chain(C.byref(gcfg), L.ptr(pos), M, L.ptr(I), L.ptr(D), L.ptr(r2), L.ptr(cloud_pos), L.ptr(dwn_col),
                                          L.ptr(dpos_col), L.ptr(d_pos), L.stream()), 'psl_idw_chain')
        else:
            geometry_backward(dwn_col, dpos_col)
            if scatter_args is not None:
                scatter()
        d_geo, d_col = (scatter_args[2], scatter_args[3]) if scatter_args is not None else (None, None)
        return d_pos, d_geo, d_col, grads, d_aff
    L.check(lib.psl_decode_bwd(C.byref(cfg), C.byref(pstruct), L.ptr(packed), L.ptr(pos), M, L.ptr(I), L.ptr(D),
                               L.ptr(nn), L.ptr(r2), L.ptr(cloud_pos), L.ptr(geo), L.ptr(col), L.ptr(affine), L.ptr(raw),
                               L.ptr(save), L.ptr(d_raw), L.ptr(d_pos), L.ptr(d_cg), L.ptr(wn), L.ptr(d_colpair),
                               C.byref(gstruct), L.ptr(d_aff), None, None, L.ptr(ws), ws_bytes, L.stream()), 'psl_decode_bwd')
    d_geo = d_col = None
    if want_geo or want_col:
        ws2_bytes = lib.psl_feat_scatter_ws_bytes(M)
        ws2 = torch.empty(ws2_bytes, dtype=torch.uint8, device=dev)
        if scatter_to is not None:
            row_map, n_rows, d_geo, d_col = scatter_to
            d_geo = d_geo if want_geo else None
            d_col = d_col if want_col else None
        else:
            row_map, n_rows = None, geo.shape[0]
            d_geo = torch.zeros_like(geo) if want_geo else None
            d_col = torch.zeros_like(col) if want_col else None
        L.check(lib.psl_feat_scatter_mapped(L.ptr(I), M, L.ptr(row_map), n_rows, L.ptr(wn), L.ptr(d_cg),
                                            L.ptr(d_colpair) if rel else None, None if rel else L.ptr(d_colpair),
                                            L.ptr(d_geo), L.ptr(d_col), L.ptr(ws2), ws2_bytes, L.stream()), 'psl_feat_scatter')
    return d_pos, d_geo, d_col, grads, d_aff


L_PARAM_NAMES = PARAM_ORDER


class RenderSaved:
    """What render_backward needs from render_forward (plain attribute bag; the autograd node stores its tensors)."""
    FIELDS = ('z_vals', 'pos', 'I', 'D', 'nn', 'r2_ray', 'cloud', 'geo', 'col', 'aff', 'raw', 'has_nb', 'save', 'tsave')

    def __init__(self, st, cfg, tensors, params):
        self.st, self.cfg, self.params = st, cfg, params
        for k, v in zip(self.FIELDS, tensors):
            setattr(self, k, v)

    def tensors(self):
        return tuple(getattr(self, k) for k in self.FIELDS)


def warm_allocator(device, large_bytes=1 << 30, small_bytes=128 << 20):
    """Leave `large_bytes` (one block) and `small_bytes` (2 MB segments) of free memory in the caching allocator's pools.  The
    per-frame map update allocates tensors whose sizes change from frame to frame (#kept rays, #selected rows); whenever no cached
    block fits, the allocator calls cudaMalloc, which took 40-100 ms in a process holding the instantiated iteration graphs -- one
    frame step in twenty.  With the pools pre-filled those requests are served by splitting cached blocks.  Called by the
    iteration-graph classes after every capture (torch.cuda.graph empties the cache when a capture begins)."""
    if not WARM_ALLOCATOR:
        return
    big = torch.empty(int(large_bytes), dtype=torch.uint8, device=device)
    small = [torch.empty(1 << 19, dtype=torch.uint8, device=device) for _ in range(max(int(small_bytes) >> 19, 1))]
    del big, small


_TAIL_WS = {}


def _tail_ws(dev, nbytes):
    """Zero-initialised ticket + per-block partials of psl_render_tail (the kernel re-arms the ticket, so one buffer per device
    serves every launch on the stream; grown, never shrunk)."""
    w = _TAIL_WS.get(str(dev))
    if w is None or w.numel() < nbytes:
        w = _TAIL_WS[str(dev)] = torch.zeros(max(int(nbytes), 4096), dtype=torch.uint8, device=dev)
    return w


def render_forward(st: RenderSettings, grid: SpatialHash, params_c, ro, rd, gt_depth, z_override, r2_ray, rand_geo, rand_col,
                   cloud, geo, col, aff, need_grad, colour_param_grads=True, geo_param_grads=True, pack=None, prepacked=False,
                   tail=None, pack_backward=False):
    """Ray-march + kNN -> decode -> composite on contiguous fp32 device tensors, without autograd.
    -> depth (R,), var (R,), rgb (R,3), ray_mask (R,) uint8, RenderSaved (activations only when need_grad).
    tail = dict(mode 0 tracking / 1 mapping, depth_in (R,), inside (R,) u8, b_color (R,3) or None, w_color, loss_out ()): composite,
    ray mask, the iteration's loss and the composite backward run as ONE launch (psl_render_tail); the saved state then carries
    d_raw and render_backward(sv, None, None, None, ...) starts from it.
    pack_backward: also rebuild the tensor-core backward's operand image here (then render_backward(..., repack=False))."""
    lib = L.load()
    dev = ro.device
    R, S = ro.shape[0], st.S
    M = R * S
    z_vals = torch.empty((R, S), dtype=torch.float32, device=dev)
    pos = torch.empty((M, 3), dtype=torch.float32, device=dev)
    I = torch.empty((M, 8), dtype=torch.int32, device=dev)
    D = torch.empty((M, 8), dtype=torch.float32, device=dev)
    nn = torch.empty((M,), dtype=torch.int32, device=dev)
    r2s = float(np.float32(st.radius_query ** 2))
    if prepacked is not True and OVERLAP_BRANCHES:
        # the operand images depend on the parameters only, the ray march + kNN on the rays and the cloud only: the (serial, latency-
        # bound) packing kernels run on the forked stream while the kNN kernel runs, instead of between it and the decode
        pk = pack if pack is not None else _default_pack(dev)
        main, side = torch.cuda.current_stream(dev), _side_stream(dev)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            _pack_images(st, params_c, pk, prepacked, need_grad, colour_param_grads, backward=pack_backward)
        packed_early = True
    else:
        packed_early = False
    L.check(lib.psl_raymarch_knn(C.byref(grid.struct), L.ptr(ro), L.ptr(rd), L.ptr(gt_depth), R, S,
                                 L.ptr(surface_t_vals(S, dev)), st.near_surface, st.far_surface, L.ptr(z_override),
                                 L.ptr(r2_ray), r2s, L.ptr(z_vals), L.ptr(pos), L.ptr(I), L.ptr(D), L.ptr(nn),
                                 L.stream()), 'psl_raymarch_knn')
    cfg = st.cfg(S, r2s)
    if packed_early:
        main.wait_stream(side)
        prepacked = True
    elif pack_backward:
        _pack_images(st, params_c, pack if pack is not None else _default_pack(dev), prepacked, need_grad, colour_param_grads, backward=True)
        prepacked = True
    raw, has_nb, save, tsave, _ = _decode_forward(st, cfg, params_c, pos, I, D, nn, r2_ray, cloud, geo, col, rand_geo,
                                                  rand_col, aff, need_grad, colour_param_grads=colour_param_grads,
                                                  geo_param_grads=geo_param_grads, pack=pack, prepacked=prepacked)
    depth = torch.empty((R,), dtype=torch.float32, device=dev)
    var = torch.empty((R,), dtype=torch.float32, device=dev)
    rgb = torch.empty((R, 3), dtype=torch.float32, device=dev)
    ray_mask = torch.empty((R,), dtype=torch.uint8, device=dev)
    d_raw = None
    if tail is not None:
        d_raw = torch.empty((M, 4), dtype=torch.float32, device=dev)
        ws = _tail_ws(dev, lib.psl_render_tail_ws_bytes(R))
        L.check(lib.psl_render_tail(int(tail['mode']), R, S, st.coef, int(S / 2 + 1), L.ptr(raw), L.ptr(has_nb), L.ptr(z_vals),
                                    L.ptr(tail['depth_in']), L.ptr(tail['inside']), L.ptr(tail.get('b_color')), float(tail['w_color']),
                                    L.ptr(depth), L.ptr(var), L.ptr(rgb), L.ptr(ray_mask), L.ptr(tail['loss_out']), L.ptr(d_raw),
                                    L.ptr(ws), ws.numel(), L.stream()), 'psl_render_tail')
    else:
        L.check(lib.psl_composite_fwd(L.ptr(raw), L.ptr(has_nb), L.ptr(z_vals), R, S, st.coef, L.ptr(depth), L.ptr(var),
                                      L.ptr(rgb), None, L.stream()), 'psl_composite_fwd')
        L.check(lib.psl_ray_mask(L.ptr(has_nb), R, S, int(S / 2 + 1), L.ptr(ray_mask), L.stream()), 'psl_ray_mask')
    saved = RenderSaved(st, cfg, (z_vals, pos, I, D, nn, r2_ray, cloud, geo, col, aff, raw, has_nb, save, tsave), params_c)
    saved.d_raw = d_raw
    return depth, var, rgb, ray_mask, saved


def render_backward(sv: RenderSaved, d_depth, d_var, d_rgb, want_o, want_d, want_geo, want_col, want_aff, needs,
                    pack=None, repack=True, flat_out=None, scatter_to=None):
    """Backward of render_forward.  d_* : contiguous fp32 gradients of depth / var / rgb (None = zero);
    needs: per-parameter flags in PARAM_ORDER.  -> d_rays_o, d_rays_d, d_geo, d_col, d_affine, [param grads]"""
    lib = L.load()
    st = sv.st
    R, S = sv.z_vals.shape
    dev = sv.z_vals.device
    d_raw = getattr(sv, 'd_raw', None)          # already produced by the fused render tail (render_forward(tail=...))
    if d_raw is None:
        d_raw = torch.empty((R * S, 4), dtype=torch.float32, device=dev)
        L.check(lib.psl_composite_bwd(L.ptr(sv.raw), L.ptr(sv.has_nb), L.ptr(sv.z_vals), R, S, st.coef, L.ptr(d_depth), L.ptr(d_var),
                                      L.ptr(d_rgb), L.ptr(d_raw), L.stream()), 'psl_composite_bwd')
    else:
        assert d_depth is None and d_var is None and d_rgb is None, 'the fused render tail already applied the loss gradients'
    want_pos = want_o or want_d
    d_pos, d_geo, d_col, grads, d_aff = _decode_backward(st, sv.cfg, sv.params, needs, sv.pos, sv.I, sv.D, sv.nn, sv.r2_ray,
                                                         sv.cloud, sv.geo, sv.col, sv.aff, sv.raw, sv.save, d_raw, want_pos,
                                                         want_geo, want_col, want_aff, tsave=sv.tsave, pack=pack, repack=repack,
                                                         flat_out=flat_out, scatter_to=scatter_to)
    d_o = d_d = None
    if want_pos:
        d_o = torch.empty((R, 3), dtype=torch.float32, device=dev) if want_o else None
        d_d = torch.empty((R, 3), dtype=torch.float32, device=dev) if want_d else None
        L.check(lib.psl_rays_bwd(L.ptr(d_pos), L.ptr(sv.z_vals), R, S, L.ptr(d_o), L.ptr(d_d), L.stream()), 'psl_rays_bwd')
    return d_o, d_d, d_geo, d_col, (d_aff if want_aff else None), grads


class _RenderFn(torch.autograd.Function):
    """render_batch_ray core: ray-march + kNN -> decode -> composite, one autograd node."""

    @staticmethod
    def forward(ctx, st: RenderSettings, grid: SpatialHash, gt_depth, z_override, r2_ray, rand_geo, rand_col,
                cloud_pos, rays_o, rays_d, geo_feats, col_feats, affine, *params):
        ro, rd = _f32c(rays_o), _f32c(rays_d)
        geo = _f32c(geo_feats)
        col = _f32c(col_feats) if col_feats is not None else None
        cloud = _f32c(cloud_pos)
        params_c = [_f32c(p) for p in params]
        aff = _f32c(affine).reshape(-1) if affine is not None else None
        nig = ctx.needs_input_grad
        need_grad = st.grad_mode and any(nig)     # grad mode is sampled by the caller: it is off inside forward()
        cpg = any(n and name.startswith('c_') for n, name in zip(nig[13:], L_PARAM_NAMES)) or bool(nig[12])
        gpg = any(n and name.startswith('g_') for n, name in zip(nig[13:], L_PARAM_NAMES))
        depth, var, rgb, ray_mask, sv = render_forward(st, grid, params_c, ro, rd, gt_depth, z_override, r2_ray, rand_geo,
                                                       rand_col, cloud, geo, col, aff, need_grad, colour_param_grads=cpg,
                                                       geo_param_grads=gpg)
        ctx.st, ctx.cfg = st, sv.cfg
        ctx.save_for_backward(*sv.tensors(), *params_c)
        ctx.mark_non_differentiable(ray_mask)
        return depth, var, rgb, ray_mask.bool()

    @staticmethod
    def backward(ctx, d_depth, d_var, d_rgb, _d_mask):
        n = len(RenderSaved.FIELDS)
        sv = RenderSaved(ctx.st, ctx.cfg, ctx.saved_tensors[:n], list(ctx.saved_tensors[n:]))
        dd = _f32c(d_depth) if d_depth is not None else None
        dv = _f32c(d_var) if d_var is not None else None
        dc = _f32c(d_rgb) if d_rgb is not None else None
        nig = ctx.needs_input_grad            # (st, grid, gt_depth, z_override, r2, rand_geo, rand_col, cloud, o, d, geo, col, affine, *params)
        d_o, d_d, d_geo, d_col, d_aff, grads = render_backward(sv, dd, dv, dc, nig[8], nig[9], nig[10], nig[11], nig[12],
                                                               list(nig[13:]))
        return (None, None, None, None, None, None, None, None, d_o, d_d, d_geo, d_col, d_aff, *grads)


class _DecodeFn(torch.autograd.Function):
    """POINT.forward core (decoder.py:476-518) on explicit sample positions."""

    @staticmethod
    def forward(ctx, st: RenderSettings, grid: SpatialHash, r2_pts, r2_group, rand_geo, rand_col, cloud_pos,
                p, geo_feats, col_feats, affine, *params):
        dev = p.device
        pos = _f32c(p).reshape(-1, 3)
        geo = _f32c(geo_feats)
        col = _f32c(col_feats) if col_feats is not None else None
        cloud = _f32c(cloud_pos)
        params_c = [_f32c(q) for q in params]
        aff = _f32c(affine).reshape(-1) if affine is not None else None
        D, I, nn = knn_query_r2(grid, pos, r2_pts, st.radius_query, r2_group)
        r2s = float(np.float32(st.radius_query ** 2))
        cfg = st.cfg(r2_group, r2s)
        need_grad = st.grad_mode and any(ctx.needs_input_grad)     # grad mode is sampled by the caller: it is off inside forward()
        nig = ctx.needs_input_grad
        cpg = any(n and name.startswith('c_') for n, name in zip(nig[11:], L_PARAM_NAMES)) or bool(nig[10])
        gpg = any(n and name.startswith('g_') for n, name in zip(nig[11:], L_PARAM_NAMES))
        raw, has_nb, save, tsave, _ = _decode_forward(st, cfg, params_c, pos, I, D, nn, r2_pts, cloud, geo, col, rand_geo,
                                                      rand_col, aff, need_grad, colour_param_grads=cpg, geo_param_grads=gpg)
        ctx.st, ctx.cfg = st, cfg
        ctx.save_for_backward(pos, I, D, nn, r2_pts, cloud, geo, col, aff, raw, save, tsave, *params_c)
        hb = has_nb.bool()
        ctx.mark_non_differentiable(hb)
        return raw, hb

    @staticmethod
    def backward(ctx, d_raw, _d_mask):
        st, cfg = ctx.st, ctx.cfg
        pos, I, D, nn, r2, cloud, geo, col, aff, raw, save, tsave = ctx.saved_tensors[:12]
        params = list(ctx.saved_tensors[12:])
        nig = ctx.needs_input_grad            # (st, grid, r2, r2_group, rand_geo, rand_col, cloud, p, geo, col, affine, *params)
        d_pos, d_geo, d_col, grads, d_aff = _decode_backward(st, cfg, params, list(nig[11:]), pos, I, D, nn, r2, cloud,
                                                             geo, col, aff, raw, save, _f32c(d_raw), nig[7], nig[8],
                                                             nig[9], nig[10], tsave=tsave)
        return (None, None, None, None, None, None, None, d_pos, d_geo, d_col, d_aff if nig[10] else None, *grads)


def knn_query_r2(grid, pos, r2, radius, group):
    """kNN with an already squared float64 radius tensor (or None -> scalar radius)."""
    lib = L.load()
    M = pos.shape[0]
    dev = pos.device
    I = torch.empty((M, 8), dtype=torch.int32, device=dev)
    D = torch.empty((M, 8), dtype=torch.float32, device=dev)
    nn = torch.empty((M,), dtype=torch.int32, device=dev)
    if M:
        L.check(lib.psl_knn_query(C.byref(grid.struct), L.ptr(pos), M, L.ptr(r2), float(np.float32(radius ** 2)),
                                  int(group), L.ptr(I), L.ptr(D), L.ptr(nn), L.stream()), 'psl_knn_query')
    return D, I, nn


class _CompositeFn(torch.autograd.Function):
    """raw2outputs_nerf_color (common.py:298-336); `has_nb` carries the Renderer.py:189-190 masking."""

    @staticmethod
    def forward(ctx, raw, z_vals, has_nb, coef):
        lib = L.load()
        R, S = z_vals.shape
        dev = raw.device
        rawc, zc = _f32c(raw).reshape(R * S, 4), _f32c(z_vals)
        hb = has_nb.to(torch.uint8).contiguous() if has_nb is not None else torch.ones(R * S, dtype=torch.uint8, device=dev)
        depth = torch.empty((R,), dtype=torch.float32, device=dev)
        var = torch.empty((R,), dtype=torch.float32, device=dev)
        rgb = torch.empty((R, 3), dtype=torch.float32, device=dev)
        w = torch.empty((R, S), dtype=torch.float32, device=dev)
        L.check(lib.psl_composite_fwd(L.ptr(rawc), L.ptr(hb), L.ptr(zc), R, S, float(coef), L.ptr(depth), L.ptr(var),
                                      L.ptr(rgb), L.ptr(w), L.stream()), 'psl_composite_fwd')
        ctx.save_for_backward(rawc, zc, hb)
        ctx.coef = float(coef)
        ctx.mark_non_differentiable(w)
        return depth, var, rgb, w

    @staticmethod
    def backward(ctx, d_depth, d_var, d_rgb, _dw):
        lib = L.load()
        rawc, zc, hb = ctx.saved_tensors
        R, S = zc.shape
        d_raw = torch.empty_like(rawc)
        L.check(lib.psl_composite_bwd(L.ptr(rawc), L.ptr(hb), L.ptr(zc), R, S, ctx.coef,
                                      L.ptr(_f32c(d_depth)) if d_depth is not None else None,
                                      L.ptr(_f32c(d_var)) if d_var is not None else None,
                                      L.ptr(_f32c(d_rgb)) if d_rgb is not None else None, L.ptr(d_raw), L.stream()),
                'psl_composite_bwd')
        return d_raw.reshape(R, S, 4), None, None, None


def render(st: RenderSettings, grid: SpatialHash, params: Sequence[torch.Tensor], rays_o, rays_d, gt_depth,
           cloud_pos, geo_feats, col_feats, r2_ray=None, z_override=None, rand_geo=None, rand_col=None, affine=None):
    """Fused render_batch_ray core.  -> depth (R,), var (R,), rgb (R,3), ray_mask (R,) bool."""
    dev = rays_o.device
    if rand_geo is None:
        rand_geo = torch.zeros(32, device=dev)
    if rand_col is None:
        rand_col = torch.zeros(32, device=dev)
    st.grad_mode = torch.is_grad_enabled()
    return _RenderFn.apply(st, grid, _f32c(gt_depth).reshape(-1), z_override, r2_ray, _f32c(rand_geo), _f32c(rand_col),
                           cloud_pos, rays_o, rays_d, geo_feats, col_feats, affine, *params)


def decode(st: RenderSettings, grid: SpatialHash, params, p, cloud_pos, geo_feats, col_feats, r2_pts=None, r2_group=1,
           rand_geo=None, rand_col=None, affine=None):
    dev = p.device
    if rand_geo is None:
        rand_geo = torch.zeros(32, device=dev)
    if rand_col is None:
        rand_col = torch.zeros(32, device=dev)
    st.grad_mode = torch.is_grad_enabled()
    return _DecodeFn.apply(st, grid, r2_pts, int(r2_group), _f32c(rand_geo), _f32c(rand_col), cloud_pos, p, geo_feats,
                           col_feats, affine, *params)


def composite(raw, z_vals, has_nb=None, coef=0.1):
    return _CompositeFn.apply(raw, z_vals, has_nb, coef)


# ------------------------------------------------------------------------------------------------------------------
# map maintenance between renders (SURVEY.md section 8f rank 1)
# ------------------------------------------------------------------------------------------------------------------
_STEPS = {}


def _add_steps(n_add: int, fixed_interval: bool, device) -> torch.Tensor:
    """linspace(0,1,N_add) / linspace(-0.04,0.04,N_add) of neural_point.py:126-131, evaluated by torch on the CPU."""
    key = (int(n_add), bool(fixed_interval), str(device))
    if key not in _STEPS:
        lo, hi = (-0.04, 0.04) if fixed_interval else (0.0, 1.0)
        _STEPS[key] = torch.linspace(lo, hi, steps=int(n_add), dtype=torch.float32).to(device)
    return _STEPS[key]


def add_points(grid: SpatialHash, rays_o, rays_d, gt_depth, gt_color, new_pos: torch.Tensor, radius: float,
               dynamic_radius=None, n_add: int = 3, fixed_interval: bool = False, near_surface: float = 0.98,
               far_surface: float = 1.02):
    """add_neural_points geometry (neural_point.py:107-145) in one library call, no host synchronisation:
    writes the kept rays' N_add points, compacted in ray order, into `new_pos` (room for n*n_add points) and returns
    (counts (2,) int32 device = [#depth>0 rays, #kept rays], input_pos (n,3), input_rgb (n,3)) -- the first counts[1] rows
    of the two (n,3) tensors are valid.  `dynamic_radius` has one entry per depth > 0 ray, like the reference's call."""
    lib = L.load()
    ro, rd, dep = _f32c(rays_o).reshape(-1, 3), _f32c(rays_d).reshape(-1, 3), _f32c(gt_depth).reshape(-1)
    n = dep.shape[0]
    dev = ro.device
    col = _f32c(gt_color).reshape(-1, 3) if gt_color is not None else None
    assert new_pos.is_contiguous() and new_pos.dtype == torch.float32 and new_pos.numel() >= n * n_add * 3
    counts = torch.zeros(2, dtype=torch.int32, device=dev)
    in_pos = torch.empty((n, 3), dtype=torch.float32, device=dev)
    in_rgb = torch.empty((n, 3), dtype=torch.float32, device=dev)
    if n == 0:
        return counts, in_pos, in_rgb
    r2 = None
    r2s = float(np.float32(radius ** 2))
    if dynamic_radius is not None:
        assert dynamic_radius.numel() <= n, 'shape mis-match for input points and dynamic radius'
        r2 = (dynamic_radius.detach().reshape(-1).to(device=dev) ** 2).to(torch.float64)
        if r2.shape[0] < n:                # length is checked against #(depth > 0) by the caller once the counts are known
            r2 = torch.cat([r2, torch.zeros(n - r2.shape[0], dtype=torch.float64, device=dev)])
        r2 = r2.contiguous()
    ws_bytes = lib.psl_add_points_ws_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    steps = _add_steps(n_add, fixed_interval, dev)
    L.check(lib.psl_add_points(C.byref(grid.struct), L.ptr(ro), L.ptr(rd), L.ptr(dep), L.ptr(col), n, L.ptr(r2), r2s,
                               int(n_add), int(bool(fixed_interval)), float(near_surface), float(far_surface), L.ptr(steps),
                               L.ptr(new_pos), L.ptr(in_pos), L.ptr(in_rgb), L.ptr(counts), L.ptr(ws), ws_bytes, L.stream()),
            'psl_add_points')
    return counts, in_pos, in_rgb


_FRUSTUM_SCRATCH = {}


def frustum_select(cloud_pos: torch.Tensor, c2w, depth: torch.Tensor, H, W, fx, fy, cx, cy, edge: int = -4,
                   return_mask: bool = False, reuse: bool = False):
    """Mapper.get_mask_from_c2w (Mapper.py:120-168) on the device: -> ascending int64 indices of the selected points
    (a device tensor where the reference returns a Python list; both index the feature tensors the same way).
    `c2w`: (4,4) or (3,4) pose (tensor / array); it is inverted on the host in float32 like the reference does.
    reuse=True: outputs and workspace live in a per-device scratch that is kept between calls (the per-frame callers: no allocator
    traffic between two host syncs of the map update -- an occasional 40 ms stall of one of these allocations was the one outlier
    step of the bench); the returned index tensor is then a VIEW that the next reuse=True call on the device overwrites."""
    lib = L.load()
    pos = _f32c(cloud_pos).reshape(-1, 3)
    n = pos.shape[0]
    dev = pos.device
    c = c2w.detach().cpu().numpy() if torch.is_tensor(c2w) else np.asarray(c2w)
    c = c.astype(np.float32)
    if c.shape[0] == 3:
        c = np.concatenate([c, np.array([[0, 0, 0, 1]], np.float32)], 0)
    w2c = np.linalg.inv(c).astype(np.float64)
    w = (C.c_double * 12)(*w2c[:3].reshape(-1).tolist())
    depth = depth if torch.is_tensor(depth) else torch.from_numpy(np.ascontiguousarray(depth))
    depth = depth.to(device=dev, dtype=torch.float32).contiguous()
    assert depth.shape == (H, W)
    ws_bytes = lib.psl_frustum_select_ws_bytes(n) if n else 0
    if reuse:
        sc = _FRUSTUM_SCRATCH.get(str(dev))
        if sc is None or sc['cap'] < n or sc['ws'].numel() < ws_bytes:
            cap = max(int(n * 1.5), 1024)
            sc = _FRUSTUM_SCRATCH[str(dev)] = dict(
                cap=cap, mask=torch.empty(cap, dtype=torch.uint8, device=dev), idx=torch.empty(cap, dtype=torch.int64, device=dev),
                count=torch.zeros(1, dtype=torch.int32, device=dev),
                ws=torch.empty(max(lib.psl_frustum_select_ws_bytes(cap), 256), dtype=torch.uint8, device=dev))
        mask, idx, count, ws = sc['mask'][:n], sc['idx'][:n], sc['count'], sc['ws']
        count.zero_()
    else:
        mask = torch.empty(n, dtype=torch.uint8, device=dev)
        idx = torch.empty(n, dtype=torch.int64, device=dev)
        count = torch.zeros(1, dtype=torch.int32, device=dev)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    if n:
        L.check(lib.psl_frustum_select(L.ptr(pos), n, w, float(fx), float(fy), float(cx), float(cy), L.ptr(depth), int(H), int(W),
                                       int(edge), L.ptr(mask), L.ptr(idx), L.ptr(count), L.ptr(ws), ws.numel(), L.stream()),
                'psl_frustum_select')
    k = int(count.item())                  # the one synchronisation: the caller sizes its optimisable slices with it
    return (idx[:k], mask.bool()) if return_mask else idx[:k]


# ------------------------------------------------------------------------------------------------------------------
# per-frame colour gradient: dynamic-radius maps and gradient-based pixel selection (csrc/psl_frame.cu)
# ------------------------------------------------------------------------------------------------------------------
GRAD_RATIO = 15              # get_selected_index_with_grad(ratio=15), common.py:92 (DESIGN.md section 1, stated assumptions)


def frame_grad(color: torch.Tensor, cfg, maps: bool = True, mag_out: Optional[torch.Tensor] = None):
    """The dynamic-radius maps of Tracker.py:237-248 / Mapper.py:686-704 and the gradient magnitude they come from, on the device:
    -> (r_add, r_query, mag), float64 (H,W) each, equal to synth.sobel_radius_map(color, ...) for the maps.  `cfg`: the
    configuration (its `pointcloud` section: radius_add_max, radius_add_min, radius_query_ratio, color_grad_threshold).
    maps=False computes mag only (r_add, r_query are None); mag_out: a float64 (H,W) tensor to write mag into."""
    lib = L.load()
    pc = cfg['pointcloud'] if 'pointcloud' in cfg else cfg
    col = _f32c(color)
    H, W = int(col.shape[0]), int(col.shape[1])
    assert col.shape == (H, W, 3), 'color must be (H,W,3)'
    kw = dict(dtype=torch.float64, device=col.device)
    mag = mag_out if mag_out is not None else torch.empty(H, W, **kw)
    assert mag.shape == (H, W) and mag.dtype == torch.float64
    r_add = torch.empty(H, W, **kw) if maps else None
    r_query = torch.empty(H, W, **kw) if maps else None
    L.check(lib.psl_frame_grad(L.ptr(col), H, W, float(pc['radius_add_max']), float(pc['radius_add_min']),
                               float(pc['radius_query_ratio']), float(pc['color_grad_threshold']), L.ptr(mag), L.ptr(r_add),
                               L.ptr(r_query), L.stream()), 'psl_frame_grad')
    return r_add, r_query, mag


def grad_capacity(n: int, H: int, W: int, ratio: int = GRAD_RATIO) -> int:
    """Length of the candidate list of get_selected_index_with_grad for n samples: ratio * n, at most the image."""
    return min(int(ratio) * int(n), int(H) * int(W))


def grad_candidates(mag: torch.Tensor, depth: torch.Tensor, n: int, ratio: int = GRAD_RATIO, window=None, depth_max=None,
                    cand: Optional[torch.Tensor] = None, count: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None):
    """get_selected_index_with_grad (common.py:92-159) on the device, no host synchronisation: of the ratio * n pixels of
    largest `mag` over the whole image (ties: smaller flat index first), the ones inside window = (H0, H1, W0, W1) (default: the
    whole image) with 0 < depth <= depth_max (None: no upper bound).  -> (cand, count): cand (grad_capacity) int64, its first
    count[0] entries the ascending flat indices row * W + column; count (1,) int32 on the device.  cand / count / ws may be
    passed in (fixed buffers of a captured caller)."""
    lib = L.load()
    H, W = int(mag.shape[0]), int(mag.shape[1])
    dev = mag.device
    assert mag.dtype == torch.float64 and mag.is_contiguous()
    dep = _f32c(depth)
    assert dep.shape == (H, W)
    H0, H1, W0, W1 = window if window is not None else (0, H, 0, W)
    k = grad_capacity(n, H, W, ratio)
    cand = cand if cand is not None else torch.empty(k, dtype=torch.int64, device=dev)
    count = count if count is not None else torch.empty(1, dtype=torch.int32, device=dev)
    assert cand.numel() >= k and cand.dtype == torch.int64 and count.dtype == torch.int32
    ws_bytes = lib.psl_grad_candidates_ws_bytes(H * W)
    ws = ws if ws is not None else torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    assert ws.numel() >= ws_bytes
    dmax = float('inf') if depth_max is None else float(depth_max)
    L.check(lib.psl_grad_candidates(L.ptr(mag), L.ptr(dep), H, W, int(H0), int(H1), int(W0), int(W1), dmax, k, L.ptr(cand),
                                    L.ptr(count), L.ptr(ws), ws.numel(), L.stream()), 'psl_grad_candidates')
    return cand, count


def pick_candidates(cand: torch.Tensor, count: torch.Tensor, n: int, W: int, window=None, generator=None,
                    pix: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None):
    """n distinct candidates out of cand[:count] drawn uniformly without replacement (random_select / np.random.choice with
    replace=False after get_selected_index_with_grad), as the window-relative flat indices psl_sample_rays takes:
    (row - H0) * (W1 - W0) + column - W0 for window = (H0, H1, W0, W1) (default: the whole image of width W).  Slots beyond
    count[0] are -1.  Static shapes and no host synchronisation: safe inside a CUDA-graph capture (the keys come from
    torch.randint on `generator`, default: the device's default generator)."""
    lib = L.load()
    cap = int(cand.numel())
    dev = cand.device
    assert 1 <= n <= cap, 'need 1 <= n <= the candidate capacity'
    H0, _, W0, W1 = window if window is not None else (0, None, 0, W)
    keys = torch.randint(2 ** 31 - 1, (cap,), dtype=torch.int32, device=dev, generator=generator)
    pix = pix if pix is not None else torch.empty(n, dtype=torch.int64, device=dev)
    assert pix.numel() == n and pix.dtype == torch.int64
    ws_bytes = lib.psl_pick_candidates_ws_bytes(cap)
    ws = ws if ws is not None else torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    assert ws.numel() >= ws_bytes
    L.check(lib.psl_pick_candidates(L.ptr(cand), L.ptr(count), cap, L.ptr(keys), int(n), int(W), int(H0), int(W0), int(W1 - W0),
                                    L.ptr(pix), L.ptr(ws), ws.numel(), L.stream()), 'psl_pick_candidates')
    return pix
