"""ctypes binding of libpointslam_b200.so (the C ABI declared in include/pointslam_b200.h).

The shared library is built in-tree by `build()` (called from `__graft_entry__.build()`); there is NO
fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
# PSL_LIB: load another build of the same sources (A/B experiments, e.g. one compiled with -DPSL_PRECISE_TRIG)
LIB_PATH = os.environ.get('PSL_LIB') or os.path.join(_HERE, 'libpointslam_b200.so')
SOURCES = ['psl_api.cu', 'psl_grid.cu', 'psl_decode_fwd.cu', 'psl_decode_bwd.cu', 'psl_geo_mma.cu', 'psl_composite.cu', 'psl_color_tc.cu', 'psl_color_tc_w16.cu', 'psl_color_h2.cu', 'psl_color_bwd_h2.cu', 'psl_color_bwd_tc.cu', 'psl_color_bwd_tc_w16.cu', 'psl_wgrad_tc.cu', 'psl_shell.cu', 'psl_map.cu', 'psl_frame.cu']
HEADERS = ['psl_common.cuh', 'psl_decode.cuh', 'psl_grid.cuh', 'psl_tc.cuh', 'psl_tc_layout.cuh', 'psl_color_tc.cuh', 'psl_color_bwd_tc.cuh', 'psl_composite.cuh']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC', '--threads', '4']

_vp, _i32, _i64, _f32, _f64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_size_t


class Grid(C.Structure):                                   # psl_grid
    _fields_ = [('sorted_pts', _vp), ('table_keys', _vp), ('table_vals', _vp), ('capacity', C.c_uint32),
                ('n', _i32), ('cell', _f32), ('r_small', _f32), ('meta', _vp)]


N_PARAMS = 1 + 5 * 4 + 2 + 6 + 5 * 4 + 2                   # 51 pointers in psl_decoder_params


class DecoderParams(C.Structure):                          # psl_decoder_params / psl_decoder_grads (same layout)
    _fields_ = [('g_B', _vp), ('g_W', _vp * 5), ('g_b', _vp * 5), ('g_Wc', _vp * 5), ('g_bc', _vp * 5),
                ('g_Wo', _vp), ('g_bo', _vp), ('c_B', _vp), ('c_Brel', _vp), ('c_N1', _vp), ('c_n1b', _vp),
                ('c_N2', _vp), ('c_n2b', _vp), ('c_W', _vp * 5), ('c_b', _vp * 5), ('c_Wc', _vp * 5),
                ('c_bc', _vp * 5), ('c_Wo', _vp), ('c_bo', _vp)]


class DecodeCfg(C.Structure):                              # psl_decode_cfg
    _fields_ = [('stage', _i32), ('encode_rel_pos', _i32), ('rgb_mode', _i32), ('weighting', _i32),
                ('min_nn', _i32), ('r2_group', _i32), ('is_tracker', _i32), ('reserved', _i32), ('r2_scalar', _f64)]


STAGE = {'geometry': 0, 'color': 1}
RGB_SIGMOID, RGB_AFFINE_SIGMOID, RGB_RAW = 0, 1, 2
WEIGHTING = {'distance': 0, 'expo': 1}

_SIGS = {
    'psl_version': (C.c_int, []),
    'psl_last_error': (C.c_char_p, []),
    'psl_device_sm_count': (C.c_int, []),
    'psl_launch_count': (C.c_uint64, []),
    'psl_timing_enable': (C.c_int, [C.c_int]),
    'psl_timing_collect': (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    'psl_grid_sort_ws_bytes': (_sz, [_i64]),
    'psl_grid_sort': (C.c_int, [_vp, _i64, _f32, _vp, _vp, _vp, _sz, C.POINTER(_i64), _vp]),
    'psl_grid_append_ws_bytes': (_sz, [_i64, _i64]),
    'psl_grid_append': (C.c_int, [_vp, _i64, _i64, _f32, _vp, _vp, _vp, _sz, C.POINTER(_i64), _vp]),
    'psl_grid_hash': (C.c_int, [_vp, _i64, _vp, _vp, C.c_uint32, _vp]),
    'psl_knn_query': (C.c_int, [C.POINTER(Grid), _vp, _i64, _vp, _f64, _i32, _vp, _vp, _vp, _vp]),
    'psl_raymarch_knn': (C.c_int, [C.POINTER(Grid), _vp, _vp, _vp, _i64, _i32, _vp, _f32, _f32, _vp, _vp, _f64,
                                   _vp, _vp, _vp, _vp, _vp, _vp]),
    'psl_raymarch_knn_stats': (C.c_int, [C.POINTER(Grid), _vp, _vp, _vp, _i64, _i32, _vp, _f32, _f32, _vp, _vp, _f64,
                                         _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'psl_packed_params_floats': (_sz, []),
    'psl_decode_save_floats_per_sample': (_sz, [C.POINTER(DecodeCfg)]),
    'psl_decode_bwd_ws_bytes': (_sz, [_i64]),
    'psl_pack_params': (C.c_int, [C.POINTER(DecoderParams), _vp, _vp]),
    'psl_decode_fwd': (C.c_int, [C.POINTER(DecodeCfg), _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _vp, _vp, _vp, _vp]),
    'psl_decode_bwd': (C.c_int, [C.POINTER(DecodeCfg), C.POINTER(DecoderParams), _vp, _vp, _i64, _vp, _vp, _vp, _vp,
                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(DecoderParams), _vp,
                                 _vp, _vp, _vp, _sz, _vp]),
    'psl_feat_scatter_ws_bytes': (_sz, [_i64]),
    'psl_feat_scatter': (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'psl_feat_scatter_mapped': (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'psl_sample_rays': (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32,
                                  _vp, _vp, _vp, _vp, _vp, _vp]),
    'psl_depth_gate': (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    'psl_shell_loss': (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp]),
    'psl_idw_chain': (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'psl_render_tail_ws_bytes': (_sz, [_i32]),
    'psl_render_tail': (C.c_int, [_i32, _i32, _i32, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'psl_pose_bwd': (C.c_int, [_vp, _i32, _i32, _i32, _i32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    'psl_adam_rows': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _f32, _f32, _f32, _f32, _i32, _vp]),
    'psl_pose_adam': (C.c_int, [_vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _i32, _vp]),
    'psl_composite_fwd': (C.c_int, [_vp, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _vp]),
    'psl_composite_bwd': (C.c_int, [_vp, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _vp]),
    'psl_rays_bwd': (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    'psl_ray_mask': (C.c_int, [_vp, _i64, _i32, _i32, _vp, _vp]),
    'psl_tc_blob_floats': (_sz, []),
    'psl_tc_pack_params': (C.c_int, [C.POINTER(DecoderParams), _vp, _vp]),
    'psl_tc_fold_params': (C.c_int, [C.POINTER(DecoderParams), _vp, _vp]),
    'psl_color_fwd_tc': (C.c_int, [C.POINTER(DecodeCfg), _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'psl_h2_blob_bytes': (_sz, []),
    'psl_h2_pack_params': (C.c_int, [C.POINTER(DecoderParams), _vp, _vp, _vp]),
    'psl_color_fwd_h2': (C.c_int, [C.POINTER(DecodeCfg), _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'psl_h2_bwd_blob_bytes': (_sz, []),
    'psl_h2_bwd_pack_params': (C.c_int, [C.POINTER(DecoderParams), _vp, _vp, _vp]),
    'psl_color_bwd_h2': (C.c_int, [C.POINTER(DecodeCfg), _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _vp, _vp, _i32, C.POINTER(_i32), _vp]),
    'psl_wgrad_tc_ws_floats': (_sz, [_i64]),
    'psl_wgrad_tc': (C.c_int, [C.POINTER(DecodeCfg), C.POINTER(DecoderParams), _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32,
                               C.POINTER(DecoderParams), _vp, _vp, _sz, _vp]),
    'psl_tc_fold_offset_floats': (_sz, []),
    'psl_tc_bwd_blob_floats': (_sz, []),
    'psl_tc_save_floats': (_sz, [_i64, _i32]),
    'psl_tc_bwd_tmp_floats': (_sz, [_i64, _i32]),
    'psl_tc_bwd_pack_params': (C.c_int, [C.POINTER(DecoderParams), _vp, _sz, _vp, _vp]),
    'psl_color_bwd_tc': (C.c_int, [C.POINTER(DecodeCfg), _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _vp, _vp, _i32, C.POINTER(_i32), _vp]),
    'psl_add_points_ws_bytes': (_sz, [_i64]),
    'psl_add_points': (C.c_int, [C.POINTER(Grid), _vp, _vp, _vp, _vp, _i64, _vp, _f64, _i32, _i32, _f32, _f32, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _sz, _vp]),
    'psl_frustum_select_ws_bytes': (_sz, [_i64]),
    'psl_frustum_select': (C.c_int, [_vp, _i64, C.POINTER(_f64), _f64, _f64, _f64, _f64, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp,
                                     _sz, _vp]),
    'psl_frame_grad': (C.c_int, [_vp, _i32, _i32, _f64, _f64, _f64, _f64, _vp, _vp, _vp, _vp]),
    'psl_grad_candidates_ws_bytes': (_sz, [_i32]),
    'psl_grad_candidates': (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _f32, _i32, _vp, _vp, _vp, _sz, _vp]),
    'psl_pick_candidates_ws_bytes': (_sz, [_i32]),
    'psl_pick_candidates': (C.c_int, [_vp, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
}
EXPORTS = sorted(_SIGS)

_lib = None


# the tcgen05 building-block self-test (csrc/psl_tc_test.cu) is test infrastructure: its own small library, not in the product .so
TEST_LIB_PATH = os.path.join(_HERE, 'libpsl_tctest.so')
TEST_SOURCES = ['psl_tc_test.cu', 'psl_api.cu']
_TEST_SIGS = {
    'psl_tc_gemm_test': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    'psl_tc_gemm_test_h': (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
}
_test_lib = None


def build_test_lib(force: bool = False) -> str:
    deps = [os.path.join(_HERE, 'csrc', f) for f in TEST_SOURCES + ['psl_tc.cuh', 'psl_common.cuh']]
    if not force and os.path.exists(TEST_LIB_PATH) and all(os.path.getmtime(d) <= os.path.getmtime(TEST_LIB_PATH) for d in deps):
        return TEST_LIB_PATH
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    cmd = [nvcc] + NVCC_FLAGS + ['-shared', '-o', TEST_LIB_PATH] + [os.path.join(_HERE, 'csrc', f) for f in TEST_SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + res.stdout + res.stderr)
    return TEST_LIB_PATH


def load_test_lib():
    global _test_lib
    if _test_lib is None:
        if not os.path.exists(TEST_LIB_PATH):
            raise RuntimeError(f'{TEST_LIB_PATH} is missing: __graft_entry__.build() compiles it')
        lib = C.CDLL(TEST_LIB_PATH)
        for name, (res, args) in _TEST_SIGS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _test_lib = lib
    return _test_lib


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(_HERE, 'csrc', f) for f in SOURCES + HEADERS] + [os.path.join(_ROOT, 'include', 'pointslam_b200.h')]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str = None, defines=()) -> str:
    """Compile the CUDA sources for sm_100a into point_slam_b200/libpointslam_b200.so (nvcc cross-compiles
    without a GPU).  `out` / `defines`: an experiment build next to the product one (see PSL_LIB)."""
    if out is None and not force and not needs_build():
        return LIB_PATH
    out = out or LIB_PATH
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    srcs = [os.path.join(_HERE, 'csrc', f) for f in SOURCES]
    cmd = [nvcc] + NVCC_FLAGS + [f'-D{d}' for d in defines] + ['-shared', '-o', out] + srcs
    if verbose:
        print(' '.join(cmd), file=sys.stderr)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed:\n' + res.stdout + res.stderr)
    return out


def load():
    """Load the library (never builds implicitly on a GPU box; never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                           '(point_slam_b200 has no CPU or PyTorch fallback path)')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)            # AttributeError here == header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f'{what} failed ({rc}): {load().psl_last_error().decode()}')


def ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda, 'point_slam_b200 ops need CUDA tensors (no CPU path)'
    assert t.is_contiguous(), 'tensor must be contiguous'
    if dtype is not None:
        assert t.dtype == dtype, f'expected {dtype}, got {t.dtype}'
    return C.c_void_p(t.data_ptr())


TIMING_NAMES = ['knn', 'decode_fwd', 'decode_bwd', 'composite', 'scatter', 'pack', 'reduce', 'color_fwd_tc', 'color_bwd_tc', 'wgrad_tc', 'shell', 'map']


def timing_enable(on: bool):
    load().psl_timing_enable(int(on))


def timing_collect():
    """-> {name: (total_ms, launches)} since the last enable/collect (synchronises the device)."""
    ms = (C.c_float * len(TIMING_NAMES))()
    cnt = (C.c_int * len(TIMING_NAMES))()
    check(load().psl_timing_collect(ms, cnt), 'psl_timing_collect')
    return {n: (float(ms[i]), int(cnt[i])) for i, n in enumerate(TIMING_NAMES)}


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
