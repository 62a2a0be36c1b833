"""Gradient-based pixel selection of the reference (src/common.py:92-159, get_selected_index_with_grad) restated in numpy
--  TEST INFRASTRUCTURE ONLY, like the rest of oracle/.  The device kernels (csrc/psl_frame.cu) are held to it by
tests/test_gpu_frame_grad.py; it fixes the tie order that np.argpartition leaves open (DESIGN.md section 1, stated assumptions).
"""
from __future__ import annotations

import numpy as np


def grad_candidates(mag: np.ndarray, depth: np.ndarray, n: int, ratio: int = 15, window=None, depth_max=None) -> np.ndarray:
    """get_selected_index_with_grad (src/common.py:92-159) with the tie order fixed: the k = ratio * n (at most H*W) pixels of
    largest `mag` over the whole image, equal magnitudes taken in ascending flat index (np.argpartition leaves that order
    open); of those, the ones inside window = (H0, H1, W0, W1) with 0 < depth (<= depth_max when given).  -> ascending flat
    indices row * W + column (int64); there may be fewer than n."""
    H, W = mag.shape
    flat = np.asarray(mag, np.float64).reshape(-1)
    k = min(int(ratio) * int(n), flat.size)
    top = np.lexsort((np.arange(flat.size), -flat))[:k]          # primary key: -mag ascending; secondary: index
    y, x = top // W, top % W
    H0, H1, W0, W1 = window if window is not None else (0, H, 0, W)
    d = np.asarray(depth, np.float32).reshape(-1)[top]
    keep = (y >= H0) & (y < H1) & (x >= W0) & (x < W1) & (d > 0)
    if depth_max is not None:
        keep &= d <= np.float32(depth_max)
    return np.sort(top[keep]).astype(np.int64)
