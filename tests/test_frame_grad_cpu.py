"""The gradient-based pixel selection as the oracle states it (oracle.grad_select.grad_candidates): top ratio * n
magnitudes with the smaller flat index first among equal ones, then the window and depth masks.  The device kernels are held
to this restatement by tests/test_gpu_frame_grad.py."""
import numpy as np

from oracle import grad_select as O


def _planted(H=12, W=16, seed=0):
    """Magnitudes with planted ties: a few distinct levels, each shared by many pixels."""
    rng = np.random.default_rng(seed)
    mag = rng.choice(np.array([0.0, 0.05, 0.1, 0.2, 0.3]), size=(H, W), p=[0.5, 0.2, 0.15, 0.1, 0.05])
    depth = rng.uniform(0.5, 6.0, size=(H, W)).astype(np.float32)
    return mag, depth


def _brute(mag, depth, k, window, depth_max):
    """The definition read literally: walk the pixels by (magnitude descending, index ascending), stop after k."""
    H, W = mag.shape
    order = sorted(range(H * W), key=lambda p: (-mag.flat[p], p))[:k]
    H0, H1, W0, W1 = window
    out = [p for p in order if H0 <= p // W < H1 and W0 <= p % W < W1 and depth.flat[p] > 0
           and (depth_max is None or depth.flat[p] <= np.float32(depth_max))]
    return np.array(sorted(out), dtype=np.int64)


def test_top_k_takes_the_smaller_index_among_equal_magnitudes():
    mag, depth = _planted()
    H, W = mag.shape
    n, ratio = 3, 15                                   # k = 45 cuts through the 0.05 level (more than 45 pixels reach it)
    got = O.grad_candidates(mag, depth, n, ratio)
    k = n * ratio
    assert got.size == k                               # every depth > 0, whole-image window: nothing masked
    flat = mag.reshape(-1)
    cut = np.sort(flat)[::-1][k - 1]
    assert (flat[got] >= cut).all() and (flat > cut).sum() < k < (flat >= cut).sum()   # the cut splits a tie
    tied = np.nonzero(flat == cut)[0]
    n_tied = k - int((flat > cut).sum())
    assert np.array_equal(np.intersect1d(got, tied), tied[:n_tied])      # the first tied indices in index order
    assert np.array_equal(got, _brute(mag, depth, k, (0, H, 0, W), None))
    assert np.all(np.diff(got) > 0)


def test_window_and_depth_masks_apply_after_the_cut():
    mag, depth = _planted(seed=1)
    H, W = mag.shape
    depth[3, :] = 0.0                                  # holes
    depth[5, :] = 5.5                                  # beyond a 5 m bound
    win = (2, H - 2, 3, W - 3)
    for dmax in (None, 5.0):
        got = O.grad_candidates(mag, depth, 4, 15, window=win, depth_max=dmax)
        assert np.array_equal(got, _brute(mag, depth, 60, win, dmax))
        y, x = got // W, got % W
        assert ((y >= 2) & (y < H - 2) & (x >= 3) & (x < W - 3)).all()
        assert (depth.reshape(-1)[got] > 0).all()
        if dmax is not None:
            assert (depth.reshape(-1)[got] <= 5.0).all() and not (y == 5).any()
    # the window masks after the cut: pixels outside it still take places among the top k, so the windowed list is a subset
    # of the whole-image one
    whole = O.grad_candidates(mag, depth, 4, 15, depth_max=5.0)
    assert set(got.tolist()) < set(whole.tolist())


def test_fewer_candidates_than_samples():
    mag, depth = _planted(seed=2)
    H, W = mag.shape
    depth[:, : W - 2] = 0.0                            # only the last two columns have depth
    n = 10
    got = O.grad_candidates(mag, depth, n, ratio=2)
    assert got.size < n
    assert np.array_equal(got, _brute(mag, depth, 2 * n, (0, H, 0, W), None))
    assert O.grad_candidates(mag, np.zeros_like(depth), n).size == 0


def test_k_is_capped_at_the_image():
    mag, depth = _planted(seed=3)
    got = O.grad_candidates(mag, depth, 1000, 15)
    assert np.array_equal(got, np.arange(mag.size))
