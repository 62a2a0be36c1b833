// Per-frame image pass of the callers: the colour-gradient magnitude that both the dynamic-radius maps (Tracker.py:237-248,
// Mapper.py:686-704) and the gradient-based pixel selection (common.py:92-159, get_selected_index_with_grad) are built from.
//
//   psl_frame_grad        grey = 0.2125 R + 0.7154 G + 0.0721 B (float64), 3x3 Sobel with [1,2,1]/4 smoothing and a zeroed
//                         1-pixel border, mag = sqrt(gx^2 + gy^2), r_add = np.interp(clip(mag, 0, thresh), [0, 0.01, thresh],
//                         [r_max, r_max, r_min]), r_query = ratio * r_add -- synth.sobel_radius_map operation for operation
//                         (no contraction), one thread per pixel over a shared-memory tile of the grey image.
//   psl_grad_candidates   the ratio*n pixels of largest mag over the whole image (ties: smaller flat index first), of those the
//                         ones inside the window with 0 < depth <= depth_max, as ascending flat indices and a device count:
//                         stable descending radix sort of (mag bits, index), flag, DeviceSelect::Flagged.
//   psl_pick_candidates   n distinct candidates drawn uniformly WITHOUT replacement (np.random.choice(replace=False) /
//                         random_select): the caller's random key per candidate slot, slots >= count pushed to the end, stable
//                         ascending radix sort, the first n slots.  Static shapes (capacity k, count read on the device), so
//                         one captured tracking graph serves every frame.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "psl_common.cuh"

namespace psl {

static inline size_t al256f(size_t x) { return (x + 255) & ~(size_t)255; }
static inline unsigned nblkf(long long n, int tb) { return (unsigned)((n + tb - 1) / tb); }

constexpr int FG_TX = 32, FG_TY = 8;

struct FrameGradArgs {
    const float* color;                 // (H,W,3)
    int H, W;
    double r_max, r_min, thresh, slope, ratio;
    double* mag; double* r_add; double* r_query;
};

// numpy: color.astype(float64) @ [0.2125, 0.7154, 0.0721], summed left to right
__device__ __forceinline__ double grey_of(const float* __restrict__ c) {
    return __dadd_rn(__dadd_rn(__dmul_rn((double)__ldg(c), 0.2125), __dmul_rn((double)__ldg(c + 1), 0.7154)),
                     __dmul_rn((double)__ldg(c + 2), 0.0721));
}
// (a + 2 b) + c, the order numpy evaluates `g[..] + 2 * g[..] + g[..]` in
__device__ __forceinline__ double sobel_row(double a, double b, double c) { return __dadd_rn(__dadd_rn(a, __dmul_rn(2.0, b)), c); }

__global__ void __launch_bounds__(FG_TX * FG_TY) k_frame_grad(FrameGradArgs a) {
    __shared__ double g[FG_TY + 2][FG_TX + 2];
    const int x0 = blockIdx.x * FG_TX - 1, y0 = blockIdx.y * FG_TY - 1;
    for (int t = threadIdx.y * FG_TX + threadIdx.x; t < (FG_TY + 2) * (FG_TX + 2); t += FG_TX * FG_TY) {
        const int ty = t / (FG_TX + 2), tx = t % (FG_TX + 2);
        const int x = x0 + tx, y = y0 + ty;
        g[ty][tx] = (x >= 0 && x < a.W && y >= 0 && y < a.H) ? grey_of(a.color + ((size_t)y * a.W + x) * 3) : 0.0;
    }
    __syncthreads();
    const int x = blockIdx.x * FG_TX + threadIdx.x, y = blockIdx.y * FG_TY + threadIdx.y;
    if (x >= a.W || y >= a.H) return;
    double m = 0.0;                                                      // zero border: gx = gy = 0
    if (x > 0 && y > 0 && x < a.W - 1 && y < a.H - 1) {
        const int cx = threadIdx.x + 1, cy = threadIdx.y + 1;
        const double gy = __dmul_rn(__dsub_rn(sobel_row(g[cy + 1][cx - 1], g[cy + 1][cx], g[cy + 1][cx + 1]),
                                              sobel_row(g[cy - 1][cx - 1], g[cy - 1][cx], g[cy - 1][cx + 1])), 0.25);   // / 4.0: exact
        const double gx = __dmul_rn(__dsub_rn(sobel_row(g[cy - 1][cx + 1], g[cy][cx + 1], g[cy + 1][cx + 1]),
                                              sobel_row(g[cy - 1][cx - 1], g[cy][cx - 1], g[cy + 1][cx - 1])), 0.25);
        m = __dsqrt_rn(__dadd_rn(__dmul_rn(gx, gx), __dmul_rn(gy, gy)));
    }
    const size_t p = (size_t)y * a.W + x;
    if (a.mag) a.mag[p] = m;
    if (a.r_add || a.r_query) {
        // np.interp over xp = [0, 0.01, thresh], fp = [r_max, r_max, r_min] of np.clip(mag, 0, thresh) (numpy's arr_interp:
        // a knot returns its value, inside an interval slope * (x - xp[j]) + fp[j])
        const double c = fmin(fmax(m, 0.0), a.thresh);
        double r;
        if (c == a.thresh) r = a.r_min;
        else if (c <= 0.01) r = a.r_max;                                 // flat first interval: 0 * x + r_max
        else r = __dadd_rn(__dmul_rn(a.slope, __dsub_rn(c, 0.01)), a.r_max);
        if (a.r_add) a.r_add[p] = r;
        if (a.r_query) a.r_query[p] = __dmul_rn(a.ratio, r);
    }
}

// ---- candidate list ------------------------------------------------------------------------------------------------------------
__global__ void k_mag_keys(const double* __restrict__ mag, int n, unsigned long long* __restrict__ keys, int* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long b = (unsigned long long)__double_as_longlong(mag[i]);
    keys[i] = (b >> 63) ? 0ull : b;                 // mag >= 0: the bit pattern orders like the value (-0.0 -> +0.0)
    vals[i] = i;
}

__global__ void k_cand_flag(const int* __restrict__ order, int k, int W, int H0, int H1, int W0, int W1, const float* __restrict__ depth,
                            float depth_max, uint8_t* __restrict__ flags) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= k) return;
    const int p = order[s];
    const int y = p / W, x = p - (p / W) * W;
    const float d = depth[p];
    flags[p] = (y >= H0 && y < H1 && x >= W0 && x < W1 && d > 0.f && d <= depth_max) ? 1 : 0;
}

// ---- draw without replacement --------------------------------------------------------------------------------------------------
__global__ void k_pick_keys(const uint32_t* __restrict__ rnd, const int32_t* __restrict__ count, int cap, uint32_t* __restrict__ keys,
                            int* __restrict__ slots) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= cap) return;
    keys[s] = s < count[0] ? rnd[s] : 0xffffffffu;   // empty slots sort last (stable sort: after every filled slot)
    slots[s] = s;
}

__global__ void k_pick_emit(const int* __restrict__ slots, const int32_t* __restrict__ count, const int64_t* __restrict__ cand, int n,
                            int W, int H0, int W0, int ww, int64_t* __restrict__ pix) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int s = slots[t];
    if (s < count[0]) {
        const long long p = cand[s];
        const long long y = p / W, x = p - y * W;
        pix[t] = (y - H0) * ww + (x - W0);
    } else {
        pix[t] = -1;                                   // fewer than n candidates: no pixel (psl_sample_rays gives it depth 0)
    }
}

}  // namespace psl

using namespace psl;

extern "C" int psl_frame_grad(const float* color, int32_t H, int32_t W, double r_add_max, double r_add_min, double radius_query_ratio,
                              double color_grad_threshold, double* mag, double* r_add, double* r_query, psl_stream_t stream) {
    PSL_REQUIRE(color, "NULL argument");
    PSL_REQUIRE(H > 0 && W > 0 && (long long)H * W < (1ll << 31), "bad image size");
    PSL_REQUIRE(color_grad_threshold > 0.01, "color_grad_threshold must exceed the 0.01 knot of the radius map");
    if (!mag && !r_add && !r_query) return 0;
    FrameGradArgs a{};
    a.color = color; a.H = H; a.W = W;
    a.r_max = r_add_max; a.r_min = r_add_min; a.thresh = color_grad_threshold; a.ratio = radius_query_ratio;
    a.slope = (r_add_min - r_add_max) / (color_grad_threshold - 0.01);       // numpy's precomputed interval slope
    a.mag = mag; a.r_add = r_add; a.r_query = r_query;
    cudaStream_t st = as_stream(stream);
    TimingScope ts(T_MAP, st);
    k_frame_grad<<<dim3(nblkf(W, FG_TX), nblkf(H, FG_TY)), dim3(FG_TX, FG_TY), 0, st>>>(a);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

static size_t grad_cand_cub_bytes(int n) {
    size_t sort_b = 0, sel_b = 0;
    cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_b, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                              (const int*)nullptr, (int*)nullptr, n, 0, 64);
    cub::CountingInputIterator<int64_t> it(0);
    cub::DeviceSelect::Flagged(nullptr, sel_b, it, (const uint8_t*)nullptr, (int64_t*)nullptr, (int32_t*)nullptr, n);
    return sort_b > sel_b ? sort_b : sel_b;
}

extern "C" size_t psl_grad_candidates_ws_bytes(int32_t n_pixels) {
    const size_t n = n_pixels > 0 ? (size_t)n_pixels : 0;
    return 2 * al256f(sizeof(unsigned long long) * n) + 2 * al256f(sizeof(int) * n) + al256f(n) +
           al256f(grad_cand_cub_bytes((int)n)) + 256;
}

extern "C" int psl_grad_candidates(const double* mag, const float* depth, int32_t H, int32_t W, int32_t H0, int32_t H1, int32_t W0,
                                   int32_t W1, float depth_max, int32_t k, int64_t* cand, int32_t* count, void* ws, size_t ws_bytes,
                                   psl_stream_t stream) {
    PSL_REQUIRE(mag && depth && cand && count && ws, "NULL argument");
    PSL_REQUIRE(H > 0 && W > 0 && (long long)H * W < (1ll << 31), "bad image size");
    PSL_REQUIRE(0 <= H0 && H0 <= H1 && H1 <= H && 0 <= W0 && W0 <= W1 && W1 <= W, "bad window");
    const int n = H * W;
    PSL_REQUIRE(k >= 1 && k <= n, "k must lie in [1, H*W]");
    PSL_REQUIRE(ws_bytes >= psl_grad_candidates_ws_bytes(n), "workspace too small");
    unsigned char* w = static_cast<unsigned char*>(ws);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(w); w += al256f(sizeof(unsigned long long) * n);
    unsigned long long* keys_s = reinterpret_cast<unsigned long long*>(w); w += al256f(sizeof(unsigned long long) * n);
    int* vals = reinterpret_cast<int*>(w); w += al256f(sizeof(int) * n);
    int* vals_s = reinterpret_cast<int*>(w); w += al256f(sizeof(int) * n);
    uint8_t* flags = w; w += al256f((size_t)n);
    size_t cub_bytes = ws_bytes - (size_t)(w - static_cast<unsigned char*>(ws));
    cudaStream_t st = as_stream(stream);
    TimingScope ts(T_MAP, st, 4);
    PSL_CHECK_CUDA(cudaMemsetAsync(flags, 0, (size_t)n, st));
    k_mag_keys<<<nblkf(n, 256), 256, 0, st>>>(mag, n, keys, vals);
    PSL_CHECK_CUDA(cudaGetLastError());
    // stable: equal magnitudes keep ascending index order, so the cut at k takes the smaller flat indices first
    PSL_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(w, cub_bytes, keys, keys_s, vals, vals_s, n, 0, 64, st));
    k_cand_flag<<<nblkf(k, 256), 256, 0, st>>>(vals_s, k, W, H0, H1, W0, W1, depth, depth_max, flags);
    PSL_CHECK_CUDA(cudaGetLastError());
    cub::CountingInputIterator<int64_t> it(0);
    PSL_CHECK_CUDA(cub::DeviceSelect::Flagged(w, cub_bytes, it, flags, cand, count, n, st));
    return 0;
}

static size_t pick_cub_bytes(int cap) {
    size_t b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int*)nullptr, (int*)nullptr, cap,
                                    0, 32);
    return b;
}

extern "C" size_t psl_pick_candidates_ws_bytes(int32_t capacity) {
    const size_t c = capacity > 0 ? (size_t)capacity : 0;
    return 2 * al256f(sizeof(uint32_t) * c) + 2 * al256f(sizeof(int) * c) + al256f(pick_cub_bytes((int)c)) + 256;
}

extern "C" int psl_pick_candidates(const int64_t* cand, const int32_t* count, int32_t capacity, const uint32_t* keys, int32_t n,
                                   int32_t W, int32_t H0, int32_t W0, int32_t win_w, int64_t* pix, void* ws, size_t ws_bytes,
                                   psl_stream_t stream) {
    PSL_REQUIRE(cand && count && keys && pix && ws, "NULL argument");
    PSL_REQUIRE(capacity >= 1 && n >= 1 && n <= capacity, "need 1 <= n <= capacity");
    PSL_REQUIRE(W > 0 && win_w > 0 && H0 >= 0 && W0 >= 0 && W0 + win_w <= W, "bad sampling window");
    PSL_REQUIRE(ws_bytes >= psl_pick_candidates_ws_bytes(capacity), "workspace too small");
    unsigned char* w = static_cast<unsigned char*>(ws);
    uint32_t* k_in = reinterpret_cast<uint32_t*>(w); w += al256f(sizeof(uint32_t) * capacity);
    uint32_t* k_out = reinterpret_cast<uint32_t*>(w); w += al256f(sizeof(uint32_t) * capacity);
    int* s_in = reinterpret_cast<int*>(w); w += al256f(sizeof(int) * capacity);
    int* s_out = reinterpret_cast<int*>(w); w += al256f(sizeof(int) * capacity);
    size_t cub_bytes = ws_bytes - (size_t)(w - static_cast<unsigned char*>(ws));
    cudaStream_t st = as_stream(stream);
    TimingScope ts(T_SHELL, st, 3);
    k_pick_keys<<<nblkf(capacity, 256), 256, 0, st>>>(keys, count, capacity, k_in, s_in);
    PSL_CHECK_CUDA(cudaGetLastError());
    PSL_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(w, cub_bytes, k_in, k_out, s_in, s_out, capacity, 0, 32, st));
    k_pick_emit<<<nblkf(n, 256), 256, 0, st>>>(s_out, count, cand, n, W, H0, W0, win_w, pix);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}
