// The iteration shell around the render call, as a handful of kernels instead of ~250 tiny ATen launches:
// pixel -> ray sampling from a pose (Tracker.py:118-141, Mapper.py:459-500; common.py:40-56, 225-267), the depth-outlier gate
// (Tracker.py:142-148 / Mapper.py:507-513), the tracking / mapping losses WITH their gradients (Tracker.py:158-180,
// Mapper.py:524-552), the pose chain rule back to [quaternion, T], and Adam on the pose / the selected feature rows
// (torch.optim.Adam semantics).  Every reduction is a fixed-order tree inside one CTA: results are bit-reproducible.
#include "psl_composite.cuh"

namespace psl {

// rotation of an UN-normalised quaternion (w,x,y,z), common.py:225-248 (same expression order, no FMA contraction; the
// 4-term sum in the order ATen's CUDA reduction uses, (a0 + a2) + (a1 + a3), so that rays are bit-identical to the torch ops)
__device__ __forceinline__ void quat_to_rot(const float* __restrict__ q, float R[9]) {
    const float qr = q[0], qi = q[1], qj = q[2], qk = q[3];
    const float n = __fadd_rn(__fadd_rn(__fmul_rn(qr, qr), __fmul_rn(qj, qj)), __fadd_rn(__fmul_rn(qi, qi), __fmul_rn(qk, qk)));
    const float s = __fdiv_rn(2.0f, n);
    const float ii = __fmul_rn(qi, qi), jj = __fmul_rn(qj, qj), kk = __fmul_rn(qk, qk);
    R[0] = __fsub_rn(1.0f, __fmul_rn(s, __fadd_rn(jj, kk)));
    R[1] = __fmul_rn(s, __fsub_rn(__fmul_rn(qi, qj), __fmul_rn(qk, qr)));
    R[2] = __fmul_rn(s, __fadd_rn(__fmul_rn(qi, qk), __fmul_rn(qj, qr)));
    R[3] = __fmul_rn(s, __fadd_rn(__fmul_rn(qi, qj), __fmul_rn(qk, qr)));
    R[4] = __fsub_rn(1.0f, __fmul_rn(s, __fadd_rn(ii, kk)));
    R[5] = __fmul_rn(s, __fsub_rn(__fmul_rn(qj, qk), __fmul_rn(qi, qr)));
    R[6] = __fmul_rn(s, __fsub_rn(__fmul_rn(qi, qk), __fmul_rn(qj, qr)));
    R[7] = __fmul_rn(s, __fadd_rn(__fmul_rn(qj, qk), __fmul_rn(qi, qr)));
    R[8] = __fsub_rn(1.0f, __fmul_rn(s, __fadd_rn(ii, jj)));
}

__device__ __forceinline__ void pixel_dir(float i, float j, float fx, float fy, float cx, float cy, float d[3]) {
    // common.py:49-50; ATen's CUDA division by a host scalar multiplies by the fp32 reciprocal -- do the same (bit-identical rays)
    d[0] = __fmul_rn(__fsub_rn(i, cx), __frcp_rn(fx));
    d[1] = -__fmul_rn(__fsub_rn(j, cy), __frcp_rn(fy));
    d[2] = -1.0f;
}

struct SampleArgs {
    const long long* pix;      // (K*per) flattened window index per sample
    int K, per, H, W, H0, W0, ww;
    const float* cam;          // (7) [quat, T] (K must be 1) or NULL
    const float* c2w;          // (K,3,4) or NULL
    const float* color;        // (K,H,W,3)
    const float* depth;        // (K,H,W)
    const double* dyn;         // (K,H,W) or NULL
    float fx, fy, cx, cy;
    float* rays_o; float* rays_d; float* b_depth; float* b_color; double* r2;
};

__global__ void k_sample_rays(SampleArgs a) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.K * a.per) return;
    const int k = t / a.per;
    const long long p_in = a.pix[t];
    const bool none = p_in < 0;                        // no pixel (psl_pick_candidates with fewer candidates than samples)
    const long long p = none ? 0 : p_in;
    const int jj = (int)(p / a.ww) + a.H0, ii = (int)(p % a.ww) + a.W0;
    float R[9], T[3];
    if (a.cam) {
        quat_to_rot(a.cam, R);
        T[0] = a.cam[4]; T[1] = a.cam[5]; T[2] = a.cam[6];
    } else {
        const float* m = a.c2w + (size_t)k * 12;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            R[r * 3] = m[r * 4]; R[r * 3 + 1] = m[r * 4 + 1]; R[r * 3 + 2] = m[r * 4 + 2];
            T[r] = m[r * 4 + 3];
        }
    }
    float d[3];
    pixel_dir((float)ii, (float)jj, a.fx, a.fy, a.cx, a.cy, d);
#pragma unroll
    for (int r = 0; r < 3; ++r) {                      // rays_d = sum(dirs * c2w[:3,:3], -1), common.py:53; ATen's order: (x + z) + y
        a.rays_d[t * 3 + r] = __fadd_rn(__fadd_rn(__fmul_rn(d[0], R[r * 3]), __fmul_rn(d[2], R[r * 3 + 2])), __fmul_rn(d[1], R[r * 3 + 1]));
        a.rays_o[t * 3 + r] = T[r];
    }
    const size_t px = ((size_t)k * a.H + jj) * a.W + ii;
    a.b_depth[t] = none ? 0.f : a.depth[px];          // depth 0: outside the depth gate, zero loss weight
    a.b_color[t * 3] = a.color[px * 3]; a.b_color[t * 3 + 1] = a.color[px * 3 + 1]; a.b_color[t * 3 + 2] = a.color[px * 3 + 2];
    if (a.r2) { const double r = a.dyn[px]; a.r2[t] = r * r; }
}

// ---- depth gate: inside = depth > 0 and depth <= min(10 * median(valid), 1.2 * max(valid)) --------------------------------------
// The lower median (torch.median) is the k-th smallest valid depth, k = (count - 1) / 2: found by a 4-pass MSB-first radix
// select over the float bit patterns (positive floats order like their bits) with a 256-bin shared histogram per pass.
constexpr int GATE_MAX = 8192;
__global__ void __launch_bounds__(1024, 1) k_depth_gate(const float* __restrict__ b_depth, int n, float* __restrict__ depth_in,
                                                        unsigned char* __restrict__ inside) {
    __shared__ unsigned hist[256];
    __shared__ unsigned s_red[32], s_max[32];
    __shared__ unsigned s_prefix, s_k;
    constexpr int PER = GATE_MAX / 1024;
    unsigned key[PER];
    unsigned cnt = 0, mx = 0;
#pragma unroll
    for (int e = 0; e < PER; ++e) {
        const int i = threadIdx.x + e * 1024;
        const float d = i < n ? b_depth[i] : 0.f;
        key[e] = d > 0.f ? __float_as_uint(d) : 0u;      // 0 = not valid (valid keys are > 0)
        cnt += key[e] != 0u;
        mx = max(mx, key[e]);
    }
    for (int o = 16; o; o >>= 1) { cnt += __shfl_xor_sync(0xffffffffu, cnt, o); mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
    if ((threadIdx.x & 31) == 0) { s_red[threadIdx.x >> 5] = cnt; s_max[threadIdx.x >> 5] = mx; }
    if (threadIdx.x < 256) hist[threadIdx.x] = 0;
    __syncthreads();
    unsigned total = 0, gmax = 0;
    for (int w = 0; w < 32; ++w) { total += s_red[w]; gmax = max(gmax, s_max[w]); }
    if (threadIdx.x == 0) { s_prefix = 0; s_k = total ? (total - 1) >> 1 : 0; }
    __syncthreads();
    for (int shift = 24; shift >= 0 && total; shift -= 8) {
        const unsigned prefix = s_prefix;
        const unsigned himask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
        for (int e = 0; e < PER; ++e)
            if (key[e] != 0u && (key[e] & himask) == prefix) atomicAdd(&hist[(key[e] >> shift) & 255u], 1u);
        __syncthreads();
        if (threadIdx.x < 32) {                          // warp 0: find the bin holding rank k (8 bins per lane + shuffle scan)
            unsigned c[8], sum = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { c[q] = hist[threadIdx.x * 8 + q]; sum += c[q]; }
            unsigned incl = sum;
            for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += v; }
            const unsigned excl = incl - sum, k = s_k;
            if (k >= excl && k < incl) {
                unsigned run = excl;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (k >= run && k < run + c[q]) { s_prefix = prefix | ((unsigned)(threadIdx.x * 8 + q) << shift); s_k = k - run; }
                    run += c[q];
                }
            }
        }
        __syncthreads();
        if (threadIdx.x < 256) hist[threadIdx.x] = 0;
        __syncthreads();
    }
    float thr = __int_as_float(0x7fc00000);            // no valid depth: NaN -> nothing is inside
    if (total > 0) thr = fminf(__fmul_rn(10.0f, __uint_as_float(s_prefix)), __fmul_rn(1.2f, __uint_as_float(gmax)));
#pragma unroll
    for (int e = 0; e < PER; ++e) {
        const int i = threadIdx.x + e * 1024;
        if (i < n) {
            const float d = __uint_as_float(key[e]);
            const bool in = key[e] != 0u && d <= thr;
            inside[i] = in;
            depth_in[i] = in ? d : 0.f;
        }
    }
}

// ---- block-wide fixed-order sum --------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum(float v, float* sh) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();                                   // sh may still be read from a previous call
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[w];
    return t;
}

// mode 0: tracking loss (Tracker.py:158-180): tmp = |gt - d| / sqrt(var + 1e-10) (var detached), mask = ok & tmp < 10 * mean_inside(tmp),
//         loss = sum_mask clamp(tmp, 0, 1e3) + w_color * sum_mask |gt_rgb - rgb|
// mode 1: mapping loss (Mapper.py:524-552): mask = inside & ray_mask & !isnan(d), loss = sum_mask |gt - d| (+ w_color * sum_mask |gt_rgb - rgb|)
__global__ void __launch_bounds__(1024, 1) k_shell_loss(int mode, int n, const float* __restrict__ depth_in,
                                                        const unsigned char* __restrict__ inside,
                                                        const unsigned char* __restrict__ ray_mask, const float* __restrict__ depth,
                                                        const float* __restrict__ var, const float* __restrict__ rgb,
                                                        const float* __restrict__ b_color, float w_color, float* __restrict__ loss,
                                                        float* __restrict__ d_depth, float* __restrict__ d_rgb) {
    __shared__ float sh[32];
    float thr = 0.f;
    if (mode == 0) {
        float a = 0.f, c = 0.f;
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            if (inside[i]) { a += fabsf(depth_in[i] - depth[i]) / sqrtf(var[i] + 1e-10f); c += 1.f; }
        const float sa = block_sum(a, sh), sc = block_sum(c, sh);
        thr = 10.0f * (sa / fmaxf(sc, 1.0f));
    }
    float ld = 0.f, lc = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float d = depth[i], g = depth_in[i];
        bool m = inside[i] && !isnan(d);
        float gd = 0.f;
        if (mode == 0) {
            const float v = var[i];
            const float inv = 1.0f / sqrtf(v + 1e-10f);
            const float tmp = fabsf(g - d) * inv;
            m = m && !isnan(v) && tmp < thr;
            if (m) {
                ld += fminf(fmaxf(tmp, 0.f), 1e3f);
                const float sg = (g > d) ? 1.f : ((g < d) ? -1.f : 0.f);
                gd = (tmp <= 1e3f) ? -sg * inv : 0.f;
            }
        } else {
            m = m && ray_mask[i];
            if (m) {
                ld += fabsf(g - d);
                gd = (g > d) ? -1.f : ((g < d) ? 1.f : 0.f);
            }
        }
        d_depth[i] = gd;
        if (d_rgb) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float t = b_color[i * 3 + c], r = rgb[i * 3 + c];
                float gc = 0.f;
                if (m) {
                    lc += fabsf(t - r);
                    gc = (t > r) ? -w_color : ((t < r) ? w_color : 0.f);
                }
                d_rgb[i * 3 + c] = gc;
            }
        }
    }
    const float sd = block_sum(ld, sh), sc = block_sum(lc, sh);
    if (threadIdx.x == 0) loss[0] = d_rgb ? sd + w_color * sc : sd;
}

// ---- fused render tail: composite -> ray mask -> loss -> composite backward, ONE single-CTA launch ------------------------------------
// The four stand-alone kernels it replaces (k_composite_fwd, k_ray_mask, k_shell_loss, k_composite_bwd) move < 1 MB each and are
// pure launch latency inside an iteration graph.  Same per-ray arithmetic (psl_composite.cuh), same thread <-> ray mapping and
// summation order as k_shell_loss, so loss and gradients are those of the separate kernels.
__global__ void __launch_bounds__(1024, 1) k_render_tail(int mode, int n, int S, float coef, int min_count,
                                                         const float4* __restrict__ raw, const unsigned char* __restrict__ has_nb,
                                                         const float* __restrict__ z_vals, const float* __restrict__ depth_in,
                                                         const unsigned char* __restrict__ inside, const float* __restrict__ b_color,
                                                         float w_color, float* __restrict__ depth, float* __restrict__ var,
                                                         float* __restrict__ rgb, unsigned char* __restrict__ ray_mask,
                                                         float* __restrict__ loss, float4* __restrict__ d_raw) {
    __shared__ float sh[32];
    // phase 1: composite + ray validity
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const RayOut o = composite_fwd_ray(raw, has_nb, z_vals, i, S, coef, nullptr);
        depth[i] = o.depth; var[i] = o.var;
        rgb[i * 3] = o.r; rgb[i * 3 + 1] = o.g; rgb[i * 3 + 2] = o.b;
        int c = 0;
        for (int s = 0; s < S; ++s) c += has_nb[(long long)i * S + s] ? 1 : 0;
        ray_mask[i] = c >= min_count;
    }
    // (every thread re-reads only the rays it wrote itself: no barrier needed for the global round trip)
    float thr = 0.f;
    if (mode == 0) {
        float a = 0.f, c = 0.f;
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            if (inside[i]) { a += fabsf(depth_in[i] - depth[i]) / sqrtf(var[i] + 1e-10f); c += 1.f; }
        const float sa = block_sum(a, sh), sc = block_sum(c, sh);
        thr = 10.0f * (sa / fmaxf(sc, 1.0f));
    }
    float ld = 0.f, lc = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float d = depth[i], g = depth_in[i];
        bool m = inside[i] && !isnan(d);
        float gd = 0.f, gc[3] = {0.f, 0.f, 0.f};
        if (mode == 0) {
            const float v = var[i];
            const float inv = 1.0f / sqrtf(v + 1e-10f);
            const float tmp = fabsf(g - d) * inv;
            m = m && !isnan(v) && tmp < thr;
            if (m) {
                ld += fminf(fmaxf(tmp, 0.f), 1e3f);
                const float sg = (g > d) ? 1.f : ((g < d) ? -1.f : 0.f);
                gd = (tmp <= 1e3f) ? -sg * inv : 0.f;
            }
        } else {
            m = m && ray_mask[i];
            if (m) {
                ld += fabsf(g - d);
                gd = (g > d) ? -1.f : ((g < d) ? 1.f : 0.f);
            }
        }
        if (b_color) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float t = b_color[i * 3 + c], r = rgb[i * 3 + c];
                if (m) {
                    lc += fabsf(t - r);
                    gc[c] = (t > r) ? -w_color : ((t < r) ? w_color : 0.f);
                }
            }
        }
        composite_bwd_ray(raw, has_nb, z_vals, i, S, coef, gd, 0.f, gc[0], gc[1], gc[2], d_raw);
    }
    const float sd = block_sum(ld, sh), sc = block_sum(lc, sh);
    if (threadIdx.x == 0) loss[0] = b_color ? sd + w_color * sc : sd;
}

// mapping variant, one thread per ray over as many CTAs as the rays need: the mapping loss has no batch statistic (no 10 x mean gate),
// so a ray's gradient depends on that ray only.  The loss value is reduced in a fixed order: per-block sums -> partial[block], the
// block that draws the last ticket adds the partials by block index (deterministic whichever block that is) and re-arms the ticket.
__global__ void __launch_bounds__(128) k_render_tail_map(int n, int S, float coef, int min_count, const float4* __restrict__ raw,
                                                         const unsigned char* __restrict__ has_nb, const float* __restrict__ z_vals,
                                                         const float* __restrict__ depth_in, const unsigned char* __restrict__ inside,
                                                         const float* __restrict__ b_color, float w_color, float* __restrict__ depth,
                                                         float* __restrict__ var, float* __restrict__ rgb,
                                                         unsigned char* __restrict__ ray_mask, float* __restrict__ loss,
                                                         float4* __restrict__ d_raw, float2* __restrict__ partial, unsigned* __restrict__ ticket) {
    __shared__ float sh[8];
    __shared__ bool last;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float ld = 0.f, lc = 0.f;
    if (i < n) {
        const RayOut o = composite_fwd_ray(raw, has_nb, z_vals, i, S, coef, nullptr);
        depth[i] = o.depth; var[i] = o.var;
        rgb[i * 3] = o.r; rgb[i * 3 + 1] = o.g; rgb[i * 3 + 2] = o.b;
        int c = 0;
        for (int s = 0; s < S; ++s) c += has_nb[(long long)i * S + s] ? 1 : 0;
        const bool rm = c >= min_count;
        ray_mask[i] = rm;
        const float d = o.depth, g = depth_in[i];
        const bool m = inside[i] && !isnan(d) && rm;
        float gd = 0.f, gc[3] = {0.f, 0.f, 0.f};
        if (m) {
            ld = fabsf(g - d);
            gd = (g > d) ? -1.f : ((g < d) ? 1.f : 0.f);
            if (b_color) {
                const float pr[3] = {o.r, o.g, o.b};
#pragma unroll
                for (int c3 = 0; c3 < 3; ++c3) {
                    const float t = b_color[i * 3 + c3];
                    lc += fabsf(t - pr[c3]);
                    gc[c3] = (t > pr[c3]) ? -w_color : ((t < pr[c3]) ? w_color : 0.f);
                }
            }
        }
        composite_bwd_ray(raw, has_nb, z_vals, i, S, coef, gd, 0.f, gc[0], gc[1], gc[2], d_raw);
    }
    for (int o = 16; o; o >>= 1) { ld += __shfl_xor_sync(0xffffffffu, ld, o); lc += __shfl_xor_sync(0xffffffffu, lc, o); }
    if ((threadIdx.x & 31) == 0) { sh[threadIdx.x >> 5] = ld; sh[4 + (threadIdx.x >> 5)] = lc; }
    __syncthreads();
    if (threadIdx.x == 0) {
        partial[blockIdx.x] = make_float2((sh[0] + sh[1]) + (sh[2] + sh[3]), (sh[4] + sh[5]) + (sh[6] + sh[7]));
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
        if (last) {
            __threadfence();
            float sd = 0.f, sc = 0.f;
            for (unsigned b = 0; b < gridDim.x; ++b) { const float2 p = __ldcg(partial + b); sd += p.x; sc += p.y; }
            loss[0] = b_color ? sd + w_color * sc : sd;
            *ticket = 0u;
        }
    }
}

// ---- pose chain rule: (d_rays_o, d_rays_d) -> d[quat, T] ---------------------------------------------------------------------
__global__ void __launch_bounds__(1024, 1) k_pose_bwd(const long long* __restrict__ pix, int n, int H0, int W0, int ww, float fx, float fy,
                                                      float cx, float cy, const float* __restrict__ cam, const float* __restrict__ d_o,
                                                      const float* __restrict__ d_d, float* __restrict__ d_cam) {
    __shared__ float part[32][12];
    __shared__ float acc[12];
    float G[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, gT[3] = {0.f, 0.f, 0.f};
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        const long long p = pix[t] < 0 ? 0 : pix[t];     // the ray psl_sample_rays made for "no pixel" (its gradient is zero)
        float d[3];
        pixel_dir((float)((int)(p % ww) + W0), (float)((int)(p / ww) + H0), fx, fy, cx, cy, d);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float g = d_d[t * 3 + r];
            G[r * 3] += g * d[0]; G[r * 3 + 1] += g * d[1]; G[r * 3 + 2] += g * d[2];
            gT[r] += d_o[t * 3 + r];
        }
    }
#pragma unroll
    for (int e = 0; e < 12; ++e) {                     // warp shuffles, then one fixed-order pass over the 32 warp partials
        float v = e < 9 ? G[e] : gT[e - 9];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5][e] = v;
    }
    __syncthreads();
    if (threadIdx.x < 12) {
        float t = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w][threadIdx.x];
        acc[threadIdx.x] = t;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const float r = cam[0], i = cam[1], j = cam[2], k = cam[3];
    const float nn = r * r + i * i + j * j + k * k, s = 2.0f / nn;
    const float* g = acc;
    const float dLds = -g[0] * (j * j + k * k) + g[1] * (i * j - k * r) + g[2] * (i * k + j * r) + g[3] * (i * j + k * r) -
                       g[4] * (i * i + k * k) + g[5] * (j * k - i * r) + g[6] * (i * k - j * r) + g[7] * (j * k + i * r) -
                       g[8] * (i * i + j * j);
    const float c = -s * s * dLds;                     // ds/dq_a = -s^2 q_a
    d_cam[0] = s * (-g[1] * k + g[2] * j + g[3] * k - g[5] * i - g[6] * j + g[7] * i) + c * r;
    d_cam[1] = s * (g[1] * j + g[2] * k + g[3] * j - 2.f * g[4] * i - g[5] * r + g[6] * k + g[7] * r - 2.f * g[8] * i) + c * i;
    d_cam[2] = s * (-2.f * g[0] * j + g[1] * i + g[2] * r + g[3] * i + g[5] * k - g[6] * r + g[7] * k - 2.f * g[8] * j) + c * j;
    d_cam[3] = s * (-2.f * g[0] * k - g[1] * r + g[2] * i + g[3] * r - 2.f * g[4] * k + g[5] * j + g[6] * i + g[7] * j) + c * k;
    d_cam[4] = acc[9]; d_cam[5] = acc[10]; d_cam[6] = acc[11];
}

// ---- Adam (torch.optim.Adam, no weight decay / amsgrad) on rows of a 2-D tensor selected by an index list -----------------------
__global__ void k_adam_tick(int* step) { step[0] += 1; }

struct AdamArgs {
    float* param; float* grad; float* m; float* v;
    const long long* rows; long long n_slots; int width; const int* step;
    float lr, b1, b2, eps; int zero_grad;
};

__device__ __forceinline__ float adam_update(float p, float g, float& m, float& v, float b1, float b2, float step_size, float inv_sqrt_bc2,
                                             float eps) {
    m = m + (g - m) * (1.0f - b1);                     // exp_avg.lerp_(grad, 1 - beta1)
    v = b2 * v + (1.0f - b2) * g * g;                  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) * inv_sqrt_bc2 + eps; // sqrt(v) / sqrt(bias_correction2) + eps
    return p - step_size * (m / denom);
}

// VEC = 4: one thread per 4 consecutive channels (width % 4 == 0, 16-byte aligned rows); VEC = 1: generic.
// Grid-stride over (slot, channel group): the bias corrections (two powf + a block barrier) are computed once per resident
// block instead of once per 256 elements -- with 131 072 slots of which a frustum uses ~30 000 the per-block prologue was
// most of the kernel's 18 us.
template <int VEC>
__global__ void k_adam_rows(AdamArgs a) {
    __shared__ float s_c[2];
    if (threadIdx.x == 0) {
        const float t = (float)a.step[0];
        s_c[0] = a.lr / (1.0f - powf(a.b1, t));
        s_c[1] = 1.0f / sqrtf(1.0f - powf(a.b2, t));
    }
    __syncthreads();
    const float step_size = s_c[0], isb = s_c[1];
    const int wv = a.width / VEC;
    const long long total = a.n_slots * wv, stride = (long long)gridDim.x * blockDim.x;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        const long long slot = e / wv;
        const int c = (int)(e - slot * wv) * VEC;
        const long long row = a.rows ? a.rows[slot] : slot;
        if (row < 0) continue;
        const long long so = slot * a.width + c, po = row * a.width + c;
        if (VEC == 4) {
            const float4 g = *reinterpret_cast<const float4*>(a.grad + so);
            float4 m = *reinterpret_cast<const float4*>(a.m + so), v = *reinterpret_cast<const float4*>(a.v + so);
            float4 p = *reinterpret_cast<const float4*>(a.param + po);
            p.x = adam_update(p.x, g.x, m.x, v.x, a.b1, a.b2, step_size, isb, a.eps);
            p.y = adam_update(p.y, g.y, m.y, v.y, a.b1, a.b2, step_size, isb, a.eps);
            p.z = adam_update(p.z, g.z, m.z, v.z, a.b1, a.b2, step_size, isb, a.eps);
            p.w = adam_update(p.w, g.w, m.w, v.w, a.b1, a.b2, step_size, isb, a.eps);
            *reinterpret_cast<float4*>(a.m + so) = m;
            *reinterpret_cast<float4*>(a.v + so) = v;
            *reinterpret_cast<float4*>(a.param + po) = p;
            if (a.zero_grad) *reinterpret_cast<float4*>(a.grad + so) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            const float g = a.grad[so];
            float m = a.m[so], v = a.v[so];
            a.param[po] = adam_update(a.param[po], g, m, v, a.b1, a.b2, step_size, isb, a.eps);
            a.m[so] = m; a.v[so] = v;
            if (a.zero_grad) a.grad[so] = 0.f;
        }
    }
}

// ---- pose step of the tracker: Adam on [quat(4), T(3)] with separate learning rates + the reference's candidate bookkeeping --------
// Tracker.py:289-349: with tracking.separate_LR the quaternion steps with lr/5 (two parameter groups of ONE optimizer, hence one
// shared step count); the frame's result is the pose of the iteration with the smallest loss -- the pose that iteration RENDERED
// with when separate_LR is on (camera_tensor is re-built with torch.cat before each call), the stepped pose otherwise
// (the Variable is updated in place before .detach().clone()).
__global__ void k_pose_adam(float* cam, const float* d_cam, float* m, float* v, int* step, float lr_q, float lr_t, float b1, float b2,
                            float eps, const float* loss, float* best_loss, float* best_cam, int cand_pre_step) {
    const int i = threadIdx.x;
    const int t_new = step[0] + 1;
    __syncthreads();
    if (i == 0) step[0] = t_new;
    const bool better = best_loss && loss[0] < best_loss[0];
    float p = 0.f, p_old = 0.f;
    if (i < 7) {
        const float t = (float)t_new;
        const float lr = i < 4 ? lr_q : lr_t;
        const float step_size = lr / (1.0f - powf(b1, t)), isb = 1.0f / sqrtf(1.0f - powf(b2, t));
        float mm = m[i], vv = v[i];
        p_old = cam[i];
        p = adam_update(p_old, d_cam[i], mm, vv, b1, b2, step_size, isb, eps);
        m[i] = mm; v[i] = vv; cam[i] = p;
    }
    __syncthreads();
    if (better) {
        if (i < 7) best_cam[i] = cand_pre_step ? p_old : p;
        if (i == 0) best_loss[0] = loss[0];
    }
}

}  // namespace psl

using namespace psl;

static inline unsigned nblk(long long n, int tb) { return (unsigned)((n + tb - 1) / tb); }

extern "C" int psl_sample_rays(const int64_t* pix, int32_t n_frames, int32_t per_frame, int32_t H, int32_t W, int32_t H0,
                               int32_t W0, int32_t win_w, const float* cam, const float* c2w, const float* color,
                               const float* depth, const double* dyn_radius, float fx, float fy, float cx, float cy,
                               float* rays_o, float* rays_d, float* b_depth, float* b_color, double* r2, psl_stream_t stream) {
    PSL_REQUIRE(pix && color && depth && rays_o && rays_d && b_depth && b_color, "NULL argument");
    PSL_REQUIRE((cam != nullptr) != (c2w != nullptr), "exactly one of cam / c2w");
    PSL_REQUIRE(!cam || n_frames == 1, "a [quat,T] pose describes one frame");
    PSL_REQUIRE((r2 == nullptr) == (dyn_radius == nullptr), "r2 and dyn_radius go together");
    PSL_REQUIRE(win_w > 0 && H0 >= 0 && W0 >= 0 && W0 + win_w <= W, "bad sampling window");
    const long long n = (long long)n_frames * per_frame;
    if (n == 0) return 0;
    SampleArgs a{reinterpret_cast<const long long*>(pix), n_frames, per_frame, H, W, H0, W0, win_w, cam, c2w, color, depth, dyn_radius,
                 fx, fy, cx, cy, rays_o, rays_d, b_depth, b_color, r2};
    TimingScope ts(T_SHELL, as_stream(stream));
    k_sample_rays<<<nblk(n, 128), 128, 0, as_stream(stream)>>>(a);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int psl_depth_gate(const float* b_depth, int32_t n, float* depth_in, uint8_t* inside, psl_stream_t stream) {
    PSL_REQUIRE(b_depth && depth_in && inside, "NULL argument");
    PSL_REQUIRE(n >= 0 && n <= GATE_MAX, "psl_depth_gate handles at most 8192 rays per call");
    if (n == 0) return 0;
    TimingScope ts(T_SHELL, as_stream(stream));
    k_depth_gate<<<1, 1024, 0, as_stream(stream)>>>(b_depth, n, depth_in, inside);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int psl_shell_loss(int32_t mode, int32_t n, const float* depth_in, const uint8_t* inside, const uint8_t* ray_mask,
                              const float* depth, const float* var, const float* rgb, const float* b_color, float w_color,
                              float* loss, float* d_depth, float* d_rgb, psl_stream_t stream) {
    PSL_REQUIRE(depth_in && inside && depth && loss && d_depth, "NULL argument");
    PSL_REQUIRE(mode == 0 || mode == 1, "mode: 0 tracking, 1 mapping");
    PSL_REQUIRE(mode == 1 || var, "tracking loss needs the depth variance");
    PSL_REQUIRE(mode == 0 || ray_mask, "mapping loss needs the ray mask");
    PSL_REQUIRE(!d_rgb || (rgb && b_color), "colour term needs rgb and b_color");
    TimingScope ts(T_SHELL, as_stream(stream));
    k_shell_loss<<<1, 1024, 0, as_stream(stream)>>>(mode, n, depth_in, inside, ray_mask, depth, var, rgb, b_color, w_color, loss,
                                                   d_depth, d_rgb);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" size_t psl_render_tail_ws_bytes(int32_t n) { return 16 + sizeof(float2) * (size_t)((n + 127) / 128); }

extern "C" int psl_render_tail(int32_t mode, int32_t n, int32_t n_samples, float coef, int32_t min_count, const float* raw,
                               const uint8_t* has_nb, const float* z_vals, const float* depth_in, const uint8_t* inside,
                               const float* b_color, float w_color, float* depth, float* var, float* rgb, uint8_t* ray_mask,
                               float* loss, float* d_raw, void* ws, size_t ws_bytes, psl_stream_t stream) {
    PSL_REQUIRE(raw && has_nb && z_vals && depth_in && inside && depth && var && rgb && ray_mask && loss && d_raw, "NULL argument");
    PSL_REQUIRE(mode == 0 || mode == 1, "mode: 0 tracking, 1 mapping");
    PSL_REQUIRE(n >= 1, "no rays");
    PSL_REQUIRE(n_samples >= 1 && n_samples <= MAX_S, "n_samples > 64 not supported by the composite backward");
    TimingScope ts(T_SHELL, as_stream(stream));
    if (mode == 1) {
        const unsigned nb = (unsigned)((n + 127) / 128);
        PSL_REQUIRE(ws && ws_bytes >= psl_render_tail_ws_bytes(n), "mapping mode needs the zero-initialised workspace");
        unsigned* ticket = static_cast<unsigned*>(ws);
        float2* partial = reinterpret_cast<float2*>(static_cast<unsigned char*>(ws) + 16);
        k_render_tail_map<<<nb, 128, 0, as_stream(stream)>>>(n, n_samples, coef, min_count, reinterpret_cast<const float4*>(raw), has_nb,
                                                           z_vals, depth_in, inside, b_color, w_color, depth, var, rgb, ray_mask, loss,
                                                           reinterpret_cast<float4*>(d_raw), partial, ticket);
    } else {
        k_render_tail<<<1, 1024, 0, as_stream(stream)>>>(mode, n, n_samples, coef, min_count, reinterpret_cast<const float4*>(raw), has_nb,
                                                        z_vals, depth_in, inside, b_color, w_color, depth, var, rgb, ray_mask, loss,
                                                        reinterpret_cast<float4*>(d_raw));
    }
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int psl_pose_bwd(const int64_t* pix, int32_t n, int32_t H0, int32_t W0, int32_t win_w, float fx, float fy, float cx,
                            float cy, const float* cam, const float* d_rays_o, const float* d_rays_d, float* d_cam,
                            psl_stream_t stream) {
    PSL_REQUIRE(pix && cam && d_rays_o && d_rays_d && d_cam, "NULL argument");
    PSL_REQUIRE(win_w > 0, "bad sampling window");
    TimingScope ts(T_SHELL, as_stream(stream));
    k_pose_bwd<<<1, 1024, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(pix), n, H0, W0, win_w, fx, fy, cx, cy, cam,
                                                 d_rays_o, d_rays_d, d_cam);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int psl_adam_rows(float* param, float* grad, float* exp_avg, float* exp_avg_sq, const int64_t* rows, int64_t n_slots,
                             int32_t width, int32_t* step, float lr, float beta1, float beta2, float eps, int32_t zero_grad,
                             psl_stream_t stream) {
    PSL_REQUIRE(param && grad && exp_avg && exp_avg_sq && step, "NULL argument");
    PSL_REQUIRE(width > 0 && n_slots >= 0, "bad shape");
    if (n_slots == 0) return 0;
    cudaStream_t st = as_stream(stream);
    TimingScope ts(T_SHELL, st, 2);
    k_adam_tick<<<1, 1, 0, st>>>(step);
    AdamArgs a{param, grad, exp_avg, exp_avg_sq, reinterpret_cast<const long long*>(rows), n_slots, width, step, lr, beta1, beta2, eps,
               zero_grad};
    const bool vec = width % 4 == 0 && ((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) |
                                         reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0;
    const unsigned cap = (unsigned)sm_count() * 8u;                      // one resident wave; the kernel strides over the rest
    const unsigned nb = vec ? nblk(n_slots * (width / 4), 256) : nblk(n_slots * width, 256);
    if (vec) k_adam_rows<4><<<nb < cap ? nb : cap, 256, 0, st>>>(a);
    else k_adam_rows<1><<<nb < cap ? nb : cap, 256, 0, st>>>(a);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int psl_pose_adam(float* cam, const float* d_cam, float* exp_avg, float* exp_avg_sq, int32_t* step, float lr_quat, float lr_trans,
                             float beta1, float beta2, float eps, const float* loss, float* best_loss, float* best_cam,
                             int32_t candidate_pre_step, psl_stream_t stream) {
    PSL_REQUIRE(cam && d_cam && exp_avg && exp_avg_sq && step, "NULL argument");
    PSL_REQUIRE(!best_loss || (loss && best_cam), "candidate bookkeeping needs loss and best_cam");
    TimingScope ts(T_SHELL, as_stream(stream));
    k_pose_adam<<<1, 32, 0, as_stream(stream)>>>(cam, d_cam, exp_avg, exp_avg_sq, step, lr_quat, lr_trans, beta1, beta2, eps, loss,
                                                 best_loss, best_cam, candidate_pre_step);
    PSL_CHECK_CUDA(cudaGetLastError());
    return 0;
}
