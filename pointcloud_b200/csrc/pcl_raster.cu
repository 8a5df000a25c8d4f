// pcl_raster.cu -- rasterize points and the point compositors (forward + backward) for sm_100a.
//
// Replaces pytorch3d.renderer.points.rasterize_points and pytorch3d.renderer.compositing's alpha_composite /
// norm_weighted_sum / weighted_sum (0.7.2, restated from memory: parity with pytorch3d itself is unpinned; the contract is
// in include/pcl.h, and tests/raster_ref.py is the specification).
//
// Rasterizer forward.  A pixel keeps the K hitting points of smallest key (bits(z + 0) << 32) | i: z >= 0 is finite, so
// the bit order of z is its float order, and the key is a total order -- the result does not depend on the order in which
// points are visited.  A CTA owns a block of 16 x TH pixels (one thread per pixel) and stages candidate points through
// shared memory, 16 * TH per round, dropping every point whose conservative pixel box (point_box) misses the block; each
// thread then tests the staged points and inserts hits into its sorted list (registers for K <= 8, shared memory above).
//   naive   (bin_size == 0): the candidates are the whole cloud.  One launch.
//   binned  (bin_size  > 0): a coarse pass appends every point to each (cloud, bin) whose pixels its box reaches, up to
//           `cap` entries (the count keeps counting); the fine pass reads its bin's list, or -- when the bin overflowed --
//           the whole cloud.  Overflow costs time, never correctness, and nothing is read back to the host.  A memset of
//           the counts and two launches.
// Rasterizer backward: one thread per (pixel, slot), fp32 red.add onto the zero-filled grad_points.
//
// Compositors: forward one thread per (pixel, group of 4 channels), sums in slot order (bit-reproducible); backward one
// thread per pixel writes grad_alphas without atomics and adds grad_features with red.add.
#include <cmath>

#include "pcl_common.cuh"

namespace pcl {
namespace {

constexpr int RAST_MAX_K = 150;         // pytorch3d's kMaxPointsPerPixel
constexpr int RAST_MAX_SIZE = 16384;    // H, W
constexpr int RAST_TW = 16;             // fine-pass block width in pixels; bin_size must be a multiple of it
constexpr int RAST_REG_K = 8;           // K <= 8: the per-pixel list lives in registers, 256 pixels per CTA
constexpr int RAST_LIST_BYTES = 40960;  // K > 8: shared-memory lists of 128 / 64 / 32 pixels per CTA, at most this size
constexpr int COARSE_THREADS = 256;
constexpr int BWD_THREADS = 256;
constexpr int COMP_THREADS = 128;
constexpr int COMP_CG = 4;              // channels per compositor forward thread
constexpr unsigned long long EMPTY = ~0ull;

// fp32 pixel centre of index i along an axis of S1 pixels (the other axis has S2), every operation rounded:
// -off + (range * i + off) / S1, range = S1 > S2 ? (S1 * 2) / S2 : 2, off = range / 2.  Column c uses i = W - 1 - c,
// row r uses i = H - 1 - r.
__device__ __forceinline__ float ndc(int i, int S1, int S2) {
    const float range = S1 > S2 ? __fdiv_rn((float)(S1 * 2), (float)S2) : 2.f;
    const float off = __fmul_rn(range, 0.5f);
    return __fadd_rn(-off, __fdiv_rn(__fadd_rn(__fmul_rn(range, (float)i), off), (float)S1));
}

struct RPoint {
    float x, y, z, r2;
    bool ok;  // finite x, y, z, r and z >= 0
    float r;
};

__device__ __forceinline__ RPoint load_point(const Pts &pts, const float *radius, float rscalar, int b, int i, int P) {
    const float3 p = ld_xyz(pts, b, i);
    const float r = radius ? __ldg(radius + (int64_t)b * P + i) : rscalar;
    RPoint q;
    q.x = p.x; q.y = p.y; q.z = p.z; q.r = r;
    q.r2 = __fmul_rn(r, r);
    q.ok = isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && isfinite(r) && p.z >= 0.f;
    return q;
}

// The indices i of an axis (S1 pixels, the other S2) whose fp32 centre x_i can satisfy fl(fl(x_i - p)^2) <= fl(r^2):
// [lo, hi], empty when lo > hi.  Conservative: such a centre has |x_i - p| <= |r| (1 + 2.1 * 2^-24) (or r^2 overflowed:
// every pixel), the half-width R below exceeds that, the fp32 centres are within far less than a pixel of the exact
// -off + (range * i + off) / S1 (S1 <= 16384), whose inverse is i = (x + off) * min(S1, S2) / 2 - 1/2, and the range is
// widened by one pixel each way.  Everything is in double (off = S1 / S2 through a reciprocal: its relative error of
// 2^-52 moves i by far less than the slack) and clamped to [-1, S1] before the conversion, so huge coordinates and radii
// give in-range indices.  No division, so no call into a division slow path.
__device__ __forceinline__ void axis_box(float p, const RPoint &q, int S1, int S2, int &lo, int &hi) {
    const double off = S1 > S2 ? (double)S1 * __drcp_rn((double)S2) : 1.0, half = 0.5 * (S1 < S2 ? S1 : S2);
    const double R = isinf(q.r2) ? (double)INFINITY : fabs((double)q.r) * (1.0 + 0x1p-20) + 0x1p-60;
    double a = ((double)p - R + off) * half - 1.5;
    double z = ((double)p + R + off) * half + 0.5;
    a = fmin(fmax(a, -1.0), (double)S1);
    z = fmin(fmax(z, -1.0), (double)S1);
    lo = max((int)ceil(a), 0);
    hi = min((int)floor(z), S1 - 1);
}

// column range [c0, c1] and row range [r0, r1] a valid point may reach
__device__ __forceinline__ void point_box(const RPoint &q, int H, int W, int &c0, int &c1, int &r0, int &r1) {
    int lo, hi;
    axis_box(q.x, q, W, H, lo, hi);
    c0 = W - 1 - hi; c1 = W - 1 - lo;
    axis_box(q.y, q, H, W, lo, hi);
    r0 = H - 1 - hi; r1 = H - 1 - lo;
}

// sum of the clamped lengths of clouds 0..b-1 (b * P without lengths), by one warp
__device__ __forceinline__ int64_t warp_cloud_offset(const int64_t *len, int b, int P) {
    if (!len) return (int64_t)b * P;
    int64_t s = 0;
    for (int j = (int)(threadIdx.x & 31); j < b; j += 32) s += len_of(len, j, P);
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

__global__ void __launch_bounds__(COARSE_THREADS)
raster_coarse_kernel(Pts pts, const int64_t *__restrict__ len, const float *__restrict__ radius, float rscalar, int P, int H,
                     int W, int bin_size, int nbx, int nbins, int cap, int32_t *__restrict__ counts, int32_t *__restrict__ bins) {
    const int i = blockIdx.x * COARSE_THREADS + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= len_of(len, b, P)) return;
    const RPoint q = load_point(pts, radius, rscalar, b, i, P);
    if (!q.ok) return;
    int c0, c1, r0, r1;
    point_box(q, H, W, c0, c1, r0, r1);
    if (c0 > c1 || r0 > r1) return;
    for (int by = r0 / bin_size; by <= r1 / bin_size; by++)
        for (int bx = c0 / bin_size; bx <= c1 / bin_size; bx++) {
            const int64_t bin = (int64_t)b * nbins + by * nbx + bx;
            const int slot = atomicAdd(counts + bin, 1);
            if (slot < cap) bins[bin * cap + slot] = i;
        }
}

// KR = 1 or 8: the list in registers (K <= KR), 256 pixels per CTA.  KR = 0: the list in dynamic shared memory,
// keys[k * PIX + t], K <= 150.
template <int KR>
__global__ void __launch_bounds__(256)
raster_fine_kernel(Pts pts, const int64_t *__restrict__ len, const float *__restrict__ radius, float rscalar, int P, int H,
                   int W, int K, int bin_size, int nbx, int nbins, int cap, const int32_t *__restrict__ counts,
                   const int32_t *__restrict__ bins, int32_t *__restrict__ out_idx, float *__restrict__ out_z,
                   float *__restrict__ out_d) {
    extern __shared__ unsigned long long s_list[];
    __shared__ float4 s_pt[256];
    __shared__ int s_i[256];
    __shared__ int s_n;
    __shared__ int64_t s_off;
    const int PIX = blockDim.x, TH = PIX / RAST_TW, t = threadIdx.x;
    const int b = blockIdx.z;
    const int bc0 = blockIdx.x * RAST_TW, br0 = blockIdx.y * TH;
    const int bc1 = min(bc0 + RAST_TW, W) - 1, br1 = min(br0 + TH, H) - 1;
    const int c = bc0 + t % RAST_TW, r = br0 + t / RAST_TW;
    // the centres first: their IEEE divisions may call a slow path, and nothing else is live yet
    const float xf = ndc(W - 1 - c, W, H), yf = ndc(H - 1 - r, H, W);
    const int n = len_of(len, b, P);
    if (t < 32) {
        const int64_t o = warp_cloud_offset(len, b, P);
        if (t == 0) s_off = o;
    }
    __syncthreads();
    const int32_t *list = nullptr;
    int total = n;
    if (bins) {
        const int64_t bin = (int64_t)b * nbins + (br0 / bin_size) * nbx + bc0 / bin_size;
        const int cnt = __ldg(counts + bin);
        if (cnt <= cap) { list = bins + bin * cap; total = cnt; }
    }
    unsigned long long reg[KR > 0 ? KR : 1];
#pragma unroll
    for (int k = 0; k < (KR > 0 ? KR : 1); k++) reg[k] = EMPTY;
    unsigned long long worst = EMPTY;  // the K-th key once the list is full
    int m = 0;                         // KR = 0: entries in the list
    for (int base = 0; base < total; base += PIX) {
        if (t == 0) s_n = 0;
        __syncthreads();
        const int j = base + t;
        if (j < total) {
            const int i = list ? __ldg(list + j) : j;
            const RPoint q = load_point(pts, radius, rscalar, b, i, P);
            if (q.ok) {
                int c0, c1, r0, r1;
                point_box(q, H, W, c0, c1, r0, r1);
                if (c0 <= bc1 && c1 >= bc0 && r0 <= br1 && r1 >= br0) {
                    const int s = atomicAdd(&s_n, 1);
                    s_pt[s] = make_float4(q.x, q.y, __fadd_rn(q.z, 0.f), q.r2);  // + 0: -0.0 keys as +0.0
                    s_i[s] = i;
                }
            }
        }
        __syncthreads();
        const int ns = s_n;
        for (int s = 0; s < ns; s++) {
            const float4 q = s_pt[s];
            const float dx = __fsub_rn(xf, q.x), dy = __fsub_rn(yf, q.y);
            const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
            if (!(d2 <= q.w)) continue;
            unsigned long long key = ((unsigned long long)__float_as_uint(q.z) << 32) | (unsigned)s_i[s];
            if (key >= worst) continue;
            if constexpr (KR > 0) {
#pragma unroll
                for (int k = 0; k < KR; k++) {
                    const unsigned long long lo = key < reg[k] ? key : reg[k];
                    key = key < reg[k] ? reg[k] : key;
                    reg[k] = lo;
                }
                worst = reg[0];  // reg[K - 1], as a chain of selects (an index would put reg in local memory)
#pragma unroll
                for (int k = 1; k < KR; k++) worst = k < K ? reg[k] : worst;
            } else {
                int p = m < K ? m : K - 1;
                while (p > 0 && s_list[(p - 1) * PIX + t] > key) {
                    s_list[p * PIX + t] = s_list[(p - 1) * PIX + t];
                    p--;
                }
                s_list[p * PIX + t] = key;
                if (m < K) m++;
                if (m == K) worst = s_list[(K - 1) * PIX + t];
            }
        }
        __syncthreads();
    }
    if (r > br1 || c > bc1) return;
    const int64_t o = (((int64_t)b * H + r) * W + c) * K;
    const int64_t off = s_off;
    auto emit = [&](int k, unsigned long long key) {
        if (key == EMPTY) {
            out_idx[o + k] = -1; out_z[o + k] = -1.f; out_d[o + k] = -1.f;
            return;
        }
        const int i = (int)(unsigned)key;
        const float3 p = ld_xyz(pts, b, i);
        const float dx = __fsub_rn(xf, p.x), dy = __fsub_rn(yf, p.y);
        out_idx[o + k] = (int32_t)(off + i);
        out_z[o + k] = p.z;
        out_d[o + k] = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    };
    if constexpr (KR > 0) {
#pragma unroll
        for (int k = 0; k < KR; k++)
            if (k < K) emit(k, reg[k]);
    } else {
        for (int k = 0; k < K; k++) emit(k, k < m ? s_list[k * PIX + t] : EMPTY);
    }
}

// one thread per (pixel, slot) of cloud b = blockIdx.y
__global__ void __launch_bounds__(BWD_THREADS)
raster_bwd_kernel(Pts pts, const int64_t *__restrict__ len, int P, int H, int W, int K, const int32_t *__restrict__ idx,
                  const float *__restrict__ gz, const float *__restrict__ gd, float *__restrict__ grad) {
    __shared__ int64_t s_off;
    const int b = blockIdx.y;
    if (threadIdx.x < 32) {
        const int64_t o = warp_cloud_offset(len, b, P);
        if (threadIdx.x == 0) s_off = o;
    }
    __syncthreads();
    const int64_t HWK = (int64_t)H * W * K;
    const int64_t e = (int64_t)blockIdx.x * BWD_THREADS + threadIdx.x;
    if (e >= HWK) return;
    const int64_t slot = (int64_t)b * HWK + e;
    const int64_t i = (int64_t)__ldg(idx + slot) - s_off;
    if (i < 0 || i >= len_of(len, b, P)) return;  // -1 slots (and anything that is not a point of this cloud)
    float *g = grad + ((int64_t)b * P + i) * 3;
    if (gz) atomicAdd(g + 2, __ldg(gz + slot));
    if (gd) {
        const int pix = (int)(e / K), r = pix / W, c = pix % W;
        const float xf = ndc(W - 1 - c, W, H), yf = ndc(H - 1 - r, H, W);
        const float3 p = ld_xyz(pts, b, i);
        const float g2 = __fmul_rn(2.f, __ldg(gd + slot));
        atomicAdd(g + 0, __fmul_rn(g2, __fsub_rn(p.x, xf)));
        atomicAdd(g + 1, __fmul_rn(g2, __fsub_rn(p.y, yf)));
    }
}

// ------------------------------------------------------------------------------------------------ compositors ---------

struct Idx4 {
    const void *p;
    int i64;
    int64_t s[4];
};
struct F4 {
    const float *p;
    int64_t s[4];
};
struct Feat {
    const float *p;
    int64_t sc, sp, P;  // channel stride, point stride, P_total
};

__device__ __forceinline__ int64_t ld_idx(const Idx4 &a, int n, int k, int h, int w) {
    const int64_t o = n * a.s[0] + k * a.s[1] + h * a.s[2] + w * a.s[3];
    return a.i64 ? __ldg(reinterpret_cast<const long long *>(a.p) + o) : (int64_t)__ldg(reinterpret_cast<const int *>(a.p) + o);
}
__device__ __forceinline__ float ld_a(const F4 &a, int n, int k, int h, int w) {
    return __ldg(a.p + n * a.s[0] + k * a.s[1] + h * a.s[2] + w * a.s[3]);
}
__device__ __forceinline__ float ld_f(const Feat &f, int c, int64_t p) { return __ldg(f.p + c * f.sc + p * f.sp); }

// max(sum of the valid alphas in slot order, 1e-4); a NaN sum stays NaN, as torch.clamp keeps it
__device__ __forceinline__ float norm_weight(const Idx4 &ix, const F4 &al, const Feat &f, int n, int K, int h, int w,
                                             float *sum) {
    float s = 0.f;
    for (int k = 0; k < K; k++) {
        const int64_t id = ld_idx(ix, n, k, h, w);
        if (id >= 0 && id < f.P) s = __fadd_rn(s, ld_a(al, n, k, h, w));
    }
    *sum = s;
    return s < 1e-4f ? 1e-4f : s;
}

__global__ void __launch_bounds__(COMP_THREADS)
composite_fwd_kernel(Idx4 ix, F4 al, Feat f, int K, int H, int W, int C, int mode, float *__restrict__ out) {
    const int pix = blockIdx.x * COMP_THREADS + threadIdx.x;
    if (pix >= H * W) return;
    const int n = blockIdx.z, h = pix / W, w = pix % W, c0 = blockIdx.y * COMP_CG;
    const int nc = min(COMP_CG, C - c0);
    float acc[COMP_CG] = {0.f, 0.f, 0.f, 0.f};
    float s, wn = 1.f, T = 1.f;
    if (mode == PCL_COMPOSITE_NORM_WEIGHTED) wn = norm_weight(ix, al, f, n, K, h, w, &s);
    for (int k = 0; k < K; k++) {
        const int64_t id = ld_idx(ix, n, k, h, w);
        const bool valid = id >= 0 && id < f.P;
        const float a = ld_a(al, n, k, h, w);
        if (valid) {
            const float wa = mode == PCL_COMPOSITE_ALPHA ? __fmul_rn(T, a) : a;
#pragma unroll
            for (int q = 0; q < COMP_CG; q++) {
                if (q >= nc) break;
                float v = __fmul_rn(wa, ld_f(f, c0 + q, id));
                if (mode == PCL_COMPOSITE_NORM_WEIGHTED) v = __fdiv_rn(v, wn);
                acc[q] = __fadd_rn(acc[q], v);
            }
        }
        if (mode == PCL_COMPOSITE_ALPHA) T = __fmul_rn(T, __fsub_rn(1.f, a));
    }
    const int64_t o = ((int64_t)n * C + c0) * H * W + pix;
#pragma unroll
    for (int q = 0; q < COMP_CG; q++)
        if (q < nc) out[o + (int64_t)q * H * W] = acc[q];
}

// One thread per pixel.  e_k = sum_c g_c F[c, id_k] (0 for an invalid slot).
//   weighted:      ga_k = e_k;                                   gF[c, id_k] += g_c a_k
//   norm weighted: ga_k = (e_k - [S >= 1e-4] sum_c g_c out_c) / w;  gF[c, id_k] += g_c a_k / w
//   alpha:         ga_j = T_j (e_j - R_j), R_j = sum_{k>j} prod_{j<t<k} (1 - a_t) a_k e_k (no division by 1 - a_j);
//                  gF[c, id_j] += g_c T_j a_j.  T_j is parked in ga[j] by a first sweep.
__global__ void __launch_bounds__(COMP_THREADS)
composite_bwd_kernel(Idx4 ix, F4 al, Feat f, int K, int H, int W, int C, int mode, const float *__restrict__ gout,
                     float *__restrict__ ga, float *__restrict__ gf) {
    const int pix = blockIdx.x * COMP_THREADS + threadIdx.x;
    if (pix >= H * W) return;
    const int n = blockIdx.y, h = pix / W, w = pix % W;
    const int64_t HW = (int64_t)H * W;
    const float *g = gout + (int64_t)n * C * HW + pix;
    float *gak = ga ? ga + (int64_t)n * K * HW + pix : nullptr;
    auto e_of = [&](int64_t id) {
        float e = 0.f;
        for (int c = 0; c < C; c++) e = __fadd_rn(e, __fmul_rn(__ldg(g + c * HW), ld_f(f, c, id)));
        return e;
    };
    auto add_f = [&](int64_t id, float s) {
        if (!gf) return;
        for (int c = 0; c < C; c++) atomicAdd(gf + c * f.P + id, __fmul_rn(__ldg(g + c * HW), s));
    };
    if (mode == PCL_COMPOSITE_WEIGHTED) {
        for (int k = 0; k < K; k++) {
            const int64_t id = ld_idx(ix, n, k, h, w);
            const bool valid = id >= 0 && id < f.P;
            const float a = ld_a(al, n, k, h, w);
            if (gak) gak[k * HW] = valid ? e_of(id) : 0.f;
            if (valid) add_f(id, a);
        }
    } else if (mode == PCL_COMPOSITE_NORM_WEIGHTED) {
        float s;
        const float wn = norm_weight(ix, al, f, n, K, h, w, &s);
        float G = 0.f;  // sum_c g_c out_c
        if (gak && s >= 1e-4f) {
            for (int c = 0; c < C; c++) {
                float o = 0.f;
                for (int k = 0; k < K; k++) {
                    const int64_t id = ld_idx(ix, n, k, h, w);
                    if (id >= 0 && id < f.P) o = __fadd_rn(o, __fdiv_rn(__fmul_rn(ld_a(al, n, k, h, w), ld_f(f, c, id)), wn));
                }
                G = __fadd_rn(G, __fmul_rn(__ldg(g + c * HW), o));
            }
        }
        for (int k = 0; k < K; k++) {
            const int64_t id = ld_idx(ix, n, k, h, w);
            const bool valid = id >= 0 && id < f.P;
            if (gak) gak[k * HW] = valid ? __fdiv_rn(__fsub_rn(e_of(id), G), wn) : 0.f;
            if (valid) add_f(id, __fdiv_rn(ld_a(al, n, k, h, w), wn));
        }
    } else {
        if (gak) {
            float T = 1.f;
            for (int k = 0; k < K; k++) {
                gak[k * HW] = T;
                T = __fmul_rn(T, __fsub_rn(1.f, ld_a(al, n, k, h, w)));
            }
        }
        float R = 0.f, T = 1.f;
        if (!gak) {  // gF only: T_j forward
            for (int k = 0; k < K; k++) {
                const int64_t id = ld_idx(ix, n, k, h, w);
                const float a = ld_a(al, n, k, h, w);
                if (id >= 0 && id < f.P) add_f(id, __fmul_rn(T, a));
                T = __fmul_rn(T, __fsub_rn(1.f, a));
            }
            return;
        }
        for (int j = K - 1; j >= 0; j--) {
            const int64_t id = ld_idx(ix, n, j, h, w);
            const bool valid = id >= 0 && id < f.P;
            const float a = ld_a(al, n, j, h, w);
            const float Tj = gak[j * HW];
            const float e = valid ? e_of(id) : 0.f;
            gak[j * HW] = __fmul_rn(Tj, __fsub_rn(e, R));
            if (valid) add_f(id, __fmul_rn(Tj, a));
            R = __fadd_rn(__fmul_rn(a, e), __fmul_rn(__fsub_rn(1.f, a), R));
        }
    }
}

int raster_check(const char *who, const void *points, int dtype, int B, int P, int H, int W, int K) {
    if (B < 0 || P < 0) { set_error("%s: negative size B=%d P=%d", who, B, P); return PCL_E_SHAPE; }
    if ((int64_t)B * P >= (int64_t)1 << 31) { set_error("%s: B*P = %lld must be below 2^31", who, (long long)B * P); return PCL_E_SHAPE; }
    if (B > 65535) { set_error("%s: B=%d > 65535", who, B); return PCL_E_SHAPE; }
    if (H < 1 || H > RAST_MAX_SIZE || W < 1 || W > RAST_MAX_SIZE) {
        set_error("%s: image %d x %d: H and W must be in 1..%d", who, H, W, RAST_MAX_SIZE);
        return PCL_E_SHAPE;
    }
    if (K < 1 || K > RAST_MAX_K) { set_error("%s: K=%d must be in 1..%d", who, K, RAST_MAX_K); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B > 0 && P > 0 && !points) { set_error("%s: null points", who); return PCL_E_ARG; }
    return PCL_OK;
}

int bin_cap(int P, int max_points_per_bin) {
    const int def = P / 5 > 10000 ? P / 5 : 10000;  // pytorch3d's default
    const int cap = max_points_per_bin > 0 ? max_points_per_bin : def;
    return cap < P ? cap : (P > 0 ? P : 1);
}

int composite_check(const char *who, int mode, const void *idx, int idx_i64, const float *alphas, const float *features,
                    int N, int K, int H, int W, int C, int64_t P_total) {
    if (N < 0 || K < 0 || H < 0 || W < 0 || C < 0 || P_total < 0) {
        set_error("%s: negative size N=%d K=%d H=%d W=%d C=%d", who, N, K, H, W, C);
        return PCL_E_SHAPE;
    }
    if (N > 65535 || (C + COMP_CG - 1) / COMP_CG > 65535) { set_error("%s: N=%d or C=%d too large", who, N, C); return PCL_E_SHAPE; }
    if ((int64_t)H * W >= (int64_t)1 << 31) { set_error("%s: H*W too large", who); return PCL_E_SHAPE; }
    if (mode != PCL_COMPOSITE_ALPHA && mode != PCL_COMPOSITE_NORM_WEIGHTED && mode != PCL_COMPOSITE_WEIGHTED) {
        set_error("%s: bad mode %d", who, mode);
        return PCL_E_ARG;
    }
    if (idx_i64 != 0 && idx_i64 != 1) { set_error("%s: bad idx type %d", who, idx_i64); return PCL_E_ARG; }
    const bool work = (int64_t)N * K * H * W > 0;
    if (work && (!idx || !alphas)) { set_error("%s: null input", who); return PCL_E_ARG; }
    if (work && C > 0 && P_total > 0 && !features) { set_error("%s: null features", who); return PCL_E_ARG; }
    return PCL_OK;
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_raster_max_k(void) { return RAST_MAX_K; }

extern "C" size_t pcl_rasterize_points_workspace_bytes(int B, int P, int H, int W, int bin_size, int max_points_per_bin) {
    if (bin_size <= 0 || B <= 0 || H <= 0 || W <= 0) return 0;
    const int64_t nbins = (int64_t)((H + bin_size - 1) / bin_size) * ((W + bin_size - 1) / bin_size);
    return (size_t)B * nbins * (1 + (size_t)bin_cap(P, max_points_per_bin)) * sizeof(int32_t);
}

extern "C" int pcl_rasterize_points_fwd(const void *points, int dtype, int64_t bs, int64_t rs, const int64_t *lengths,
                                        const float *radius, float radius_scalar, int B, int P, int H, int W, int K,
                                        int bin_size, int max_points_per_bin, int32_t *idx, float *zbuf, float *dists,
                                        void *workspace, size_t workspace_bytes, void *stream) {
    int rc = raster_check("rasterize_points", points, dtype, B, P, H, W, K);
    if (rc) return rc;
    if (bin_size < 0 || bin_size % RAST_TW) {
        set_error("rasterize_points: bin_size=%d must be 0 or a positive multiple of %d", bin_size, RAST_TW);
        return PCL_E_ARG;
    }
    if (B > 0 && (!idx || !zbuf || !dists)) { set_error("rasterize_points: null output"); return PCL_E_ARG; }
    const size_t need = pcl_rasterize_points_workspace_bytes(B, P, H, W, bin_size, max_points_per_bin);
    if (workspace_bytes < need || (need && !workspace)) {
        set_error("rasterize_points: workspace %zu < %zu bytes", workspace_bytes, need);
        return PCL_E_WORKSPACE;
    }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0) return PCL_OK;
    const cudaStream_t st = (cudaStream_t)stream;
    const Pts a{points, bs, rs, dtype};
    const int nbx = bin_size ? (W + bin_size - 1) / bin_size : 0, nby = bin_size ? (H + bin_size - 1) / bin_size : 0;
    const int nbins = nbx * nby, cap = bin_cap(P, max_points_per_bin);
    int32_t *counts = nullptr, *bins = nullptr;
    if (bin_size) {
        counts = (int32_t *)workspace;
        bins = counts + (int64_t)B * nbins;
        PCL_CUDA(cudaMemsetAsync(counts, 0, (size_t)B * nbins * sizeof(int32_t), st));
        if (P > 0)
            raster_coarse_kernel<<<dim3((P + COARSE_THREADS - 1) / COARSE_THREADS, B), COARSE_THREADS, 0, st>>>(
                a, lengths, radius, radius_scalar, P, H, W, bin_size, nbx, nbins, cap, counts, bins);
    }
    int pix = 256;
    if (K > RAST_REG_K) pix = K * 128 * 8 <= RAST_LIST_BYTES ? 128 : (K * 64 * 8 <= RAST_LIST_BYTES ? 64 : 32);
    const int th = pix / RAST_TW;
    const dim3 grid((W + RAST_TW - 1) / RAST_TW, (H + th - 1) / th, B);
    if (K == 1)
        raster_fine_kernel<1><<<grid, pix, 0, st>>>(a, lengths, radius, radius_scalar, P, H, W, K, bin_size, nbx, nbins, cap,
                                                     counts, bins, idx, zbuf, dists);
    else if (K <= RAST_REG_K)
        raster_fine_kernel<RAST_REG_K><<<grid, pix, 0, st>>>(a, lengths, radius, radius_scalar, P, H, W, K, bin_size, nbx,
                                                              nbins, cap, counts, bins, idx, zbuf, dists);
    else
        raster_fine_kernel<0><<<grid, pix, (size_t)pix * K * 8, st>>>(a, lengths, radius, radius_scalar, P, H, W, K, bin_size,
                                                                      nbx, nbins, cap, counts, bins, idx, zbuf, dists);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_rasterize_points_bwd(const void *points, int dtype, int64_t bs, int64_t rs, const int64_t *lengths, int B,
                                        int P, int H, int W, int K, const int32_t *idx, const float *grad_zbuf,
                                        const float *grad_dists, float *grad_points, void *stream) {
    int rc = raster_check("rasterize_points_bwd", points, dtype, B, P, H, W, K);
    if (rc) return rc;
    if (B > 0 && P > 0 && (!grad_points || !idx)) { set_error("rasterize_points_bwd: null idx or grad_points"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P == 0) return PCL_OK;
    const cudaStream_t st = (cudaStream_t)stream;
    PCL_CUDA(cudaMemsetAsync(grad_points, 0, (size_t)B * P * 3 * sizeof(float), st));
    if (!grad_zbuf && !grad_dists) return PCL_OK;
    const int64_t HWK = (int64_t)H * W * K;
    const Pts a{points, bs, rs, dtype};
    raster_bwd_kernel<<<dim3((unsigned)((HWK + BWD_THREADS - 1) / BWD_THREADS), B), BWD_THREADS, 0, st>>>(
        a, lengths, P, H, W, K, idx, grad_zbuf, grad_dists, grad_points);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_composite_fwd(int mode, const void *idx, int idx_int64, const int64_t *idx_strides_host,
                                 const float *alphas, const int64_t *alpha_strides_host, const float *features,
                                 const int64_t *feature_strides_host, int N, int K, int H, int W, int C, int64_t P_total,
                                 float *out, void *stream) {
    int rc = composite_check("composite", mode, idx, idx_int64, alphas, features, N, K, H, W, C, P_total);
    if (rc) return rc;
    if ((int64_t)N * C * H * W > 0 && !out) { set_error("composite: null output"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if ((int64_t)N * C * H * W == 0) return PCL_OK;
    const Idx4 ix{idx, idx_int64, {idx_strides_host[0], idx_strides_host[1], idx_strides_host[2], idx_strides_host[3]}};
    const F4 al{alphas, {alpha_strides_host[0], alpha_strides_host[1], alpha_strides_host[2], alpha_strides_host[3]}};
    const Feat f{features, feature_strides_host[0], feature_strides_host[1], P_total};
    const dim3 grid((H * W + COMP_THREADS - 1) / COMP_THREADS, (C + COMP_CG - 1) / COMP_CG, N);
    composite_fwd_kernel<<<grid, COMP_THREADS, 0, (cudaStream_t)stream>>>(ix, al, f, K, H, W, C, mode, out);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_composite_bwd(int mode, const void *idx, int idx_int64, const int64_t *idx_strides_host,
                                 const float *alphas, const int64_t *alpha_strides_host, const float *features,
                                 const int64_t *feature_strides_host, int N, int K, int H, int W, int C, int64_t P_total,
                                 const float *grad_out, float *grad_alphas, float *grad_features, void *stream) {
    int rc = composite_check("composite_bwd", mode, idx, idx_int64, alphas, features, N, K, H, W, C, P_total);
    if (rc) return rc;
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    const cudaStream_t st = (cudaStream_t)stream;
    if (grad_features && (int64_t)C * P_total > 0)
        PCL_CUDA(cudaMemsetAsync(grad_features, 0, (size_t)C * P_total * sizeof(float), st));
    if ((int64_t)N * K * H * W == 0 || (!grad_alphas && !grad_features)) return PCL_OK;
    if (C > 0 && !grad_out) { set_error("composite_bwd: null grad_out"); return PCL_E_ARG; }
    const Idx4 ix{idx, idx_int64, {idx_strides_host[0], idx_strides_host[1], idx_strides_host[2], idx_strides_host[3]}};
    const F4 al{alphas, {alpha_strides_host[0], alpha_strides_host[1], alpha_strides_host[2], alpha_strides_host[3]}};
    const Feat f{features, feature_strides_host[0], feature_strides_host[1], P_total};
    composite_bwd_kernel<<<dim3((H * W + COMP_THREADS - 1) / COMP_THREADS, N), COMP_THREADS, 0, st>>>(
        ix, al, f, K, H, W, C, mode, grad_out, grad_alphas, grad_features);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
