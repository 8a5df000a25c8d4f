// pcl_volumes.cu -- points to volumes: splat point features into voxel grids (forward + backward) for sm_100a.
//
// Replaces pytorch3d.ops.add_points_features_to_volume_densities_features (0.7.2, restated from memory: parity with pytorch3d
// itself is unpinned; the contract is in include/pcl.h, and tests/volumes_ref.py is the specification).
//
// Forward: a scatter.  Thread (i, g) of cloud b handles point i and the P2V_CPT consecutive "channels" g*P2V_CPT.. of the
// C + 1 the point votes with (channel 0 is the density, channel 1 + c is feature c).  It recomputes the point's lattice
// coordinate and its 8 (trilinear) or 1 (nearest) corner weights and adds w * value with one fp32 reduction (red.global.add,
// which flushes subnormals) per in-bounds corner of nonzero weight and channel, straight into the channel-major outputs.
// The order of the reductions is not fixed, so the forward is not bit-reproducible.
//
// Backward: a gather, one thread per point, no atomics and a fixed summation order: bit-reproducible and independent of the
// rest of the batch.
#include <cmath>

#include "pcl_common.cuh"

namespace pcl {
namespace {

constexpr int P2V_THREADS = 128;
constexpr int P2V_CPT = 4;            // channels (density + features) per forward thread
constexpr int P2V_MAX_DIM = 1 << 24;  // padded D, H, W: every index is exact in fp32, so the bounds test can run in float

struct Grid {
    const int64_t *sizes;  // nullable (B, 3): D_b, H_b, W_b
    int D, H, W, s, o;     // padded sizes; (s, o) = (1, 0) with align_corners, (0, 1) without
};

// lattice coordinate of axis value p for a grid of S voxels, in fp32 with every operation rounded (no contraction):
// t = ((p + 1) * (S - s) - o) * 0.5
__device__ __forceinline__ float lattice(float p, float Sms, int o) {
    return __fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(p, 1.f), Sms), (float)o), 0.5f);
}

// One point's geometry: per axis (0 = x/W, 1 = y/H, 2 = z/D) the base index f, the fraction r, the bound and (S - s).
struct Cell {
    float f[3], r[3], lim[3], sms[3];
};

__device__ __forceinline__ void cell_of(const Pts &pts, const Grid &g, int b, int i, bool trilinear, Cell &c) {
    const int64_t o = (int64_t)b * pts.bs + (int64_t)i * pts.rs;
    const int pad[3] = {g.W, g.H, g.D};
#pragma unroll
    for (int a = 0; a < 3; a++) {
        // grid_sizes holds (D, H, W): axis a reads entry 2 - a
        const int64_t S = g.sizes ? g.sizes[(int64_t)b * 3 + 2 - a] : (int64_t)pad[a];
        const int64_t lim = S < (int64_t)pad[a] ? S : (int64_t)pad[a];
        c.lim[a] = (float)(lim < 0 ? 0 : lim);
        c.sms[a] = (float)(S - g.s);
        const float t = lattice(ld_any(pts, o + a), c.sms[a], g.o);
        c.f[a] = trilinear ? floorf(t) : roundf(t);  // roundf: half away from zero
        c.r[a] = __fsub_rn(t, c.f[a]);
    }
}

// in bounds: 0 <= v < lim, tested in float (NaN and +-inf fail), so a huge coordinate never reaches an integer conversion
__device__ __forceinline__ bool inside(float v, float lim) { return v >= 0.f && v < lim; }

__global__ void __launch_bounds__(P2V_THREADS)
p2v_fwd_kernel(Pts pts, Pts feat, const float *__restrict__ mask, Grid g, int P, int C, int trilinear,
               float *__restrict__ dens, float *__restrict__ vfeat) {
    const int i = blockIdx.x * P2V_THREADS + threadIdx.x;
    const int b = blockIdx.z;
    if (i >= P) return;
    const float m = mask ? __ldg(mask + (int64_t)b * P + i) : 1.f;
    if (m == 0.f) return;
    Cell c;
    cell_of(pts, g, b, i, trilinear, c);
    const int c0 = blockIdx.y * P2V_CPT, c1 = min(c0 + P2V_CPT, C + 1);
    float val[P2V_CPT];
    const int64_t fo = (int64_t)b * feat.bs + (int64_t)i * feat.rs;
#pragma unroll
    for (int k = 0; k < P2V_CPT; k++) val[k] = (c0 + k == 0) ? 1.f : (c0 + k < c1 ? ld_any(feat, fo + c0 + k - 1) : 0.f);
    const int64_t vox = (int64_t)g.D * g.H * g.W;
    const int ncorner = trilinear ? 8 : 1;
    for (int k = 0; k < ncorner; k++) {
        const int dx = k & 1, dy = (k >> 1) & 1, dz = k >> 2;
        const float x = c.f[0] + dx, y = c.f[1] + dy, z = c.f[2] + dz;
        if (!inside(x, c.lim[0]) || !inside(y, c.lim[1]) || !inside(z, c.lim[2])) continue;
        float w = m;
        if (trilinear) {
            const float wx = dx ? c.r[0] : __fsub_rn(1.f, c.r[0]);
            const float wy = dy ? c.r[1] : __fsub_rn(1.f, c.r[1]);
            const float wz = dz ? c.r[2] : __fsub_rn(1.f, c.r[2]);
            w = __fmul_rn(m, __fmul_rn(__fmul_rn(wz, wy), wx));
        }
        if (w == 0.f) continue;
        const int64_t v = ((int64_t)z * g.H + (int64_t)y) * g.W + (int64_t)x;
#pragma unroll
        for (int q = 0; q < P2V_CPT; q++) {
            const int ch = c0 + q;
            if (ch >= c1) break;
            if (ch == 0) atomicAdd(dens + (int64_t)b * vox + v, w);
            else atomicAdd(vfeat + ((int64_t)b * C + (ch - 1)) * vox + v, __fmul_rn(w, val[q]));
        }
    }
}

// One thread per point.  Corner k's voxel v_k, weight w_k = m prod_axes (d ? r : 1 - r) and, trilinear only,
//   grad_point_features[c] = sum_k w_k gf[c, v_k]                                  (k ascending)
//   grad_points[a] = (S_a - s) / 2 * sum_k dw_k/dt_a (gd[v_k] + sum_c f[c] gf[c, v_k])   (c ascending, then k ascending)
// in fp32.  Nearest: grad_point_features[c] = m gf[c, v], grad_points = 0.  Points with m == 0 get zeros.
__global__ void __launch_bounds__(P2V_THREADS)
p2v_bwd_kernel(Pts pts, Pts feat, const float *__restrict__ mask, Grid g, int P, int C, int trilinear,
               const float *__restrict__ gdens, const float *__restrict__ gfeat, float *__restrict__ gpts,
               float *__restrict__ gpf) {
    const int i = blockIdx.x * P2V_THREADS + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= P) return;
    const int64_t row = (int64_t)b * P + i;
    const float m = mask ? __ldg(mask + row) : 1.f;
    Cell c;
    if (m != 0.f) cell_of(pts, g, b, i, trilinear, c);
    const int64_t vox = (int64_t)g.D * g.H * g.W;
    // corner k's voxel offset, or -1 when it is out of bounds (every corner is when m == 0)
    int64_t off[8];
    float w[8];
    const int ncorner = trilinear ? 8 : 1;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        off[k] = -1;
        w[k] = 0.f;
        if (k >= ncorner || m == 0.f) continue;
        const int dx = k & 1, dy = (k >> 1) & 1, dz = k >> 2;
        const float x = c.f[0] + dx, y = c.f[1] + dy, z = c.f[2] + dz;
        if (!inside(x, c.lim[0]) || !inside(y, c.lim[1]) || !inside(z, c.lim[2])) continue;
        off[k] = ((int64_t)z * g.H + (int64_t)y) * g.W + (int64_t)x;
        w[k] = m;
        if (trilinear) {
            const float wx = dx ? c.r[0] : __fsub_rn(1.f, c.r[0]);
            const float wy = dy ? c.r[1] : __fsub_rn(1.f, c.r[1]);
            const float wz = dz ? c.r[2] : __fsub_rn(1.f, c.r[2]);
            w[k] = __fmul_rn(m, __fmul_rn(__fmul_rn(wz, wy), wx));
        }
    }
    const bool want_pts = gpts && trilinear;
    float acc[8];  // gd[v_k] + sum_c f[c] gf[c, v_k]
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = (want_pts && gdens && off[k] >= 0) ? __ldg(gdens + b * vox + off[k]) : 0.f;
    if (gfeat && (gpf || want_pts)) {
        const int64_t fo = (int64_t)b * feat.bs + (int64_t)i * feat.rs;
        for (int ch = 0; ch < C; ch++) {
            const float *gch = gfeat + ((int64_t)b * C + ch) * vox;
            const float fv = want_pts ? ld_any(feat, fo + ch) : 0.f;
            float s = 0.f;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (off[k] < 0) continue;
                const float gv = __ldg(gch + off[k]);
                s = __fadd_rn(s, __fmul_rn(w[k], gv));
                if (want_pts) acc[k] = __fadd_rn(acc[k], __fmul_rn(fv, gv));
            }
            if (gpf) gpf[row * C + ch] = s;
        }
    } else if (gpf) {
        for (int ch = 0; ch < C; ch++) gpf[row * C + ch] = 0.f;
    }
    if (!gpts) return;
    float gp[3] = {0.f, 0.f, 0.f};
    if (want_pts && m != 0.f) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            if (off[k] < 0) continue;
            const int d[3] = {k & 1, (k >> 1) & 1, k >> 2};
            float wa[3];
#pragma unroll
            for (int a = 0; a < 3; a++) wa[a] = d[a] ? c.r[a] : __fsub_rn(1.f, c.r[a]);
            // dw/dt_a = m * (+-1) * product of the other two axes' weights
            const float dwx = __fmul_rn(m, __fmul_rn(wa[2], wa[1]));
            const float dwy = __fmul_rn(m, __fmul_rn(wa[2], wa[0]));
            const float dwz = __fmul_rn(m, __fmul_rn(wa[1], wa[0]));
            gp[0] = __fadd_rn(gp[0], __fmul_rn(d[0] ? dwx : -dwx, acc[k]));
            gp[1] = __fadd_rn(gp[1], __fmul_rn(d[1] ? dwy : -dwy, acc[k]));
            gp[2] = __fadd_rn(gp[2], __fmul_rn(d[2] ? dwz : -dwz, acc[k]));
        }
#pragma unroll
        for (int a = 0; a < 3; a++) gp[a] = __fmul_rn(gp[a], __fmul_rn(c.sms[a], 0.5f));
    }
#pragma unroll
    for (int a = 0; a < 3; a++) gpts[row * 3 + a] = gp[a];
}

int check_args(const char *who, const void *points, int p_dtype, const void *features, int f_dtype, int B, int P, int C, int D,
               int H, int W, int mode, int align_corners) {
    if (B < 0 || P < 0 || D < 0 || H < 0 || W < 0) {
        set_error("%s: negative size B=%d P=%d D=%d H=%d W=%d", who, B, P, D, H, W);
        return PCL_E_SHAPE;
    }
    if (C < 1) { set_error("%s: C=%d must be at least 1", who, C); return PCL_E_SHAPE; }
    if (B > 65535) { set_error("%s: B=%d > 65535", who, B); return PCL_E_SHAPE; }
    if (D > P2V_MAX_DIM || H > P2V_MAX_DIM || W > P2V_MAX_DIM) {
        set_error("%s: grid %d x %d x %d: each size must be at most 2^24", who, D, H, W);
        return PCL_E_SHAPE;
    }
    if ((C + 1 + P2V_CPT - 1) / P2V_CPT > 65535) { set_error("%s: C=%d too large", who, C); return PCL_E_SHAPE; }
    if (mode != PCL_P2V_TRILINEAR && mode != PCL_P2V_NEAREST) { set_error("%s: bad mode %d", who, mode); return PCL_E_ARG; }
    if (align_corners != 0 && align_corners != 1) { set_error("%s: bad align_corners %d", who, align_corners); return PCL_E_ARG; }
    if (!dtype_ok(p_dtype) || !dtype_ok(f_dtype)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B > 0 && P > 0 && (!points || !features)) { set_error("%s: null input", who); return PCL_E_ARG; }
    return PCL_OK;
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_points_to_volumes_fwd(const void *points, int p_dtype, int64_t p_bs, int64_t p_rs, const void *features,
                                         int f_dtype, int64_t f_bs, int64_t f_rs, const float *mask, const int64_t *grid_sizes,
                                         int B, int P, int C, int D, int H, int W, int mode, int align_corners,
                                         float *volume_densities, float *volume_features, void *stream) {
    int rc = check_args("points_to_volumes", points, p_dtype, features, f_dtype, B, P, C, D, H, W, mode, align_corners);
    if (rc) return rc;
    const bool empty = B == 0 || P == 0 || D == 0 || H == 0 || W == 0;
    if (!empty && (!volume_densities || !volume_features)) { set_error("points_to_volumes: null output"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (empty) return PCL_OK;
    const Pts a{points, p_bs, p_rs, p_dtype}, f{features, f_bs, f_rs, f_dtype};
    const Grid g{grid_sizes, D, H, W, align_corners ? 1 : 0, align_corners ? 0 : 1};
    const dim3 grid((P + P2V_THREADS - 1) / P2V_THREADS, (C + 1 + P2V_CPT - 1) / P2V_CPT, B);
    p2v_fwd_kernel<<<grid, P2V_THREADS, 0, (cudaStream_t)stream>>>(a, f, mask, g, P, C, mode == PCL_P2V_TRILINEAR,
                                                                    volume_densities, volume_features);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_points_to_volumes_bwd(const void *points, int p_dtype, int64_t p_bs, int64_t p_rs, const void *features,
                                         int f_dtype, int64_t f_bs, int64_t f_rs, const float *mask, const int64_t *grid_sizes,
                                         int B, int P, int C, int D, int H, int W, int mode, int align_corners,
                                         const float *grad_densities, const float *grad_features, float *grad_points,
                                         float *grad_point_features, void *stream) {
    int rc = check_args("points_to_volumes_bwd", points, p_dtype, features, f_dtype, B, P, C, D, H, W, mode, align_corners);
    if (rc) return rc;
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P == 0 || (!grad_points && !grad_point_features)) return PCL_OK;
    const Pts a{points, p_bs, p_rs, p_dtype}, f{features, f_bs, f_rs, f_dtype};
    const Grid g{grid_sizes, D, H, W, align_corners ? 1 : 0, align_corners ? 0 : 1};
    p2v_bwd_kernel<<<dim3((P + P2V_THREADS - 1) / P2V_THREADS, B), P2V_THREADS, 0, (cudaStream_t)stream>>>(
        a, f, mask, g, P, C, mode == PCL_P2V_TRILINEAR, grad_densities, grad_features, grad_points, grad_point_features);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
