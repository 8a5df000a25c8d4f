// pcl_icp.cu -- weighted similarity alignment (forward + backward) and the whole ICP loop in one launch, for sm_100a.
//
// Replaces pytorch3d.ops.corresponding_points_alignment / iterative_closest_point (0.7.2, restated from memory: parity with
// pytorch3d itself is unpinned; the contract is in include/pcl.h, "points alignment and ICP").  D = 3.
//
// Shared by both entry points, so that ICP's alignment step is bit-identical to pcl_points_alignment_fwd on the same
// correspondences:
//  - the moments: fp64 per block of 32 consecutive points (a warp's xor-butterfly, which gives every lane the same bits),
//    then per cloud the blocks summed lane-strided and by the same butterfly -- no atomics, independent of the grid.  X is
//    shifted by its first point and Y by its first correspondence (in ICP the neighbour of X row 0, found by the cloud's
//    warp), so clouds far from the origin keep their bits and a constant cloud has centred moments of exactly 0;
//  - the solve: a one-sided (Hestenes) Jacobi SVD of the 3 x 3 covariance in fp64.  It acts on M itself, not on M^T M,
//    so the polar factor keeps an error of about 2^-52 sigma_1 / (sigma_i + sigma_j) instead of the squared condition an
//    eigen-decomposition of M^T M would give; U is then made proper by u3 = u1 x u2 (exact for planar, rank-2 clouds);
//  - the transform apply(x; R, T, s) = s (x R) + T in fp32 with the operation order documented in pcl.h.
#include <algorithm>
#include <cmath>

#include "pcl_common.cuh"
#include "pcl_nn.cuh"

namespace pcl {
namespace {

typedef unsigned long long u64;

constexpr int AL_THREADS = 256;           // 8 warps
constexpr int AL_WARPS = AL_THREADS / 32;
constexpr int NMOM = 24;                  // moments of one block / cloud, see point_moments
constexpr int ICP_TILE = 256;             // targets per warp tile in the ICP search
constexpr int SVD_MAX_SWEEPS = 24;        // a 3 x 3 one-sided Jacobi converges in 4-7 sweeps; the cap bounds NaN / inf inputs
constexpr double SVD_TOL = 0x1p-52;       // stop when every column pair has |cos| <= 2^-52
constexpr double RANK_TOL = 0x1p-48;      // u2 from M v2 only when |M v2| (orthogonalised) > 2^-48 sigma_1
constexpr u64 KEY_NONE = ~0ull;

__device__ __forceinline__ float ld_pt(const Pts &a, int64_t i) {  // as pcl_knn.cu: one 32-bit or one 16-bit load
    if (a.dtype == PCL_F32) return __ldg(reinterpret_cast<const float *>(a.p) + i);
    const unsigned short h = __ldg(reinterpret_cast<const unsigned short *>(a.p) + i);
    return (a.dtype == PCL_F16) ? __half2float(__ushort_as_half(h)) : __uint_as_float((unsigned)h << 16);
}

__device__ __forceinline__ void ld3(const Pts &a, int n, int j, float (&x)[3]) {
    const int64_t o = (int64_t)n * a.bs + (int64_t)j * a.rs;
#pragma unroll
    for (int c = 0; c < 3; c++) x[c] = ld_pt(a, o + c);
}

// A similarity transform as the outputs hold it: fp32 R (row-major), T, s.
struct Sim {
    float r[9], t[3], s;
};

// apply(x; R, T, s)_d = fl(fl(s * fl(fl(fl(x0 R0d) + fl(x1 R1d)) + fl(x2 R2d))) + T_d), every step rounded (no contraction)
__device__ __forceinline__ void apply_sim(const Sim &T, const float (&x)[3], float (&o)[3]) {
#pragma unroll
    for (int d = 0; d < 3; d++) {
        float acc = __fmul_rn(x[0], T.r[d]);
        acc = __fadd_rn(acc, __fmul_rn(x[1], T.r[3 + d]));
        acc = __fadd_rn(acc, __fmul_rn(x[2], T.r[6 + d]));
        o[d] = __fadd_rn(__fmul_rn(T.s, acc), T.t[d]);
    }
}

// a shift point: p when finite, else 0
__device__ __forceinline__ void ref_of(const float (&p)[3], double (&r)[3]) {
    const bool fin = isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]);
#pragma unroll
    for (int c = 0; c < 3; c++) r[c] = fin ? (double)p[c] : 0.0;
}

// shift of cloud n of X (or of Y): its first point (0 when it has no rows: P = 0, and the pointer may be NULL).  X and Y
// each get their own, so that a constant cloud has centred moments of exactly 0.
__device__ __forceinline__ void ref_point(const Pts &X, int n, int P, double (&r)[3]) {
    float x[3] = {0.f, 0.f, 0.f};
    if (P > 0) ld3(X, n, 0, x);
    ref_of(x, r);
}

// Moments of one point with weight w, coordinates shifted by ref: {w, w x, w y, w^2, w^2 x, w^2 y, w^2 x y^T, w^2 |x|^2}.
// A point of weight exactly 0 contributes nothing (not even a NaN of its coordinates).
__device__ __forceinline__ void point_moments(const float (&xf)[3], const float (&yf)[3], double w, const double (&xref)[3],
                                              const double (&yref)[3], double (&m)[NMOM]) {
#pragma unroll
    for (int k = 0; k < NMOM; k++) m[k] = 0.0;
    if (w == 0.0) return;
    double x[3], y[3];
#pragma unroll
    for (int c = 0; c < 3; c++) { x[c] = (double)xf[c] - xref[c]; y[c] = (double)yf[c] - yref[c]; }
    const double w2 = w * w;
    m[0] = w;
    m[7] = w2;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        m[1 + c] = w * x[c];
        m[4 + c] = w * y[c];
        m[8 + c] = w2 * x[c];
        m[11 + c] = w2 * y[c];
#pragma unroll
        for (int d = 0; d < 3; d++) m[14 + 3 * c + d] = w2 * x[c] * y[d];
    }
    m[23] = w2 * (x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
}

template <int N>
__device__ __forceinline__ void warp_sum(double (&m)[N]) {  // every lane ends with the same bits (fp addition commutes)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int k = 0; k < N; k++) m[k] += __shfl_xor_sync(0xffffffffu, m[k], off);
}

__device__ __forceinline__ void store_partial(double *dst, const double (&m)[NMOM], int lane) {
#pragma unroll
    for (int k = 0; k < NMOM; k++)
        if (lane == k) dst[k] = m[k];
}

// sum of the nblk block partials of one cloud (plain loads: in pcl_icp they are written by the same launch)
__device__ __forceinline__ void cloud_moments(const double *part, int nblk, int lane, double (&m)[NMOM]) {
#pragma unroll
    for (int k = 0; k < NMOM; k++) m[k] = 0.0;
    for (int b = lane; b < nblk; b += 32)
#pragma unroll
        for (int k = 0; k < NMOM; k++) m[k] += part[(size_t)b * NMOM + k];
    warp_sum(m);
}

// The per-cloud record the backward reads (PCL_ALIGN_RECORD doubles).
enum { RC_U = 0, RC_V = 9, RC_SIG = 18, RC_XM = 21, RC_YM = 24, RC_QX = 27, RC_QY = 30, RC_SW = 33, RC_WM = 34, RC_WT = 35,
       RC_XCOV = 36, RC_S = 37, RC_TRES = 38 };
static_assert(RC_TRES < PCL_ALIGN_RECORD, "record layout");

// One-sided Jacobi SVD of m: a = m V with orthogonal columns, sorted by norm descending (ties keep their order).
__device__ __forceinline__ void hestenes3(const double (&m)[3][3], double (&a)[3][3], double (&v)[3][3]) {
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) { a[r][c] = m[r][c]; v[r][c] = (r == c) ? 1.0 : 0.0; }
    auto rot = [&](int p, int q) -> bool {
        double al = 0.0, be = 0.0, ga = 0.0;
#pragma unroll
        for (int k = 0; k < 3; k++) { al += a[k][p] * a[k][p]; be += a[k][q] * a[k][q]; ga += a[k][p] * a[k][q]; }
        if (!(fabs(ga) > SVD_TOL * sqrt(al * be))) return false;  // NaN: no rotation
        const double z = (be - al) / (2.0 * ga);
        const double t = copysign(1.0, z) / (fabs(z) + sqrt(fma(z, z, 1.0)));  // z^2 = inf: t = 0
        const double c = 1.0 / sqrt(fma(t, t, 1.0)), s = c * t;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const double ap = a[k][p], aq = a[k][q], vp = v[k][p], vq = v[k][q];
            a[k][p] = c * ap - s * aq; a[k][q] = s * ap + c * aq;
            v[k][p] = c * vp - s * vq; v[k][q] = s * vp + c * vq;
        }
        return true;
    };
    for (int sweep = 0; sweep < SVD_MAX_SWEEPS; sweep++) {
        bool any = rot(0, 1);
        any |= rot(0, 2);
        any |= rot(1, 2);
        if (!any) break;
    }
    double nrm[3];
#pragma unroll
    for (int c = 0; c < 3; c++) nrm[c] = a[0][c] * a[0][c] + a[1][c] * a[1][c] + a[2][c] * a[2][c];
    auto cx = [&](int x, int y) {
        if (nrm[y] > nrm[x]) {
            const double t = nrm[x]; nrm[x] = nrm[y]; nrm[y] = t;
#pragma unroll
            for (int r = 0; r < 3; r++) {
                double u = a[r][x]; a[r][x] = a[r][y]; a[r][y] = u;
                u = v[r][x]; v[r][x] = v[r][y]; v[r][y] = u;
            }
        }
    };
    cx(0, 1);
    cx(1, 2);
    cx(0, 1);
}

__device__ __forceinline__ double det3(const double (&v)[3][3]) {
    return v[0][0] * (v[1][1] * v[2][2] - v[1][2] * v[2][1]) - v[0][1] * (v[1][0] * v[2][2] - v[1][2] * v[2][0]) +
           v[0][2] * (v[1][0] * v[2][1] - v[1][1] * v[2][0]);
}

// The solve of one cloud from its summed moments: writes the fp32 transform and, when rec != nullptr, the backward record.
// eps, weighted, est, refl: as in pcl.h.
__device__ void solve_cloud(const double (&m)[NMOM], const double (&xref)[3], const double (&yref)[3], bool weighted, bool est, bool refl, double eps,
                            Sim &out, double *rec) {
    const double Sw = m[0], Wm = fmax(Sw, eps), Q0 = m[7];
    const double Wt = weighted ? Wm : fmax(Sw, 1.0);  // unweighted: w is the 0/1 mask and Sw the point count
    double mx[3], my[3], qx[3], qy[3];                 // shifted means; w^2-moments of the centred points
#pragma unroll
    for (int c = 0; c < 3; c++) {
        mx[c] = m[1 + c] / Wm;
        my[c] = m[4 + c] / Wm;
        qx[c] = m[8 + c] - Q0 * mx[c];
        qy[c] = m[11 + c] - Q0 * my[c];
    }
    double M[3][3];
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
        for (int d = 0; d < 3; d++)
            M[c][d] = (m[14 + 3 * c + d] - m[8 + c] * my[d] - mx[c] * m[11 + d] + Q0 * mx[c] * my[d]) / Wt;
    const double cxx = m[23] - 2.0 * (mx[0] * m[8] + mx[1] * m[9] + mx[2] * m[10]) + Q0 * (mx[0] * mx[0] + mx[1] * mx[1] + mx[2] * mx[2]);
    const double xcov = cxx / Wt;

    double a[3][3], v[3][3], u[3][3], sg[3];
    hestenes3(M, a, v);
    if (det3(v) < 0.0) {
#pragma unroll
        for (int r = 0; r < 3; r++) { v[r][2] = -v[r][2]; a[r][2] = -a[r][2]; }
    }
    const double s1 = sqrt(a[0][0] * a[0][0] + a[1][0] * a[1][0] + a[2][0] * a[2][0]);
    if (!(s1 > 0.0)) {  // M = 0 (or NaN): U = V, so R = V V^T = I for M = 0
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int c = 0; c < 3; c++) u[r][c] = v[r][c];
    } else {
        double u1[3], r2[3];
#pragma unroll
        for (int r = 0; r < 3; r++) u1[r] = a[r][0] / s1;
        const double p = u1[0] * a[0][1] + u1[1] * a[1][1] + u1[2] * a[2][1];
#pragma unroll
        for (int r = 0; r < 3; r++) r2[r] = a[r][1] - p * u1[r];
        double n2 = sqrt(r2[0] * r2[0] + r2[1] * r2[1] + r2[2] * r2[2]);
        if (!(n2 > RANK_TOL * s1)) {  // rank <= 1: the axis least aligned with u1 (first on ties), orthogonalised
            int k = 0;
            if (fabs(u1[1]) < fabs(u1[k])) k = 1;
            if (fabs(u1[2]) < fabs(u1[k])) k = 2;
#pragma unroll
            for (int r = 0; r < 3; r++) r2[r] = ((r == k) ? 1.0 : 0.0) - u1[k] * u1[r];
            n2 = sqrt(r2[0] * r2[0] + r2[1] * r2[1] + r2[2] * r2[2]);
        }
#pragma unroll
        for (int r = 0; r < 3; r++) { u[r][0] = u1[r]; u[r][1] = r2[r] / n2; }
        u[0][2] = u[1][0] * u[2][1] - u[2][0] * u[1][1];
        u[1][2] = u[2][0] * u[0][1] - u[0][0] * u[2][1];
        u[2][2] = u[0][0] * u[1][1] - u[1][0] * u[0][1];
    }
#pragma unroll
    for (int c = 0; c < 3; c++) sg[c] = u[0][c] * a[0][c] + u[1][c] * a[1][c] + u[2][c] * a[2][c];  // u_c^T M v_c
    if (refl && sg[2] < 0.0) {
#pragma unroll
        for (int r = 0; r < 3; r++) u[r][2] = -u[r][2];
        sg[2] = -sg[2];
    }
    double R[3][3];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) R[r][c] = u[r][0] * v[c][0] + u[r][1] * v[c][1] + u[r][2] * v[c][2];
    const double tres = sg[0] + sg[1] + sg[2];
    const double s = est ? tres / fmax(xcov, eps) : 1.0;
    double xm[3], ym[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {  // sum w x / Wm = ref sum w / Wm + mx (Sw / Wm = 1 unless the clamp is active)
        xm[c] = xref[c] * (Sw / Wm) + mx[c];
        ym[c] = yref[c] * (Sw / Wm) + my[c];
    }
#pragma unroll
    for (int d = 0; d < 3; d++) {
        out.t[d] = (float)(ym[d] - s * (xm[0] * R[0][d] + xm[1] * R[1][d] + xm[2] * R[2][d]));
#pragma unroll
        for (int c = 0; c < 3; c++) out.r[3 * c + d] = (float)R[c][d];
    }
    out.s = (float)s;
    if (rec) {
#pragma unroll
        for (int k = 0; k < 9; k++) { rec[RC_U + k] = u[k / 3][k % 3]; rec[RC_V + k] = v[k / 3][k % 3]; }
#pragma unroll
        for (int c = 0; c < 3; c++) {
            rec[RC_SIG + c] = sg[c]; rec[RC_XM + c] = xm[c]; rec[RC_YM + c] = ym[c]; rec[RC_QX + c] = qx[c]; rec[RC_QY + c] = qy[c];
        }
        rec[RC_SW] = Sw; rec[RC_WM] = Wm; rec[RC_WT] = Wt; rec[RC_XCOV] = xcov; rec[RC_S] = s; rec[RC_TRES] = tres;
        rec[PCL_ALIGN_RECORD - 1] = 0.0;
    }
}

__device__ __forceinline__ void store_sim(const Sim &T, float *R, float *Tt, float *s, int n) {
#pragma unroll
    for (int k = 0; k < 9; k++) R[(size_t)n * 9 + k] = T.r[k];
#pragma unroll
    for (int k = 0; k < 3; k++) Tt[(size_t)n * 3 + k] = T.t[k];
    s[n] = T.s;
}

// ------------------------------------------------------------------ alignment
// Forward, pass 1: grid (ceil(nblk / AL_WARPS), B); warp = one block of 32 points -> its moment partials.
__global__ void __launch_bounds__(AL_THREADS)
align_moments_kernel(Pts X, Pts Y, const int64_t *__restrict__ len, const float *__restrict__ wts, int P, int nblk,
                     double *__restrict__ part) {
    const int n = blockIdx.y, lane = threadIdx.x & 31, blk = blockIdx.x * AL_WARPS + (threadIdx.x >> 5);
    if (blk >= nblk) return;  // warp-uniform
    const int i = blk * 32 + lane, lq = len_of(len, n, P);
    double xref[3], yref[3];
    ref_point(X, n, P, xref);
    ref_point(Y, n, P, yref);
    float x[3] = {0.f, 0.f, 0.f}, y[3] = {0.f, 0.f, 0.f};
    double w = 0.0;
    if (i < lq) {
        ld3(X, n, i, x);
        ld3(Y, n, i, y);
        w = wts ? (double)__ldg(wts + (size_t)n * P + i) : 1.0;
    }
    double m[NMOM];
    point_moments(x, y, w, xref, yref, m);
    warp_sum(m);
    store_partial(part + ((size_t)n * nblk + blk) * NMOM, m, lane);
}

// Forward, pass 2: one warp per cloud sums the partials, lane 0 solves.
__global__ void __launch_bounds__(AL_THREADS)
align_solve_kernel(Pts X, Pts Y, const double *__restrict__ part, int B, int P, int nblk, int weighted, int est, int refl, double eps,
                   float *__restrict__ R, float *__restrict__ T, float *__restrict__ s, double *__restrict__ record) {
    const int n = blockIdx.x * AL_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= B) return;
    double m[NMOM];
    cloud_moments(part + (size_t)n * nblk * NMOM, nblk, lane, m);
    if (lane != 0) return;
    double xref[3], yref[3];
    ref_point(X, n, P, xref);
    ref_point(Y, n, P, yref);
    Sim out;
    solve_cloud(m, xref, yref, weighted, est, refl, eps, out, record ? record + (size_t)n * PCL_ALIGN_RECORD : nullptr);
    store_sim(out, R, T, s, n);
}

// Backward: grid (ceil(P / AL_THREADS), B).  Thread 0 turns the record and the upstream gradients into per-cloud
// coefficients (see pcl.h); every thread then writes the gradients of its own point (one writer per element).
__global__ void __launch_bounds__(AL_THREADS)
align_bwd_kernel(Pts X, Pts Y, const int64_t *__restrict__ len, const float *__restrict__ wts, int P, int est, double eps,
                 const double *__restrict__ record, const float *__restrict__ gR, const float *__restrict__ gT,
                 const float *__restrict__ gs, float *__restrict__ gX, float *__restrict__ gY, float *__restrict__ gW) {
    // coef: A = Mbar / Wt (9), alpha = 2 Xcovbar / Wt, gxm = xmbar / Wm (3), gym = ymbar / Wm (3), xm (3), ym (3), c0
    __shared__ double coef[23];
    const int n = blockIdx.y;
    if (threadIdx.x == 0) {
        const double *rc = record + (size_t)n * PCL_ALIGN_RECORD;
        double u[3][3], v[3][3], R[3][3], sg[3], xm[3], ym[3];
#pragma unroll
        for (int k = 0; k < 9; k++) { u[k / 3][k % 3] = rc[RC_U + k]; v[k / 3][k % 3] = rc[RC_V + k]; }
#pragma unroll
        for (int c = 0; c < 3; c++) { sg[c] = rc[RC_SIG + c]; xm[c] = rc[RC_XM + c]; ym[c] = rc[RC_YM + c]; }
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int c = 0; c < 3; c++) R[r][c] = u[r][0] * v[c][0] + u[r][1] * v[c][1] + u[r][2] * v[c][2];
        const double Sw = rc[RC_SW], Wm = rc[RC_WM], Wt = rc[RC_WT], xcov = rc[RC_XCOV], s = rc[RC_S], tres = rc[RC_TRES];
        double Rb[3][3], Tb[3], sb = (gs && est) ? (double)gs[n] : 0.0;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            Tb[c] = gT ? (double)gT[(size_t)n * 3 + c] : 0.0;
#pragma unroll
            for (int d = 0; d < 3; d++) Rb[c][d] = gR ? (double)gR[(size_t)n * 9 + 3 * c + d] : 0.0;
        }
        // T = ym - s R^T xm
        double xmb[3], ymb[3];
        double rx = 0.0;  // T-bar . (R^T xm)
#pragma unroll
        for (int d = 0; d < 3; d++) rx += Tb[d] * (xm[0] * R[0][d] + xm[1] * R[1][d] + xm[2] * R[2][d]);
        if (est) sb -= rx;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            ymb[c] = Tb[c];
            xmb[c] = -s * (R[c][0] * Tb[0] + R[c][1] * Tb[1] + R[c][2] * Tb[2]);
#pragma unroll
            for (int d = 0; d < 3; d++) Rb[c][d] -= s * xm[c] * Tb[d];
        }
        // s = tr(ES) / max(Xcov, eps)
        const double sden = fmax(xcov, eps);
        const double tresb = est ? sb / sden : 0.0;
        const double xcovb = (est && xcov >= eps) ? -sb * s / sden : 0.0;
        (void)tres;
        // R = U V^T: Mbar = U H V^T, H_ij = (G_ij - G_ji) / (sg_i + sg_j), G = U^T Rbar V; tr(ES) adds tresb R
        double G[3][3], H[3][3], Mb[3][3];
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
            for (int j = 0; j < 3; j++) {
                double acc = 0.0;
#pragma unroll
                for (int c = 0; c < 3; c++)
#pragma unroll
                    for (int d = 0; d < 3; d++) acc += u[c][i] * Rb[c][d] * v[d][j];
                G[i][j] = acc;
            }
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
            for (int j = 0; j < 3; j++) H[i][j] = (i == j) ? 0.0 : (G[i][j] - G[j][i]) / (sg[i] + sg[j]);
        double mdot = 0.0;  // <Mbar, M>, M = U diag(sg) V^T
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
            for (int d = 0; d < 3; d++) {
                double acc = 0.0, mm = 0.0;
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    mm += u[c][i] * sg[i] * v[d][i];
#pragma unroll
                    for (int j = 0; j < 3; j++) acc += u[c][i] * H[i][j] * v[d][j];
                }
                Mb[c][d] = acc + tresb * R[c][d];
                mdot += Mb[c][d] * mm;
            }
        const double wtb = -(mdot + xcovb * xcov) / Wt;
        // M = sum a b^T / Wt, Xcov = sum |a|^2 / Wt with a = w (x - xm), b = w (y - ym): the means get -sum_i w_i abar_i etc.
        const double *qx = rc + RC_QX, *qy = rc + RC_QY;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            xmb[c] -= (Mb[c][0] * qy[0] + Mb[c][1] * qy[1] + Mb[c][2] * qy[2] + 2.0 * xcovb * qx[c]) / Wt;
            ymb[c] -= (Mb[0][c] * qx[0] + Mb[1][c] * qx[1] + Mb[2][c] * qx[2]) / Wt;
        }
        // xm = sum w x / Wm: x_i gets w_i xmbar / Wm; w_i gets xmbar . x_i / Wm, written as xmbar . (x_i - xm) / Wm + q
        const double q = (xmb[0] * xm[0] + xmb[1] * xm[1] + xmb[2] * xm[2] + ymb[0] * ym[0] + ymb[1] * ym[1] + ymb[2] * ym[2]) / Wm;
        const bool weighted = wts != nullptr;
        const double swb = (Sw >= eps) ? (-q + (weighted ? wtb : 0.0)) : 0.0;  // through Wm (and Wt) = max(Sw, eps)
#pragma unroll
        for (int k = 0; k < 9; k++) coef[k] = Mb[k / 3][k % 3] / Wt;
        coef[9] = 2.0 * xcovb / Wt;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            coef[10 + c] = xmb[c] / Wm; coef[13 + c] = ymb[c] / Wm; coef[16 + c] = xm[c]; coef[19 + c] = ym[c];
        }
        coef[22] = q + swb;
    }
    __syncthreads();
    const int i = blockIdx.x * AL_THREADS + threadIdx.x;
    if (i >= P) return;
    const size_t o = (size_t)n * P + i;
    const int lq = len_of(len, n, P);
    const double w = (i < lq) ? (wts ? (double)__ldg(wts + o) : 1.0) : 0.0;
    float xf[3], yf[3];
    ld3(X, n, i, xf);
    ld3(Y, n, i, yf);
    double xc[3], yc[3], ab[3], bb[3];
#pragma unroll
    for (int c = 0; c < 3; c++) { xc[c] = (double)xf[c] - coef[16 + c]; yc[c] = (double)yf[c] - coef[19 + c]; }
    double gw = coef[22];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        ab[c] = w * (coef[3 * c] * yc[0] + coef[3 * c + 1] * yc[1] + coef[3 * c + 2] * yc[2]) + coef[9] * w * xc[c];
        bb[c] = w * (coef[c] * xc[0] + coef[3 + c] * xc[1] + coef[6 + c] * xc[2]);
        gw += (ab[c] + coef[10 + c]) * xc[c] + (bb[c] + coef[13 + c]) * yc[c];
    }
#pragma unroll
    for (int c = 0; c < 3; c++) {
        gX[o * 3 + c] = (w == 0.0) ? 0.f : (float)(w * (ab[c] + coef[10 + c]));
        gY[o * 3 + c] = (w == 0.0) ? 0.f : (float)(w * (bb[c] + coef[13 + c]));
    }
    if (gW) gW[o] = (i < lq) ? (float)gw : 0.f;
}

// ------------------------------------------------------------------ ICP
// Workspace: [barrier count, generation] | pass flags (B int) | transform slots (2 x B Sim) | nn idx (B x P1 int) |
// moment partials (B x nblk x NMOM double).  Only the barrier words are read before being written in the same launch;
// the host call zeroes them on `stream` before the launch.
struct IcpWs {
    unsigned *bar;
    int *flags;
    Sim *slots;  // slot (k & 1) holds the transform of iteration k
    float *yref;  // (B, 4): the neighbour of X row 0 in the current iteration, Y's shift point
    int *idx;
    double *part;
};

inline size_t icp_ws_layout(int B, int P1, IcpWs *w, char *base) {
    const int nblk = (P1 + 31) / 32;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes, 256); return base ? base + o : nullptr; };
    char *bar = take(2 * sizeof(unsigned));
    char *flags = take((size_t)B * sizeof(int));
    char *slots = take((size_t)2 * B * sizeof(Sim));
    char *yref = take((size_t)B * 4 * sizeof(float));
    char *idx = take((size_t)B * P1 * sizeof(int));
    char *part = take((size_t)B * nblk * NMOM * sizeof(double));
    if (w) *w = IcpWs{(unsigned *)bar, (int *)flags, (Sim *)slots, (float *)yref, (int *)idx, (double *)part};
    return off;
}

__device__ __forceinline__ unsigned ld_acquire(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Grid-wide barrier of a cooperative launch (all CTAs co-resident): arrival counter bar[0], generation bar[1].
__device__ __forceinline__ void grid_barrier(unsigned *bar, unsigned &gen) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned target = gen + 1;
        __threadfence();
        if (atomicAdd(bar, 1u) == gridDim.x - 1) {
            atomicExch(bar, 0u);
            __threadfence();
            atomicExch(bar + 1, target);
        } else {
            while ((int)(ld_acquire(bar + 1) - target) < 0) __nanosleep(32);
        }
        __threadfence();
    }
    gen++;
    __syncthreads();
}

struct IcpArgs {
    Pts X, Y;
    const int64_t *len1, *len2;
    int B, P1, P2, nblk, max_it, est, refl, has_init;
    float thr;
    const float *iR, *iT, *is;
    float *Xt, *Rh, *Th, *sh, *rmse_h;
    int *status;
    IcpWs ws;
};

// the transform Xt of iteration it - 1 is computed from (it = 0: the initial one)
__device__ __forceinline__ Sim icp_transform(const IcpArgs &A, int n, int it) {
    Sim T;
    if (it > 0) return A.ws.slots[(size_t)((it - 1) & 1) * A.B + n];
#pragma unroll
    for (int k = 0; k < 9; k++) T.r[k] = A.has_init ? A.iR[(size_t)n * 9 + k] : ((k % 4 == 0) ? 1.f : 0.f);
#pragma unroll
    for (int k = 0; k < 3; k++) T.t[k] = A.has_init ? A.iT[(size_t)n * 3 + k] : 0.f;
    T.s = A.has_init ? A.is[n] : 1.f;
    return T;
}

// X row i transformed for iteration it's search (without an initial transform, iteration 0 searches with X itself)
__device__ __forceinline__ void icp_xt(const IcpArgs &A, const Sim &T, int n, int i, int it, float (&q)[3]) {
    float x[3];
    ld3(A.X, n, i, x);
    if (it == 0 && !A.has_init) {
#pragma unroll
        for (int c = 0; c < 3; c++) q[c] = x[c];
    } else {
        apply_sim(T, x, q);
    }
}

// Phase A of iteration it: work item (cloud n, block of 32 queries): transform, K = 1 search, moment partials.
template <bool FMA>
__device__ void icp_search_item(const IcpArgs &A, int item, int it, float4 *tile, int lane) {
    const int n = item / A.nblk, blk = item - n * A.nblk, i0 = blk * 32, i = i0 + lane;
    const int lq = len_of(A.len1, n, A.P1), lt = len_of(A.len2, n, A.P2);
    double m[NMOM];
    if (i0 >= lq) {  // warp-uniform: padded rows only
#pragma unroll
        for (int k = 0; k < NMOM; k++) m[k] = 0.0;
    } else {
        const bool valid = i < lq;
        const Sim T = icp_transform(A, n, it);
        float q[3] = {0.f, 0.f, 0.f}, x[3] = {0.f, 0.f, 0.f}, y[3] = {0.f, 0.f, 0.f};
        if (valid) {
            icp_xt(A, T, n, i, it, q);
            ld3(A.X, n, i, x);
        }
        u64 best = KEY_NONE;
        float best_d = __uint_as_float(0x7fffffffu);  // NaN: every target goes to the key test
        for (int t0 = 0; t0 < lt; t0 += ICP_TILE) {
            const int cnt = min(ICP_TILE, lt - t0);
            __syncwarp();  // the previous tile is consumed
            for (int e = lane; e < cnt; e += 32) {
                float t[3];
                ld3(A.Y, n, t0 + e, t);
                tile[e] = make_float4(t[0], t[1], t[2], 0.f);
            }
            __syncwarp();
#pragma unroll 4
            for (int e = 0; e < cnt; e++) {
                const float d = sqdist<FMA, 3>(q, reinterpret_cast<const float *>(tile + e));
                if (!(d > best_d)) {
                    const u64 key = knn_key(d, t0 + e);
                    if (key < best) { best = key; best_d = key_dist(key); }
                }
            }
        }
        const int j = (lt > 0) ? (int)(unsigned)best : 0;
        if (valid) {
            if (lt > 0) ld3(A.Y, n, j, y);
            A.ws.idx[(size_t)n * A.P1 + i] = j;
        }
        double xref[3], yref[3];
        ref_point(A.X, n, A.P1, xref);
        const float *yr = A.ws.yref + (size_t)n * 4;
        ref_of({yr[0], yr[1], yr[2]}, yref);
        point_moments(x, y, valid ? 1.0 : 0.0, xref, yref, m);
        warp_sum(m);
    }
    store_partial(A.ws.part + (size_t)item * NMOM, m, lane);
}

// Y's shift point for the alignment of iteration it: the neighbour of X row 0 under transform T (what
// knn_gather(Y, knn_points(Xt, Y).idx)[n, 0] is; 0 for an empty Y cloud), found by one warp with the search's key.
template <bool FMA>
__device__ void icp_row0_neighbour(const IcpArgs &A, int n, const Sim &T, int it, int lane) {
    const int lq = len_of(A.len1, n, A.P1), lt = len_of(A.len2, n, A.P2);
    float y[3] = {0.f, 0.f, 0.f};
    if (lq > 0 && lt > 0) {  // without X rows there are no moments, and the shift does not matter
        float q[3];
        icp_xt(A, T, n, 0, it, q);
        u64 best = KEY_NONE;
        for (int j = lane; j < lt; j += 32) {
            float t[3];
            ld3(A.Y, n, j, t);
            const u64 key = knn_key(sqdist<FMA, 3>(q, t), j);
            best = key < best ? key : best;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const u64 o = __shfl_xor_sync(0xffffffffu, best, off);
            best = o < best ? o : best;
        }
        ld3(A.Y, n, (int)(unsigned)best, y);
    }
    if (lane == 0) {
#pragma unroll
        for (int c = 0; c < 3; c++) A.ws.yref[(size_t)n * 4 + c] = y[c];
    }
}

// Phase B of iteration it for cloud n (one warp): solve, record, rmse of the new Xt, relative rmse, pass flag, and Y's
// shift point for iteration it + 1.
template <bool FMA>
__device__ void icp_solve_cloud(const IcpArgs &A, int n, int it, int lane) {
    double m[NMOM];
    cloud_moments(A.ws.part + (size_t)n * A.nblk * NMOM, A.nblk, lane, m);
    Sim T;
    if (lane == 0) {
        double xref[3], yref[3];
        ref_point(A.X, n, A.P1, xref);
        const float *yr = A.ws.yref + (size_t)n * 4;
        ref_of({yr[0], yr[1], yr[2]}, yref);
        solve_cloud(m, xref, yref, true, A.est, A.refl, 1e-9, T, nullptr);
        A.ws.slots[(size_t)(it & 1) * A.B + n] = T;
        const size_t h = (size_t)it * A.B;
        store_sim(T, A.Rh + h * 9, A.Th + h * 3, A.sh + h, n);
    }
#pragma unroll
    for (int k = 0; k < 9; k++) T.r[k] = __shfl_sync(0xffffffffu, T.r[k], 0);
#pragma unroll
    for (int k = 0; k < 3; k++) T.t[k] = __shfl_sync(0xffffffffu, T.t[k], 0);
    T.s = __shfl_sync(0xffffffffu, T.s, 0);
    const int lq = len_of(A.len1, n, A.P1), lt = len_of(A.len2, n, A.P2);
    double acc[1] = {0.0};
    for (int i = lane; i < lq; i += 32) {
        float x[3], q[3], y[3] = {0.f, 0.f, 0.f};
        ld3(A.X, n, i, x);
        apply_sim(T, x, q);
        if (lt > 0) ld3(A.Y, n, A.ws.idx[(size_t)n * A.P1 + i], y);
#pragma unroll
        for (int c = 0; c < 3; c++) { const double d = (double)q[c] - (double)y[c]; acc[0] += d * d; }
    }
    warp_sum(acc);
    if (lane == 0) {
        const float r = (float)sqrt(acc[0] / fmax((double)lq, 1e-9));
        A.rmse_h[(size_t)it * A.B + n] = r;
        float rel = 1.f;
        if (it > 0) {
            const float prev = A.rmse_h[(size_t)(it - 1) * A.B + n];
            rel = __fdiv_rn(__fsub_rn(prev, r), prev);
        }
        A.ws.flags[n] = (rel <= A.thr) ? 1 : 0;  // NaN (0 / 0 included) fails
    }
    if (it + 1 < A.max_it) icp_row0_neighbour<FMA>(A, n, T, it + 1, lane);
}

// The whole loop: per iteration, phase A (all warps over the work items) | barrier | phase B (a warp per cloud) | barrier |
// every CTA reads the B pass flags and takes the same decision.  Then Xt, the unused history slots and the status.
template <bool FMA>
__global__ void __launch_bounds__(AL_THREADS)
icp_kernel(IcpArgs A) {
    __shared__ float4 tiles[AL_WARPS][ICP_TILE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * AL_WARPS + warp, nw = gridDim.x * AL_WARPS;
    const int items = A.B * A.nblk;
    unsigned gen = 0;
    int iters = 0, converged = 0;
    if (A.max_it > 0) {
        for (int n = gw; n < A.B; n += nw) icp_row0_neighbour<FMA>(A, n, icp_transform(A, n, 0), 0, lane);
        grid_barrier(A.ws.bar, gen);
    }
    for (int it = 0; it < A.max_it; it++) {
        for (int item = gw; item < items; item += nw) icp_search_item<FMA>(A, item, it, tiles[warp], lane);
        grid_barrier(A.ws.bar, gen);
        for (int n = gw; n < A.B; n += nw) icp_solve_cloud<FMA>(A, n, it, lane);
        grid_barrier(A.ws.bar, gen);
        int ok = 1;
        for (int n = threadIdx.x; n < A.B; n += AL_THREADS) ok &= A.ws.flags[n];
        iters = it + 1;
        if (__syncthreads_and(ok)) { converged = 1; break; }
    }
    // Xt from the last transform (X, or the initial transform, when no iteration ran), every row
    const int it_last = iters;  // icp_transform(it) is the transform of iteration it - 1
    const size_t rows = (size_t)A.B * A.P1;
    for (size_t r = (size_t)blockIdx.x * AL_THREADS + threadIdx.x; r < rows; r += (size_t)gridDim.x * AL_THREADS) {
        const int n = (int)(r / A.P1), i = (int)(r - (size_t)n * A.P1);
        const Sim T = icp_transform(A, n, it_last);
        float q[3];
        icp_xt(A, T, n, i, it_last, q);
#pragma unroll
        for (int c = 0; c < 3; c++) A.Xt[r * 3 + c] = q[c];
    }
    const size_t used = (size_t)iters * A.B, total = (size_t)A.max_it * A.B;
    for (size_t e = used + (size_t)blockIdx.x * AL_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * AL_THREADS) {
#pragma unroll
        for (int k = 0; k < 9; k++) A.Rh[e * 9 + k] = 0.f;
#pragma unroll
        for (int k = 0; k < 3; k++) A.Th[e * 3 + k] = 0.f;
        A.sh[e] = 0.f;
        A.rmse_h[e] = 0.f;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { A.status[0] = iters; A.status[1] = converged; }
}

int check_pts(const char *who, const void *p, int dtype, int B, int P) {
    if (B < 0 || P < 0) { set_error("%s: negative size B=%d P=%d", who, B, P); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B > 0 && P > 0 && !p) { set_error("%s: null input", who); return PCL_E_ARG; }
    return PCL_OK;
}

template <bool FMA>
int launch_icp(const IcpArgs &a, int sm_count, cudaStream_t st) {
    static thread_local int cached_dev = -1, per_sm = 0;  // per instantiation: co-resident CTAs per SM
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (cached_dev != dev) {
        PCL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, icp_kernel<FMA>, AL_THREADS, 0));
        cached_dev = dev;
    }
    if (per_sm < 1) { set_error("icp: the kernel cannot be resident"); return PCL_E_UNSUPPORTED; }
    const long long want = std::max((long long)a.B * a.nblk, (long long)a.B);
    const int grid = (int)std::max(1LL, std::min((long long)per_sm * sm_count, (want + AL_WARPS - 1) / AL_WARPS));
    IcpArgs args = a;
    void *params[] = {&args};
    PCL_CUDA(cudaMemsetAsync(a.ws.bar, 0, 2 * sizeof(unsigned), st));
    PCL_CUDA(cudaLaunchCooperativeKernel((const void *)icp_kernel<FMA>, dim3(grid), dim3(AL_THREADS), params, 0, st));
    return PCL_OK;
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" size_t pcl_points_alignment_workspace_bytes(int B, int P) {
    if (B <= 0 || P <= 0) return 0;
    return (size_t)B * ((P + 31) / 32) * NMOM * sizeof(double);
}

extern "C" int pcl_points_alignment_fwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const void *y, int y_dtype,
                                        int64_t y_bs, int64_t y_rs, const int64_t *len, const float *weights, int B, int P,
                                        int estimate_scale, int allow_reflection, double eps, float *R, float *T, float *s,
                                        double *record, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = check_pts("points_alignment", x, x_dtype, B, P);
    if (!rc) rc = check_pts("points_alignment", y, y_dtype, B, P);
    if (rc) return rc;
    if (B > 65535) { set_error("points_alignment: B=%d > 65535", B); return PCL_E_SHAPE; }
    if (B > 0 && (!R || !T || !s)) { set_error("points_alignment: null output"); return PCL_E_ARG; }
    const size_t need = pcl_points_alignment_workspace_bytes(B, P);
    if (workspace_bytes < need || (need && !workspace)) {
        set_error("points_alignment: workspace %zu < %zu bytes", workspace_bytes, need); return PCL_E_ARG;
    }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0) return PCL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const Pts a{x, x_bs, x_rs, x_dtype}, b{y, y_bs, y_rs, y_dtype};
    const int nblk = (P + 31) / 32;
    double *part = (double *)workspace;
    if (nblk > 0)
        align_moments_kernel<<<dim3((nblk + AL_WARPS - 1) / AL_WARPS, B), AL_THREADS, 0, st>>>(a, b, len, weights, P, nblk, part);
    align_solve_kernel<<<(B + AL_WARPS - 1) / AL_WARPS, AL_THREADS, 0, st>>>(a, b, part, B, P, nblk, weights != nullptr || len != nullptr,
                                                                             estimate_scale, allow_reflection, eps, R, T, s, record);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_points_alignment_bwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const void *y, int y_dtype,
                                        int64_t y_bs, int64_t y_rs, const int64_t *len, const float *weights, int B, int P,
                                        int estimate_scale, double eps, const double *record, const float *grad_R,
                                        const float *grad_T, const float *grad_s, float *grad_x, float *grad_y,
                                        float *grad_weights, void *stream) {
    int rc = check_pts("points_alignment_bwd", x, x_dtype, B, P);
    if (!rc) rc = check_pts("points_alignment_bwd", y, y_dtype, B, P);
    if (rc) return rc;
    if (B > 65535) { set_error("points_alignment_bwd: B=%d > 65535", B); return PCL_E_SHAPE; }
    if (B > 0 && P > 0 && (!record || !grad_x || !grad_y)) { set_error("points_alignment_bwd: null argument"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P == 0) return PCL_OK;
    const Pts a{x, x_bs, x_rs, x_dtype}, b{y, y_bs, y_rs, y_dtype};
    align_bwd_kernel<<<dim3((P + AL_THREADS - 1) / AL_THREADS, B), AL_THREADS, 0, (cudaStream_t)stream>>>(
        a, b, len, weights, P, estimate_scale, eps, record, grad_R, grad_T, grad_s, grad_x, grad_y, grad_weights);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" size_t pcl_icp_workspace_bytes(int B, int P1, int P2, int max_iterations) {
    (void)P2; (void)max_iterations;
    if (B <= 0) return 0;
    return icp_ws_layout(B, std::max(P1, 0), nullptr, nullptr);
}

extern "C" int pcl_icp(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len, const void *y, int y_dtype,
                       int64_t y_bs, int64_t y_rs, const int64_t *y_len, int B, int P1, int P2, const float *init_R,
                       const float *init_T, const float *init_s, int max_iterations, float relative_rmse_thr, int estimate_scale,
                       int allow_reflection, int mode, float *Xt, float *R_hist, float *T_hist, float *s_hist, float *rmse_hist,
                       int32_t *status, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = check_pts("icp", x, x_dtype, B, P1);
    if (!rc) rc = check_pts("icp", y, y_dtype, B, P2);
    if (rc) return rc;
    if (max_iterations < 0) { set_error("icp: max_iterations=%d < 0", max_iterations); return PCL_E_ARG; }
    if (mode != PCL_CHAMFER_UNFUSED && mode != PCL_CHAMFER_FMA) { set_error("icp: bad mode %d", mode); return PCL_E_ARG; }
    const bool has_init = init_R || init_T || init_s;
    if (has_init && !(init_R && init_T && init_s)) { set_error("icp: init_R, init_T and init_s are given together"); return PCL_E_ARG; }
    if (B > 0 && (!status || (P1 > 0 && !Xt) || (max_iterations > 0 && (!R_hist || !T_hist || !s_hist || !rmse_hist)))) {
        set_error("icp: null output"); return PCL_E_ARG;
    }
    const size_t need = pcl_icp_workspace_bytes(B, P1, P2, max_iterations);
    if (workspace_bytes < need || (need && !workspace)) { set_error("icp: workspace %zu < %zu bytes", workspace_bytes, need); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0) return PCL_OK;
    IcpArgs a{};
    a.X = Pts{x, x_bs, x_rs, x_dtype};
    a.Y = Pts{y, y_bs, y_rs, y_dtype};
    a.len1 = x_len; a.len2 = y_len;
    a.B = B; a.P1 = P1; a.P2 = P2; a.nblk = (P1 + 31) / 32; a.max_it = max_iterations;
    a.est = estimate_scale; a.refl = allow_reflection; a.has_init = has_init; a.thr = relative_rmse_thr;
    a.iR = init_R; a.iT = init_T; a.is = init_s;
    a.Xt = Xt; a.Rh = R_hist; a.Th = T_hist; a.sh = s_hist; a.rmse_h = rmse_hist; a.status = status;
    icp_ws_layout(B, P1, &a.ws, (char *)workspace);
    cudaStream_t st = (cudaStream_t)stream;
    rc = (mode == PCL_CHAMFER_FMA) ? launch_icp<true>(a, di.sm_count, st) : launch_icp<false>(a, di.sm_count, st);
    if (rc) return rc;
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
