// pcl_normals.cu -- local coordinate frames and normals of point clouds (forward + backward) for sm_100a.
//
// Replaces pytorch3d.ops.estimate_pointcloud_local_coord_frames / estimate_pointcloud_normals (0.7.2, restated from memory:
// parity with pytorch3d itself is unpinned; the contract is in include/pcl.h).  The K neighbours of every point come from
// pcl_knn_fwd(p, p, len, len, K); this file does the per-point step after the search: mean and covariance of the
// neighbourhood, 3 x 3 symmetric eigen-decomposition (cyclic Jacobi), sign disambiguation, and the backward through the
// eigen-decomposition to the points.
//
// All arithmetic is fp64 on coordinates up-cast from the input (fp16 / bf16 first go to fp32 exactly like `.float()`); the
// outputs are rounded to fp32 once.  Jacobi runs until the off-diagonal is at most 2^-52 of the Frobenius norm (at most
// NRM_MAX_SWEEPS sweeps), so every eigenvalue is within about 1e-16 * ||C|| and every eigenvector within about
// 1e-16 * ||C|| / gap of the exact one.
//
// Both kernels: one thread per point, NRM_THREADS threads per CTA.  Each warp first copies the idx rows of its 32 points
// (one contiguous block of 32 K int32) to shared memory with coalesced loads; each lane then reads its own row there on
// every pass over its neighbours.  No atomics in the forward (bit-reproducible); the backward scatters with red.global.add.
#include <cmath>

#include "pcl_common.cuh"

namespace pcl {
namespace {

constexpr int NRM_MAX_K = 64;          // pcl_knn_max_k()
constexpr int NRM_THREADS = 128;
constexpr int NRM_MAX_SWEEPS = 16;     // a 3 x 3 Jacobi converges in 4-6 sweeps; the cap only bounds NaN / inf inputs
constexpr double NRM_TOL2 = 0x1p-104;  // (2^-52)^2: stop when ||offdiag||_F^2 <= 2^-104 ||C||_F^2

__device__ __forceinline__ float ld_pt(const Pts &a, int64_t i) {  // as pcl_knn.cu: one 32-bit or one 16-bit load
    if (a.dtype == PCL_F32) return __ldg(reinterpret_cast<const float *>(a.p) + i);
    const unsigned short h = __ldg(reinterpret_cast<const unsigned short *>(a.p) + i);
    return (a.dtype == PCL_F16) ? __half2float(__ushort_as_half(h)) : __uint_as_float((unsigned)h << 16);
}

__device__ __forceinline__ void ld_point(const Pts &a, int n, int j, double (&x)[3]) {
    const int64_t o = (int64_t)n * a.bs + (int64_t)j * a.rs;
#pragma unroll
    for (int c = 0; c < 3; c++) x[c] = (double)ld_pt(a, o + c);
}

// Copy the idx rows of this warp's points [i0, i0 + rows) to sm (row r at sm[r K]) and return this lane's row.
__device__ __forceinline__ const int *stage_rows(const int32_t *__restrict__ knn_idx, int *sm, size_t row0, int rows, int K,
                                                 int lane) {
    const int32_t *src = knn_idx + row0 * K;
    for (int e = lane; e < rows * K; e += 32) sm[e] = __ldg(src + e);
    __syncwarp();
    return sm + lane * K;
}

// mean of the K neighbours of a point (rows: this lane's idx row; j clamped into the cloud so that a bad idx cannot read
// past it)
__device__ __forceinline__ void neighbourhood_mean(const Pts &a, int n, int lq, const int *row, int K, double (&mu)[3]) {
    mu[0] = mu[1] = mu[2] = 0.0;
    for (int k = 0; k < K; k++) {
        double x[3];
        ld_point(a, n, min((unsigned)row[k], (unsigned)(lq - 1)), x);
#pragma unroll
        for (int c = 0; c < 3; c++) mu[c] += x[c];
    }
    const double inv = 1.0 / K;
#pragma unroll
    for (int c = 0; c < 3; c++) mu[c] *= inv;
}

// one Jacobi rotation that zeroes a[p][q] (Numerical Recipes' jacobi): A <- J^T A J, V <- V J
template <int p, int q>
__device__ __forceinline__ void rotate(double (&a)[3][3], double (&v)[3][3]) {
    constexpr int r = 3 - p - q;
    const double apq = a[p][q];
    if (apq == 0.0) return;
    const double theta = (a[q][q] - a[p][p]) / (2.0 * apq);
    // not hypot (its call makes ptxas spill): for |theta| > 1e154, theta^2 = inf gives t = 0, i.e. an a[p][q] below
    // 1e-154 |a[q][q] - a[p][p]| is dropped, far under the stopping tolerance
    const double t = copysign(1.0, theta) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
    const double c = 1.0 / sqrt(fma(t, t, 1.0)), s = t * c;
    const double arp = a[r][p], arq = a[r][q];
    a[p][p] -= t * apq;
    a[q][q] += t * apq;
    a[p][q] = a[q][p] = 0.0;
    a[r][p] = a[p][r] = c * arp - s * arq;
    a[r][q] = a[q][r] = s * arp + c * arq;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double vp = v[k][p], vq = v[k][q];
        v[k][p] = c * vp - s * vq;
        v[k][q] = s * vp + c * vq;
    }
}

// eigenvalues ascending in lam, eigenvector c in column c of v
__device__ __forceinline__ void eigh3(double (&a)[3][3], double (&lam)[3], double (&v)[3][3]) {
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) v[r][c] = (r == c) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < NRM_MAX_SWEEPS; sweep++) {
        const double off2 = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
        const double fro2 = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2] + 2.0 * off2;
        if (!(2.0 * off2 > NRM_TOL2 * fro2)) break;  // NaN: stop as well
        rotate<0, 1>(a, v);
        rotate<0, 2>(a, v);
        rotate<1, 2>(a, v);
    }
#pragma unroll
    for (int c = 0; c < 3; c++) lam[c] = a[c][c];
    auto swap_cols = [&](int x, int y) {  // three compare-exchanges; equal eigenvalues keep their order
        if (lam[y] < lam[x]) {
            const double t = lam[x]; lam[x] = lam[y]; lam[y] = t;
#pragma unroll
            for (int r = 0; r < 3; r++) { const double u = v[r][x]; v[r][x] = v[r][y]; v[r][y] = u; }
        }
    };
    swap_cols(0, 1);
    swap_cols(1, 2);
    swap_cols(0, 1);
}

// grid (ceil(P / NRM_THREADS), B); block NRM_THREADS; dynamic shared memory NRM_THREADS * K int32
__global__ void __launch_bounds__(NRM_THREADS)
frames_fwd_kernel(Pts a, const int64_t *__restrict__ len, int P, int K, int disambiguate, const int32_t *__restrict__ knn_idx,
                  float *__restrict__ curvatures, float *__restrict__ frames) {
    extern __shared__ int nrm_sm[];
    const int n = blockIdx.y, lane = threadIdx.x & 31;
    const int i0 = blockIdx.x * NRM_THREADS + (threadIdx.x & ~31), i = i0 + lane;
    if (i0 >= P) return;  // warp-uniform
    const int lq = len_of(len, n, P);
    float *cv = curvatures + ((size_t)n * P + i) * 3;
    float *fr = frames + ((size_t)n * P + i) * 9;
    auto zero_row = [&]() {
        if (i >= P) return;
#pragma unroll
        for (int c = 0; c < 3; c++) cv[c] = 0.f;
#pragma unroll
        for (int c = 0; c < 9; c++) fr[c] = 0.f;
    };
    if (i0 >= lq || lq <= K) { zero_row(); return; }  // warp-uniform: padded rows only, or a cloud of at most K points
    const int *row = stage_rows(knn_idx, nrm_sm + (threadIdx.x & ~31) * K, (size_t)n * P + i0, min(32, P - i0), K, lane);
    if (i >= lq) { zero_row(); return; }
    double mu[3];
    neighbourhood_mean(a, n, lq, row, K, mu);
    double cov[3][3] = {};
    for (int k = 0; k < K; k++) {
        double x[3];
        ld_point(a, n, min((unsigned)row[k], (unsigned)(lq - 1)), x);
#pragma unroll
        for (int c = 0; c < 3; c++) x[c] -= mu[c];
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int c = r; c < 3; c++) cov[r][c] = fma(x[r], x[c], cov[r][c]);
    }
    const double inv = 1.0 / K;
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = r; c < 3; c++) cov[c][r] = cov[r][c] = cov[r][c] * inv;
    double lam[3], v[3][3];
    eigh3(cov, lam, v);
    if (disambiguate) {
        // n_pos of v0 and v2: neighbours with v . (p_j - p_i) > 0; flip where 2 n_pos < K.  Then (v0, v0 x v2, v2).
        double pi[3];
        ld_point(a, n, i, pi);
        int pos0 = 0, pos2 = 0;
        for (int k = 0; k < K; k++) {
            double x[3];
            ld_point(a, n, min((unsigned)row[k], (unsigned)(lq - 1)), x);
#pragma unroll
            for (int c = 0; c < 3; c++) x[c] -= pi[c];
            pos0 += (v[0][0] * x[0] + v[1][0] * x[1] + v[2][0] * x[2]) > 0.0;
            pos2 += (v[0][2] * x[0] + v[1][2] * x[1] + v[2][2] * x[2]) > 0.0;
        }
        const double s0 = (2 * pos0 < K) ? -1.0 : 1.0, s2 = (2 * pos2 < K) ? -1.0 : 1.0;
#pragma unroll
        for (int r = 0; r < 3; r++) { v[r][0] *= s0; v[r][2] *= s2; }
        v[0][1] = v[1][0] * v[2][2] - v[2][0] * v[1][2];
        v[1][1] = v[2][0] * v[0][2] - v[0][0] * v[2][2];
        v[2][1] = v[0][0] * v[1][2] - v[1][0] * v[0][2];
    }
#pragma unroll
    for (int c = 0; c < 3; c++) cv[c] = (float)lam[c];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) fr[r * 3 + c] = (float)v[r][c];
}

// Backward.  With V = frames (columns), lam = curvatures, M = V^T Vbar and F_ij = 1 / (lam_j - lam_i) (i != j):
//   Cbar = V (diag(lam_bar) + F o M) V^T,  S = (Cbar + Cbar^T) / K,  grad_p[j] += S (p_j - mu_i) for every neighbour j of i.
// A term F_ij M_ij with M_ij == 0 is 0 (an upstream gradient that does not touch a pair of equal eigenvalues stays finite).
__global__ void __launch_bounds__(NRM_THREADS)
frames_bwd_kernel(Pts a, const int64_t *__restrict__ len, int P, int K, const int32_t *__restrict__ knn_idx,
                  const float *__restrict__ curvatures, const float *__restrict__ frames, const float *__restrict__ grad_curv,
                  const float *__restrict__ grad_frames, float *__restrict__ grad_p) {
    extern __shared__ int nrm_sm[];
    const int n = blockIdx.y, lane = threadIdx.x & 31;
    const int i0 = blockIdx.x * NRM_THREADS + (threadIdx.x & ~31), i = i0 + lane;
    if (i0 >= P) return;
    const int lq = len_of(len, n, P);
    if (i0 >= lq || lq <= K) return;  // warp-uniform: these rows have no gradient
    const int *row = stage_rows(knn_idx, nrm_sm + (threadIdx.x & ~31) * K, (size_t)n * P + i0, min(32, P - i0), K, lane);
    if (i >= lq) return;
    const size_t r0 = (size_t)n * P + i;
    double v[3][3], lam[3], g[3][3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
        lam[r] = (double)__ldg(curvatures + r0 * 3 + r);
#pragma unroll
        for (int c = 0; c < 3; c++) v[r][c] = (double)__ldg(frames + r0 * 9 + r * 3 + c);
    }
    // g = diag(lam_bar) + F o (V^T Vbar)
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) g[r][c] = 0.0;
    if (grad_frames) {
        double vb[3][3];
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int c = 0; c < 3; c++) vb[r][c] = (double)__ldg(grad_frames + r0 * 9 + r * 3 + c);
#pragma unroll
        for (int r = 0; r < 3; r++)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                if (r == c) continue;
                const double m = v[0][r] * vb[0][c] + v[1][r] * vb[1][c] + v[2][r] * vb[2][c];
                g[r][c] = (m == 0.0) ? 0.0 : m / (lam[c] - lam[r]);
            }
    }
    if (grad_curv) {
#pragma unroll
        for (int c = 0; c < 3; c++) g[c][c] = (double)__ldg(grad_curv + r0 * 3 + c);
    }
    // S = (V g V^T + V g^T V^T) / K = V (g + g^T) V^T / K
    double h[3][3], s[3][3];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) h[r][c] = g[r][c] + g[c][r];
    const double inv = 1.0 / K;
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = r; c < 3; c++) {
            double acc = 0.0;
#pragma unroll
            for (int x = 0; x < 3; x++)
#pragma unroll
                for (int y = 0; y < 3; y++) acc += v[r][x] * h[x][y] * v[c][y];
            s[r][c] = s[c][r] = acc * inv;
        }
    double mu[3];
    neighbourhood_mean(a, n, lq, row, K, mu);
    for (int k = 0; k < K; k++) {
        const int j = min((unsigned)row[k], (unsigned)(lq - 1));
        double x[3];
        ld_point(a, n, j, x);
#pragma unroll
        for (int c = 0; c < 3; c++) x[c] -= mu[c];
        float *gp = grad_p + ((size_t)n * P + j) * 3;
#pragma unroll
        for (int r = 0; r < 3; r++) atomicAdd(gp + r, (float)(s[r][0] * x[0] + s[r][1] * x[1] + s[r][2] * x[2]));
    }
}

int check_args(const char *who, const void *p, int dtype, int B, int P, int K, const int32_t *knn_idx) {
    if (B < 0 || P < 0) { set_error("%s: negative size B=%d P=%d", who, B, P); return PCL_E_SHAPE; }
    if (K < 1) { set_error("%s: K=%d must be at least 1", who, K); return PCL_E_SHAPE; }
    if (K > NRM_MAX_K) { set_error("%s: K=%d > pcl_knn_max_k() = %d", who, K, NRM_MAX_K); return PCL_E_UNSUPPORTED; }
    if (B > 65535) { set_error("%s: B=%d > 65535", who, B); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B > 0 && P > 0 && (!p || !knn_idx)) { set_error("%s: null input", who); return PCL_E_ARG; }
    return PCL_OK;
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_frames_fwd(const void *p, int dtype, int64_t bs, int64_t rs, const int64_t *len, int B, int P, int K,
                              int disambiguate, const int32_t *knn_idx, float *curvatures, float *frames, void *stream) {
    int rc = check_args("frames", p, dtype, B, P, K, knn_idx);
    if (rc) return rc;
    if (B > 0 && P > 0 && (!curvatures || !frames)) { set_error("frames: null output"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P == 0) return PCL_OK;
    const Pts a{p, bs, rs, dtype};
    frames_fwd_kernel<<<dim3((P + NRM_THREADS - 1) / NRM_THREADS, B), NRM_THREADS, NRM_THREADS * K * sizeof(int),
                        (cudaStream_t)stream>>>(a, len, P, K, disambiguate, knn_idx, curvatures, frames);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_frames_bwd(const void *p, int dtype, int64_t bs, int64_t rs, const int64_t *len, int B, int P, int K,
                              const int32_t *knn_idx, const float *curvatures, const float *frames, const float *grad_curvatures,
                              const float *grad_frames, float *grad_p, void *stream) {
    int rc = check_args("frames_bwd", p, dtype, B, P, K, knn_idx);
    if (rc) return rc;
    if (B > 0 && P > 0 && (!curvatures || !frames || !grad_p)) { set_error("frames_bwd: null argument"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P == 0) return PCL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    PCL_CUDA(cudaMemsetAsync(grad_p, 0, (size_t)B * P * 3 * sizeof(float), st));
    if (!grad_curvatures && !grad_frames) return PCL_OK;
    const Pts a{p, bs, rs, dtype};
    frames_bwd_kernel<<<dim3((P + NRM_THREADS - 1) / NRM_THREADS, B), NRM_THREADS, NRM_THREADS * K * sizeof(int), st>>>(
        a, len, P, K, knn_idx, curvatures, frames, grad_curvatures, grad_frames, grad_p);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
