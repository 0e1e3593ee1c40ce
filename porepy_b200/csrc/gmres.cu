// gmres.cu -- vector kernels of the restarted, right-preconditioned GMRES(m) with classical Gram-Schmidt and one
// reorthogonalisation pass (CGS2) that solves the contact models' Newton steps (krylov.gmres).
//
// The Krylov basis V is n x (m+1), column-major (column k at V + k n).  One Arnoldi step j:
//   z = M^-1 V[:, j]          (pb_local_block_apply_dev; no preconditioner: z = V[:, j])
//   w = V[:, j+1] = A z       (pb_csr_spmv_dev)
//   twice: h_p = V[:, :j+1]^T w  (pb_gm_dots),  w -= V[:, :j+1] h_p, ||w||^2  (pb_gm_orth)
//   pb_gm_givens: column j of the Hessenberg matrix, the stored Givens rotations, the new one, g, the residual estimate
//   pb_gm_scale:  V[:, j+1] *= 1 / h_{j+1,j}
// End of a cycle: pb_gm_ysolve (R y = g), pb_gm_combine (t = V y), z = M^-1 t, pb_gm_axpy (x += z).
// Start of a cycle: r = b - A x into V[:, 0] with ||r||^2 (pb_gm_residual), pb_gm_start (beta, g, 1 / beta), scale.
//
// Every scalar of the recurrence lives in device memory: `scal` (GS_* below), the dot buffer `hb` (two passes of m+1
// plus the two norms), the Hessenberg matrix H ((m+1) x m, column-major, overwritten by R), the rotations cs / sn and g.
// DONE is sticky: once the estimate |g_{j+1}| is below tol ||b|| (or h_{j+1,j} vanishes: the Krylov space is invariant)
// every later kernel of the cycle returns at once, so the host may read the scalars only every few steps.
#include "plan.hpp"

#define GS_BB 0       // ||b||^2
#define GS_RR 1       // ||b - A x||^2 at the start of the cycle (the true residual)
#define GS_TOLABS 2   // tol ||b||
#define GS_RES 3      // residual estimate |g_{K}|
#define GS_INVH 4     // 1 / h_{j+1,j} (1 / beta at the start of a cycle)
#define GS_DONE 5
#define GS_K 6        // Arnoldi steps of the current cycle
#define GS_SIZE 8

namespace {

constexpr int kGmThreads = 256;
constexpr int kGmCols = 4;      // basis columns per CTA row of the multi-column dot

__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// sum over the CTA of v, added to *slot by thread 0's warp
__device__ __forceinline__ void cta_add(double v, double *slot, double *part) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) part[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < (blockDim.x >> 5) ? part[lane] : 0.0;
        v = warp_sum(v);
        if (lane == 0) atomicAdd(slot, v);
    }
    __syncthreads();
}

// h[c] += V[:, c]^T w for c < ncols: blockIdx.y picks kGmCols columns, w is read once per group
__global__ void gm_dots_kernel(int64_t n, const double *__restrict__ V, int ncols, const double *__restrict__ w,
                               double *__restrict__ h, const double *__restrict__ scal) {
    if (scal[GS_DONE] != 0.0) return;
    __shared__ double part[kGmCols][kGmThreads / 32];
    const int c0 = blockIdx.y * kGmCols;
    double acc[kGmCols] = {};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double wi = w[i];
#pragma unroll
        for (int c = 0; c < kGmCols; ++c)
            if (c0 + c < ncols) acc[c] += V[(int64_t)(c0 + c) * n + i] * wi;
    }
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < kGmCols; ++c) {
        const double v = warp_sum(acc[c]);
        if (lane == 0) part[c][wp] = v;
    }
    __syncthreads();
    if (wp < kGmCols && c0 + wp < ncols) {
        double v = lane < (kGmThreads >> 5) ? part[wp][lane] : 0.0;
        v = warp_sum(v);
        if (lane == 0) atomicAdd(h + c0 + wp, v);
    }
}

// w -= V[:, :ncols] h;  *ww += ||w||^2
__global__ void gm_orth_kernel(int64_t n, const double *__restrict__ V, int ncols, const double *__restrict__ h,
                               double *__restrict__ w, double *__restrict__ ww, const double *__restrict__ scal) {
    if (scal[GS_DONE] != 0.0) return;
    extern __shared__ double sh[];
    __shared__ double part[kGmThreads / 32];
    for (int c = threadIdx.x; c < ncols; c += blockDim.x) sh[c] = h[c];
    __syncthreads();
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double wi = w[i];
        for (int c = 0; c < ncols; ++c) wi -= V[(int64_t)c * n + i] * sh[c];
        w[i] = wi;
        acc += wi * wi;
    }
    cta_add(acc, ww, part);
}

// column j of H from the two Gram-Schmidt passes, the stored rotations, a new one; g, the estimate, 1 / h_{j+1,j}
__global__ void gm_givens_kernel(int j, int m, double *__restrict__ H, double *__restrict__ hb, double *__restrict__ cs,
                                 double *__restrict__ sn, double *__restrict__ g, double *__restrict__ scal) {
    if (threadIdx.x != 0 || scal[GS_DONE] != 0.0) return;
    double *col = H + (int64_t)j * (m + 1);
    double *h2 = hb + (m + 1), *ww = hb + 2 * (m + 1);
    for (int i = 0; i <= j; ++i) col[i] = hb[i] + h2[i];
    const double hn = sqrt(fmax(ww[1], 0.0));
    for (int i = 0; i < j; ++i) {
        const double a = col[i], b = col[i + 1];
        col[i] = cs[i] * a + sn[i] * b;
        col[i + 1] = -sn[i] * a + cs[i] * b;
    }
    const double a = col[j];
    const double r = hypot(a, hn);
    const double c = r > 0.0 ? a / r : 1.0, s = r > 0.0 ? hn / r : 0.0;
    cs[j] = c;
    sn[j] = s;
    col[j] = r;
    g[j + 1] = -s * g[j];
    g[j] = c * g[j];
    const double res = fabs(g[j + 1]);
    scal[GS_RES] = res;
    scal[GS_K] = (double)(j + 1);
    scal[GS_INVH] = hn > 0.0 ? 1.0 / hn : 0.0;
    // converged estimate, or an invariant Krylov space (h_{j+1,j} negligible next to the column)
    if (!(res > scal[GS_TOLABS]) || !(hn > 1e-15 * r) || !isfinite(res)) scal[GS_DONE] = 1.0;
    for (int i = 0; i < 2 * (m + 1) + 2; ++i) hb[i] = 0.0;
}

__global__ void gm_scale_kernel(int64_t n, double *__restrict__ v, const double *__restrict__ scal) {
    if (scal[GS_DONE] != 0.0) return;
    const double f = scal[GS_INVH];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        v[i] *= f;
}

// r = b - r (r holds A x on entry);  RR += ||r||^2;  with bb != 0 also BB += ||b||^2
__global__ void gm_residual_kernel(int64_t n, const double *__restrict__ b, double *__restrict__ r,
                                   double *__restrict__ scal, int with_bb) {
    __shared__ double part[kGmThreads / 32];
    double rr = 0.0, bb = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double bi = b[i], ri = bi - r[i];
        r[i] = ri;
        rr += ri * ri;
        bb += bi * bi;
    }
    cta_add(rr, scal + GS_RR, part);
    if (with_bb) cta_add(bb, scal + GS_BB, part);
}

__global__ void gm_start_kernel(int m, double tol, double *__restrict__ hb, double *__restrict__ g,
                                double *__restrict__ scal) {
    if (threadIdx.x != 0) return;
    const double beta = sqrt(fmax(scal[GS_RR], 0.0));
    scal[GS_TOLABS] = tol * sqrt(fmax(scal[GS_BB], 0.0));
    scal[GS_RES] = beta;
    scal[GS_INVH] = beta > 0.0 ? 1.0 / beta : 0.0;
    scal[GS_K] = 0.0;
    scal[GS_DONE] = (beta > scal[GS_TOLABS] && isfinite(beta)) ? 0.0 : 1.0;
    g[0] = beta;
    for (int i = 1; i <= m; ++i) g[i] = 0.0;
    for (int i = 0; i < 2 * (m + 1) + 2; ++i) hb[i] = 0.0;
}

// back substitution R y = g over the K = scal[GS_K] steps of the cycle (R: upper triangle of H)
__global__ void gm_ysolve_kernel(int m, const double *__restrict__ H, const double *__restrict__ g,
                                 double *__restrict__ y, const double *__restrict__ scal) {
    if (threadIdx.x != 0) return;
    const int K = (int)scal[GS_K];
    for (int i = K - 1; i >= 0; --i) {
        double s = g[i];
        for (int k = i + 1; k < K; ++k) s -= H[(int64_t)k * (m + 1) + i] * y[k];
        y[i] = s / H[(int64_t)i * (m + 1) + i];
    }
    for (int i = K; i < m; ++i) y[i] = 0.0;
}

// t = V[:, :K] y (accumulate != 0: t += V y)
__global__ void gm_combine_kernel(int64_t n, const double *__restrict__ V, int m, const double *__restrict__ y,
                                  double *__restrict__ t, const double *__restrict__ scal, int accumulate) {
    extern __shared__ double sy[];
    const int K = (int)scal[GS_K];
    for (int c = threadIdx.x; c < K; c += blockDim.x) sy[c] = y[c];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double acc = accumulate ? t[i] : 0.0;
        for (int c = 0; c < K; ++c) acc += V[(int64_t)c * n + i] * sy[c];
        t[i] = acc;
    }
}

__global__ void gm_axpy_kernel(int64_t n, const double *__restrict__ z, double *__restrict__ x) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        x[i] += z[i];
}

int gm_grid(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + kGmThreads - 1) / kGmThreads, (int64_t)kSMs * 8)); }

}  // namespace

#define GM_LAUNCHED()            \
    do {                         \
        pb_count_launch_();      \
        CUDA_TRY(cudaGetLastError()); \
        return PB_OK;            \
    } while (0)

extern "C" int pb_gm_dots(int64_t n, const double *V, int ncols, const double *w, double *h, const double *scal,
                          uint64_t stream) {
    if (ncols < 1) return pb_fail_(PB_EINVAL, "pb_gm_dots: ncols < 1");
    const dim3 grid(std::min(gm_grid(n), kSMs * 2), (ncols + kGmCols - 1) / kGmCols);
    gm_dots_kernel<<<grid, kGmThreads, 0, (cudaStream_t)stream>>>(n, V, ncols, w, h, scal);
    GM_LAUNCHED();
}

extern "C" int pb_gm_orth(int64_t n, const double *V, int ncols, const double *h, double *w, double *ww,
                          const double *scal, uint64_t stream) {
    if (ncols < 1 || ncols > 4096) return pb_fail_(PB_EINVAL, "pb_gm_orth: ncols must be in [1, 4096]");
    gm_orth_kernel<<<gm_grid(n), kGmThreads, ncols * sizeof(double), (cudaStream_t)stream>>>(n, V, ncols, h, w, ww, scal);
    GM_LAUNCHED();
}

extern "C" int pb_gm_givens(int j, int m, double *H, double *hb, double *cs, double *sn, double *g, double *scal,
                            uint64_t stream) {
    if (j < 0 || j >= m) return pb_fail_(PB_EINVAL, "pb_gm_givens: step outside the cycle");
    gm_givens_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(j, m, H, hb, cs, sn, g, scal);
    GM_LAUNCHED();
}

extern "C" int pb_gm_scale(int64_t n, double *v, const double *scal, uint64_t stream) {
    gm_scale_kernel<<<gm_grid(n), kGmThreads, 0, (cudaStream_t)stream>>>(n, v, scal);
    GM_LAUNCHED();
}

extern "C" int pb_gm_residual(int64_t n, const double *b, double *r, double *scal, int with_bb, uint64_t stream) {
    gm_residual_kernel<<<gm_grid(n), kGmThreads, 0, (cudaStream_t)stream>>>(n, b, r, scal, with_bb);
    GM_LAUNCHED();
}

extern "C" int pb_gm_start(int m, double tol, double *hb, double *g, double *scal, uint64_t stream) {
    gm_start_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(m, tol, hb, g, scal);
    GM_LAUNCHED();
}

extern "C" int pb_gm_ysolve(int m, const double *H, const double *g, double *y, const double *scal, uint64_t stream) {
    gm_ysolve_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(m, H, g, y, scal);
    GM_LAUNCHED();
}

extern "C" int pb_gm_combine(int64_t n, const double *V, int m, const double *y, double *t, const double *scal,
                             int accumulate, uint64_t stream) {
    if (m < 1 || m > 4096) return pb_fail_(PB_EINVAL, "pb_gm_combine: m must be in [1, 4096]");
    gm_combine_kernel<<<gm_grid(n), kGmThreads, m * sizeof(double), (cudaStream_t)stream>>>(n, V, m, y, t, scal, accumulate);
    GM_LAUNCHED();
}

extern "C" int pb_gm_axpy(int64_t n, const double *z, double *x, uint64_t stream) {
    gm_axpy_kernel<<<gm_grid(n), kGmThreads, 0, (cudaStream_t)stream>>>(n, z, x);
    GM_LAUNCHED();
}
