// solver_check.cu -- diagnostic entry points for the dense interaction-region solvers (node_kernels.cuh): the size
// limits of every solver configuration, and one configuration's solve on a batch of caller-given augmented systems.
// The batch kernel reproduces the assembly's use of the solver exactly (assembly_kernels.cuh / launch_one in
// plan.hpp): block size, teams per CTA, grid cap, the per-team shared-memory layout [scratch | rest | A], the odd row
// stride, rowidx starting as the identity, the global-memory workspace for A, and the read-back of the solution.
// This lets the tests drive every configuration and pivoting path with matrices built for the purpose.
#include "plan.hpp"

template <class Solver>
__global__ void __launch_bounds__(Solver::team == 32 ? 128 : Solver::team, Solver::min_blocks)
    local_solve_kernel(const double *__restrict__ Ain, double *__restrict__ X, int32_t *__restrict__ ok,
                       int64_t nsys, int n, int nrhs, int scr_doubles, int rest_doubles, int a_doubles,
                       double *a_ws) {
    extern __shared__ double smem[];
    constexpr int TEAM = Solver::team;
    GpuTeam<TEAM> t;
    const int teams_per_block = blockDim.x / TEAM;
    const int team_in_block = threadIdx.x / TEAM;
    double *scratch = smem;
    if (TEAM == 32) scratch += (size_t)team_in_block * (scr_doubles + rest_doubles + (a_ws ? 0 : a_doubles));
    double *rest = scratch + scr_doubles;
    double *A = a_ws ? a_ws + ((size_t)blockIdx.x * teams_per_block + team_in_block) * a_doubles
                     : rest + rest_doubles;
    int *rowidx = (int *)rest;
    const int m = n + nrhs, W = m | 1;
    for (int64_t i = (int64_t)blockIdx.x * teams_per_block + team_in_block; i < nsys;
         i += (int64_t)gridDim.x * teams_per_block) {
        const double *src = Ain + i * n * m;
        for (int k = t.tid(); k < n * W; k += t.size()) {
            const int r = k / W, c = k - r * W;
            A[k] = c < m ? src[(int64_t)r * m + c] : 0.0;
        }
        for (int r = t.tid(); r < n; r += t.size()) rowidx[r] = r;
        t.sync();
        const bool good = Solver::solve(t, A, n, W, nrhs, rowidx, scratch);
        // X(p, c) = A[rowidx[p]*W + n + c], as phase 5 of the assembly reads it; NaN for a refused system
        double *dst = X + i * n * nrhs;
        for (int k = t.tid(); k < n * nrhs; k += t.size()) {
            const int p = k / nrhs, c = k - p * nrhs;
            dst[k] = good ? A[(int64_t)rowidx[p] * W + n + c] : __longlong_as_double(0x7FF8000000000000LL);
        }
        if (t.tid() == 0) ok[i] = good ? 1 : 0;
        t.sync();  // the next system overwrites A and rowidx
    }
}

extern "C" int pb_solver_limits(int cfg, int *team, int *max_n, int *max_w) {
    if (cfg < 0 || cfg >= kNumCfg) return pb_fail_(PB_EINVAL, "solver configuration out of range");
    if (team) *team = kCfg[cfg].team;
    if (max_n) *max_n = cfg == kCatchAll ? INT_MAX : kCfg[cfg].max_n;
    if (max_w) *max_w = cfg == kCatchAll ? INT_MAX : kCfg[cfg].max_w;
    return PB_OK;
}

template <class Solver>
static int solve_batch(int cfg, bool a_global, int64_t nsys, int n, int nrhs, const double *A, double *X,
                       int32_t *ok) {
    const int m = n + nrhs, W = m | 1;
    const int64_t scr = Solver::scratch_doubles(n);
    const int64_t rest = ((int64_t)n + 1) / 2 + 2;  // rowidx
    const int64_t a = (int64_t)n * W;
    const int team = kCfg[cfg].team;
    const int blk = team == 32 ? 128 : team;
    const int tpb = blk / team;
    const size_t smem = (size_t)(scr + rest + (a_global ? 0 : a)) * sizeof(double) * tpb;
    if (smem > kMaxSmem)
        return pb_fail_(PB_EINVAL, "system needs " + std::to_string(smem) + " B of shared memory (> 227 KB)");
    if (nsys == 0) return PB_OK;
    auto kernel = local_solve_kernel<Solver>;
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, blk, smem));
    if (per_sm < 1) per_sm = 1;
    const int64_t need = (nsys + tpb - 1) / tpb;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(need, (int64_t)kSMs * per_sm));
    const size_t in_n = (size_t)nsys * n * m, out_n = (size_t)nsys * n * nrhs;
    DevBuf dA, dX, dok, ws;
    CUDA_TRY(dA.upload(A, in_n, 0));
    CUDA_TRY(dX.ensure(out_n * sizeof(double)));
    CUDA_TRY(dok.ensure((size_t)nsys * sizeof(int32_t)));
    if (a_global) {
        // NaN-filled, so that a system that reads workspace entries it did not write comes out non-finite
        CUDA_TRY(ws.ensure((size_t)grid * tpb * a * sizeof(double)));
        CUDA_TRY(cudaMemsetAsync(ws.p, 0xFF, (size_t)grid * tpb * a * sizeof(double), 0));
    }
    kernel<<<grid, blk, smem, 0>>>(dA.as<double>(), dX.as<double>(), dok.as<int32_t>(), nsys, n, nrhs, (int)scr,
                                   (int)rest, (int)a, a_global ? ws.as<double>() : nullptr);
    pb_count_launch_();
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(X, dX.p, out_n * sizeof(double), cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaMemcpyAsync(ok, dok.p, (size_t)nsys * sizeof(int32_t), cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    return PB_OK;
}

extern "C" int pb_local_solve_batch(int cfg, int a_global, int64_t nsys, int n, int nrhs, const double *A, double *X,
                                    int32_t *ok) {
    int max_n = 0, max_w = 0;
    if (pb_solver_limits(cfg, nullptr, &max_n, &max_w)) return PB_EINVAL;
    if (n < 1 || nrhs < 1 || nsys < 0) return pb_fail_(PB_EINVAL, "need n >= 1, nrhs >= 1, nsys >= 0");
    if (n > max_n || (int64_t)n + nrhs > max_w)
        return pb_fail_(PB_EINVAL, "system of order " + std::to_string(n) + " with " + std::to_string(nrhs) +
                                       " right-hand sides exceeds solver configuration " + std::to_string(cfg));
    if ((int64_t)n * ((n + nrhs) | 1) > INT_MAX) return pb_fail_(PB_EINVAL, "system too large");
    if (nsys > 0 && (!A || !X || !ok)) return pb_fail_(PB_EINVAL, "null pointer");
    const bool g = a_global != 0;
    switch (cfg) {
        case 0: return solve_batch<Cfg0>(cfg, g, nsys, n, nrhs, A, X, ok);
        case 1: return solve_batch<Cfg1>(cfg, g, nsys, n, nrhs, A, X, ok);
        case 2: return solve_batch<Cfg2>(cfg, g, nsys, n, nrhs, A, X, ok);
        case 3: return solve_batch<Cfg3>(cfg, g, nsys, n, nrhs, A, X, ok);
        case 4: return solve_batch<Cfg4>(cfg, g, nsys, n, nrhs, A, X, ok);
        case 5: return solve_batch<Cfg5>(cfg, g, nsys, n, nrhs, A, X, ok);
        case 7: return solve_batch<Cfg7>(cfg, g, nsys, n, nrhs, A, X, ok);
        default: return solve_batch<Cfg6>(cfg, g, nsys, n, nrhs, A, X, ok);
    }
}
