// local_blocks.cu -- local-block inverse preconditioner of the contact models' saddle-point Jacobians.
//
// A block layout partitions the rows AND the columns of a square matrix into blocks: block b pairs the rows
// rows[blk_ptr[b] .. blk_ptr[b+1]) with as many columns cols[...] (s_b <= 32).  The factorisation gathers
// B_b = A[rows_b, cols_b] from the device CSR (missing entries are 0) and inverts it by Gauss-Jordan elimination with
// partial pivoting in FP64; B_b^-1 (s_b x s_b, row-major: row i <-> cols_b[i], column j <-> rows_b[j]) goes to
// inv[inv_ptr[b] ..], inv_ptr = prefix sum of s_b^2.  The application is z[cols_b] = B_b^-1 r[rows_b] for all blocks.
//
// One TEAM of lanes per block, TEAM = the power of two >= s_b (4, 8, 16 or 32): the 3-5-wide matrix-cell blocks
// that make up almost all of a layout take 4 or 8 lanes, not a warp.  The caller passes the block ids grouped by team
// size (`order`, with the host array class_ptr[5]: class c = order[class_ptr[c] .. class_ptr[c+1]), c = 0..3 for
// TEAM = 4, 8, 16, 32); one launch per non-empty class.  Lane i of a team owns row i of the augmented [B | I] in
// shared memory.
//
// A block with a non-finite entry, a pivot that is not finite or <= 1e-14 max|B_b|, or an inverse that is not finite
// stops the block and records b in a device word (atomicMin: the first failing block); the host reads it once and
// reports PB_ESINGULAR naming the block.  Nothing is replaced.  Every decision that ends a block's elimination is
// uniform across its team (team votes, the pivot row broadcast from the team's first lane), so the team's lanes never
// leave the warp-synchronous loop apart.
//
// The application takes an optional device flag (`skip`): when it is set the kernel returns at once -- the GMRES loop
// passes its sticky DONE flag, so the steps launched after convergence inside a block of steps cost no block apply.
#include "plan.hpp"

struct CsrView { int64_t nrows, ncols, nnz; int32_t *indptr, *indices; double *data; };
CsrView pb_csr_view_(const pb_csr *a);   // spmv.cu

namespace {

constexpr int kLbThreads = 64;
constexpr double kPivotRel = 1e-14;

template <int TEAM>
__device__ __forceinline__ unsigned team_mask() {
    const int lane = threadIdx.x & 31;
    return TEAM == 32 ? 0xffffffffu : (((1u << TEAM) - 1u) << (lane & ~(TEAM - 1)));
}

template <int TEAM>
__global__ void __launch_bounds__(kLbThreads)
local_block_inv_kernel(int64_t count, const int32_t *__restrict__ order, const int64_t *__restrict__ blk_ptr,
                       const int32_t *__restrict__ rows, const int32_t *__restrict__ cols,
                       const int64_t *__restrict__ inv_ptr, const int32_t *__restrict__ ip,
                       const int32_t *__restrict__ ix, const double *__restrict__ val, double *__restrict__ inv,
                       unsigned long long *__restrict__ err) {
    constexpr int LD = 2 * TEAM + 1;                                 // odd stride: no bank conflicts along a column
    __shared__ double sm[(kLbThreads / TEAM) * TEAM * LD];
    __shared__ int32_t scol[kLbThreads];
    const int lane = threadIdx.x % TEAM, team = threadIdx.x / TEAM;
    double *A = sm + team * TEAM * LD;
    int32_t *tc = scol + team * TEAM;
    const unsigned mask = team_mask<TEAM>();
    const int64_t teams = (int64_t)gridDim.x * (kLbThreads / TEAM);
    for (int64_t q = (int64_t)blockIdx.x * (kLbThreads / TEAM) + team; q < count; q += teams) {
        const int64_t b = order[q];
        const int64_t p0 = blk_ptr[b];
        const int s = (int)(blk_ptr[b + 1] - p0);
        if (lane < s) tc[lane] = cols[p0 + lane];
        __syncwarp(mask);
        // gather row `lane` of B and the identity next to it
        double amax = 0.0;
        bool bad = false;
        if (lane < s) {
            double *Ar = A + lane * LD;
            for (int j = 0; j < 2 * s; ++j) Ar[j] = (j - s == lane) ? 1.0 : 0.0;
            const int64_t row = rows[p0 + lane];
            for (int32_t e = ip[row]; e < ip[row + 1]; ++e) {
                const int32_t c = ix[e];
                for (int j = 0; j < s; ++j)
                    if (tc[j] == c) { Ar[j] += val[e]; break; }
            }
            for (int j = 0; j < s; ++j) {
                amax = fmax(amax, fabs(Ar[j]));
                bad |= !isfinite(Ar[j]);
            }
        }
        for (int o = TEAM / 2; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(mask, amax, o, TEAM));
        bool ok = !__any_sync(mask, bad);                            // a NaN / Inf entry: no inverse
        if (!ok && lane == 0) atomicMin(err, (unsigned long long)b);
        __syncwarp(mask);
        for (int k = 0; k < s && ok; ++k) {
            // pivot: the largest |A[i][k]|, i >= k (ties: the smallest i); a NaN (from overflow in the elimination)
            // ranks as +inf, so that it is chosen, and fails the test below, on every lane
            const bool cand = lane >= k && lane < s;
            const double x = cand ? A[lane * LD + k] : 0.0;
            double pv = cand ? (isnan(x) ? INFINITY : fabs(x)) : -1.0;
            int pi = lane;
            for (int o = TEAM / 2; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(mask, pv, o, TEAM);
                const int oi = __shfl_xor_sync(mask, pi, o, TEAM);
                if (ov > pv || (ov == pv && oi < pi)) { pv = ov; pi = oi; }
            }
            pi = __shfl_sync(mask, pi, 0, TEAM);                      // one pivot row for the whole team
            const double piv = A[pi * LD + k];
            __syncwarp(mask);                                         // every lane has read piv before the swap
            if (!isfinite(piv) || !(fabs(piv) > kPivotRel * amax)) {
                if (lane == 0) atomicMin(err, (unsigned long long)b);
                ok = false;
                break;
            }
            if (pi != k)
                for (int j = lane; j < 2 * s; j += TEAM) {
                    const double t = A[k * LD + j];
                    A[k * LD + j] = A[pi * LD + j];
                    A[pi * LD + j] = t;
                }
            __syncwarp(mask);
            const double rp = 1.0 / piv;
            for (int j = lane; j < 2 * s; j += TEAM) A[k * LD + j] *= rp;
            __syncwarp(mask);
            if (lane < s && lane != k) {
                double *Ar = A + lane * LD;
                const double f = Ar[k];
                if (f != 0.0)
                    for (int j = 0; j < 2 * s; ++j) Ar[j] -= f * A[k * LD + j];
            }
            __syncwarp(mask);
        }
        if (ok) {                                                    // uniform: every lane of the team votes
            bool bad_out = false;
            if (lane < s)
                for (int j = 0; j < s; ++j) bad_out |= !isfinite(A[lane * LD + s + j]);
            if (__any_sync(mask, bad_out)) {
                if (lane == 0) atomicMin(err, (unsigned long long)b);
            } else if (lane < s) {
                double *o = inv + inv_ptr[b] + (int64_t)lane * s;
                const double *Ar = A + lane * LD + s;
                for (int j = 0; j < s; ++j) o[j] = Ar[j];
            }
        }
        __syncwarp(mask);
    }
}

template <int TEAM>
__global__ void __launch_bounds__(kLbThreads)
local_block_apply_kernel(int64_t count, const int32_t *__restrict__ order, const int64_t *__restrict__ blk_ptr,
                         const int32_t *__restrict__ rows, const int32_t *__restrict__ cols,
                         const int64_t *__restrict__ inv_ptr, const double *__restrict__ inv,
                         const double *__restrict__ r, double *__restrict__ z, const double *__restrict__ skip) {
    if (skip && *skip != 0.0) return;
    const int lane = threadIdx.x % TEAM, team = threadIdx.x / TEAM;
    const int64_t teams = (int64_t)gridDim.x * (kLbThreads / TEAM);
    for (int64_t q = (int64_t)blockIdx.x * (kLbThreads / TEAM) + team; q < count; q += teams) {
        const int64_t b = order[q];
        const int64_t p0 = blk_ptr[b];
        const int s = (int)(blk_ptr[b + 1] - p0);
        if (lane < s) {
            const double *m = inv + inv_ptr[b] + (int64_t)lane * s;
            double acc = 0.0;
            for (int j = 0; j < s; ++j) acc += m[j] * r[rows[p0 + j]];
            z[cols[p0 + lane]] = acc;
        }
    }
}

int lb_grid(int64_t count, int team) {
    const int64_t per = kLbThreads / team;
    return (int)std::max<int64_t>(1, std::min<int64_t>((count + per - 1) / per, (int64_t)kSMs * 32));
}

}  // namespace

extern "C" int pb_csr_local_block_inv_dev(const pb_csr *a, int64_t nblocks, const int64_t *blk_ptr, const int32_t *rows,
                                          const int32_t *cols, const int64_t *inv_ptr, const int32_t *order,
                                          const int64_t *class_ptr, double *inv, uint64_t *err_dev, uint64_t stream) {
    if (!a || !blk_ptr || !rows || !cols || !inv_ptr || !order || !class_ptr || !inv || !err_dev)
        return pb_fail_(PB_EINVAL, "pb_csr_local_block_inv_dev: null pointer");
    if (class_ptr[0] != 0 || class_ptr[4] != nblocks)
        return pb_fail_(PB_EINVAL, "pb_csr_local_block_inv_dev: class_ptr does not cover the blocks");
    const CsrView v = pb_csr_view_(a);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *err = (unsigned long long *)err_dev;
    CUDA_TRY(cudaMemsetAsync(err, 0xff, sizeof(unsigned long long), st));
    for (int c = 0; c < 4; ++c) {
        const int64_t cnt = class_ptr[c + 1] - class_ptr[c];
        if (cnt <= 0) continue;
        const int32_t *ord = order + class_ptr[c];
        switch (c) {
            case 0: local_block_inv_kernel<4><<<lb_grid(cnt, 4), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, v.indptr, v.indices, v.data, inv, err); break;
            case 1: local_block_inv_kernel<8><<<lb_grid(cnt, 8), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, v.indptr, v.indices, v.data, inv, err); break;
            case 2: local_block_inv_kernel<16><<<lb_grid(cnt, 16), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, v.indptr, v.indices, v.data, inv, err); break;
            default: local_block_inv_kernel<32><<<lb_grid(cnt, 32), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, v.indptr, v.indices, v.data, inv, err); break;
        }
        pb_count_launch_();
        CUDA_TRY(cudaGetLastError());
    }
    unsigned long long bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, err, sizeof(bad), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (bad != ~0ull)
        return pb_fail_(PB_ESINGULAR, "block " + std::to_string(bad) + " is singular or not finite (a zero or non-finite pivot, entry or inverse)");
    return PB_OK;
}

extern "C" int pb_local_block_apply_dev(int64_t nblocks, const int64_t *blk_ptr, const int32_t *rows, const int32_t *cols,
                                        const int64_t *inv_ptr, const int32_t *order, const int64_t *class_ptr,
                                        const double *inv, const double *r, double *z, const double *skip,
                                        uint64_t stream) {
    if (!blk_ptr || !rows || !cols || !inv_ptr || !order || !class_ptr || !inv || !r || !z)
        return pb_fail_(PB_EINVAL, "pb_local_block_apply_dev: null pointer");
    if (class_ptr[0] != 0 || class_ptr[4] != nblocks)
        return pb_fail_(PB_EINVAL, "pb_local_block_apply_dev: class_ptr does not cover the blocks");
    cudaStream_t st = (cudaStream_t)stream;
    for (int c = 0; c < 4; ++c) {
        const int64_t cnt = class_ptr[c + 1] - class_ptr[c];
        if (cnt <= 0) continue;
        const int32_t *ord = order + class_ptr[c];
        switch (c) {
            case 0: local_block_apply_kernel<4><<<lb_grid(cnt, 4), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, inv, r, z, skip); break;
            case 1: local_block_apply_kernel<8><<<lb_grid(cnt, 8), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, inv, r, z, skip); break;
            case 2: local_block_apply_kernel<16><<<lb_grid(cnt, 16), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, inv, r, z, skip); break;
            default: local_block_apply_kernel<32><<<lb_grid(cnt, 32), kLbThreads, 0, st>>>(cnt, ord, blk_ptr, rows, cols, inv_ptr, inv, r, z, skip); break;
        }
        pb_count_launch_();
        CUDA_TRY(cudaGetLastError());
    }
    return PB_OK;
}
