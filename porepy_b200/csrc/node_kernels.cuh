// node_kernels.cuh -- per-interaction-region assembly routines (MPFA; MPSA/Biot in
// mpsa_node.cuh).  One TEAM of threads (a warp, or a CTA for large regions) owns one grid
// node: it gathers the sub-cell geometry and tensors, builds ONE small dense system in shared
// memory, solves it for all right-hand sides by Gauss-Jordan elimination with partial
// pivoting (FP64), and scatter-adds the sub-face rows into the face-indexed CSR value arrays.
//
// Formulation (DESIGN.md "Local systems"): the reference solves for the sub-cell gradients
// g_K (order nd*#subcells, numerics/fv/mpfa.py:926-1045).  Pressure continuity
// d_{K,f}.g_K + p_K = pbar_f holds exactly at the continuity points, and every sub-cell has
// exactly nd sub-faces at the node (_fvutils.py:735), so g_K = D_K^{-1}(pbar_{F_K} - p_K 1) and
// the only unknowns left are the continuity-point pressures pbar_f, one per sub-face: a system
// of order #subfaces (12 instead of 24 on interior Cartesian nodes, 8x fewer LU flops).  The
// flux-continuity / Neumann / Robin / Dirichlet rows and all right-hand sides are those of the
// reference (mpfa.py:997, 1080-1105, 1414-1578, 1274-1307) with g_K substituted.
//
// The routines are written against a small Team interface so that the identical source also
// compiles for the host with a 1-thread team; tests/emu uses that (test infrastructure only,
// never loaded by the product) to check the arithmetic against the oracle without a GPU.
#pragma once
#include <cmath>
#include <cstdint>

#include "views.hpp"

namespace pb {

// ------------------------------------------------------------------------------------
// teams
// ------------------------------------------------------------------------------------
struct CpuTeam {
    PB_HD int tid() const { return 0; }
    PB_HD int size() const { return 1; }
    PB_HD int lanes() const { return 1; }
    PB_HD int warp() const { return 0; }
    PB_HD int nwarps() const { return 1; }
    PB_HD int lane() const { return 0; }
    PB_HD void sync() const {}
    PB_HD void warp_argmax(double &, int &) const {}
};

#if defined(__CUDACC__)
template <int TEAM>
struct GpuTeam {
    // TEAM == 32: several teams per CTA, one warp each (__syncwarp);
    // TEAM  > 32: the CTA is the team (__syncthreads)
    __device__ __forceinline__ int tid() const { return TEAM == 32 ? (threadIdx.x & 31) : threadIdx.x; }
    __device__ __forceinline__ int size() const { return TEAM; }
    __device__ __forceinline__ int lanes() const { return 32; }
    __device__ __forceinline__ int warp() const { return TEAM == 32 ? 0 : (threadIdx.x >> 5); }
    __device__ __forceinline__ int nwarps() const { return TEAM / 32; }
    __device__ __forceinline__ int lane() const { return threadIdx.x & 31; }
    __device__ __forceinline__ void sync() const {
        if (TEAM == 32) __syncwarp(); else __syncthreads();
    }
    // max of v over the 32 lanes of the calling warp, with its index; result in all lanes
    __device__ __forceinline__ void warp_argmax(double &v, int &i) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double v2 = __shfl_xor_sync(0xffffffffu, v, o);
            int i2 = __shfl_xor_sync(0xffffffffu, i, o);
            if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
        }
    }
};
#endif

PB_HD void red_add(double *p, double v) {
#if defined(__CUDA_ARCH__)
    atomicAdd(p, v);  // result unused -> RED.E.ADD.F64 to L2
#else
    *p += v;
#endif
}

// add into the team's shared staging area from concurrent threads
PB_HD void team_add(double *p, double v) {
#if defined(__CUDA_ARCH__)
    atomicAdd(p, v);
#else
    *p += v;
#endif
}

PB_HD void flag_singular(int *err, int64_t node) {
#if defined(__CUDA_ARCH__)
    atomicMin(err, (int)node);
#else
    if ((int)node < *err) *err = (int)node;
#endif
}

// ------------------------------------------------------------------------------------
// Gauss-Jordan with partial pivoting on the augmented matrix A (n rows, row stride W, the
// first n columns are the system, the remaining nrhs the right-hand sides).  Rows are not
// swapped physically: rowidx[p] is the physical row holding pivot p.  On return
// X(p, c) = A[rowidx[p]*W + n + c] is the solution (already divided by the pivot).
// Replaces the dense np.linalg.inv per block of invert_diagonal_blocks
// (numerics/linalg/matrix_operations.py:1310-1371).
// ------------------------------------------------------------------------------------
template <class Team>
PB_HD bool gauss_jordan(Team &t, double *A, int n, int W, int nrhs, int *rowidx, double *ipiv) {
    bool ok = true;
    for (int p = 0; p < n; ++p) {
        if (t.warp() == 0) {
            double best = -1.0;
            int bi = p;
            for (int i = p + t.lane(); i < n; i += t.lanes()) {
                double v = fabs(A[rowidx[i] * W + p]);
                if (v > best) { best = v; bi = i; }
            }
            t.warp_argmax(best, bi);
            if (t.lane() == 0) {
                int r = rowidx[bi];
                rowidx[bi] = rowidx[p];
                rowidx[p] = r;
                // NaN-safe: !(best > 0) also catches NaN
                ipiv[p] = (best > 0.0) ? 1.0 / A[r * W + p] : 0.0;
            }
        }
        t.sync();
        const int pr = rowidx[p];
        const double inv = ipiv[p];
        if (inv == 0.0 || !(inv == inv)) ok = false;
        const int c0 = p + 1;
        const int wend = n + nrhs;
        for (int li = t.warp(); li < n; li += t.nwarps()) {
            if (li == p) continue;
            const int ri = rowidx[li];
            const double f = A[ri * W + p] * inv;
            if (f == 0.0) continue;
            for (int c = c0 + t.lane(); c < wend; c += t.lanes()) A[ri * W + c] -= f * A[pr * W + c];
        }
        t.sync();
    }
    // divide the right-hand sides by the pivots
    for (int p = t.warp(); p < n; p += t.nwarps()) {
        const int pr = rowidx[p];
        const double inv = ipiv[p];
        for (int c = n + t.lane(); c < n + nrhs; c += t.lanes()) A[pr * W + c] *= inv;
    }
    t.sync();
    return ok;
}

// Solver policies.  `solve` leaves X(p, c) = A[rowidx[p]*W + n + c].
struct SmemGJ {
    // Gauss-Jordan directly on the shared (or global) memory copy of A: works for any size
    // and on the host (kernel emulation); the slow path on the GPU.
    static constexpr int team = 256;
    static constexpr int min_blocks = 1;
    static PB_HD int64_t scratch_doubles(int n) { return n; }
    template <class Team>
    static PB_HD bool solve(Team &t, double *A, int n, int W, int nrhs, int *rowidx, double *scratch) {
        return gauss_jordan(t, A, n, W, nrhs, rowidx, scratch);
    }
};

#if defined(__CUDACC__)
// Register-tiled Gauss-Jordan.  The team is TR warps; warp w owns the rows {w + TR*x}, lane l
// the columns {l + 32*y}: every thread keeps an RL x CL tile of the augmented matrix in
// registers for the whole elimination (cyclic ownership keeps all threads busy while the
// active part shrinks).  Per pivot step p:
//   A  the lane that owns column p dumps it (RL values per warp) to shared memory, together
//      with |value| of the rows that have not been pivots yet;            -- barrier --
//   B  every warp finds the pivot row from the dumped column (<= 4 shared loads per lane and
//      one packed-key warp arg-max); the owner warp scales the pivot row and posts it (one
//      value per owned column);                                            -- barrier --
//   C  rank-1 update of the tile: the row factors are broadcast shared loads of the dumped
//      column, RL*CL FMAs against RL + CL shared loads.
// The column dump is double-buffered (step p+1's dump may overtake slow readers of step p).
// The loop over 32-column blocks is unrolled so that all register indices are compile-time.
// Requires n <= TR*RL <= 255 and n + nrhs <= 32*CL.
#define PB_GJ_CASE(X)                                                  \
    case X:                                                            \
        if constexpr (X < RL) {                                        \
            _Pragma("unroll") for (int y = py; y < CL; ++y) {          \
                a[X][y] *= inv;                                        \
                pw[tj + 32 * y] = a[X][y];                             \
            }                                                          \
        }                                                              \
        break;

template <int TR, int RL, int CL, int MINB>
struct RegGJ {
    static_assert(RL <= 18, "extend the PB_GJ_CASE list");
    static_assert(TR * RL <= 255, "row index must fit the 8-bit key field");
    static constexpr int team = TR * 32;
    static constexpr int min_blocks = MINB;
    static constexpr int max_n = TR * RL;
    static constexpr int max_w = 32 * CL;
    static constexpr int NP = ((max_n + 31) / 32) * 32;  // padded column length
    static __host__ __device__ constexpr int64_t scratch_doubles_c() { return 32 * CL + 4 * NP + 2; }
    static PB_HD int64_t scratch_doubles(int) { return scratch_doubles_c(); }

    template <class Team>
    static __device__ __forceinline__ bool solve(Team &t, double *A, int n, int W, int nrhs,
                                                 int *rowidx, double *scratch) {
        const int ti = t.warp(), tj = t.lane();
        const int wend = n + nrhs;
        double a[RL][CL];
#pragma unroll
        for (int x = 0; x < RL; ++x)
#pragma unroll
            for (int y = 0; y < CL; ++y) {
                const int r = ti + TR * x, c = tj + 32 * y;
                a[x][y] = (r < n && c < wend) ? A[r * W + c] : 0.0;
            }
        double *pw = scratch;             // [32*CL]  scaled pivot row
        double *col = pw + 32 * CL;       // [2][NP]  pivot column (factors), by physical row
        double *cab = col + 2 * NP;       // [2][NP]  |pivot column| of rows still unused, else 0
        for (int i = t.tid(); i < 4 * NP; i += t.size()) col[i] = 0.0;
        t.sync();
        unsigned used = 0;  // bit x: my row x has been a pivot row
        bool ok = true;
        // dump of column 0 (step 0's phase A); later dumps are issued as look-ahead inside phase C
        if (tj == 0) {
#pragma unroll
            for (int x = 0; x < RL; ++x) {
                col[ti + TR * x] = a[x][0];
                cab[ti + TR * x] = fabs(a[x][0]);
            }
        }
#pragma unroll
        for (int py = 0; py < CL; ++py) {
            if (py * 32 >= n) break;
            for (int pl = 0; pl < 32; ++pl) {
                const int p = py * 32 + pl;
                if (p >= n) break;
                const int buf = p & 1;
                double *fc = col + buf * NP;
                double *ca = cab + buf * NP;
                t.sync();
                // B: pivot = arg max |column| over unused rows (every warp redundantly)
                unsigned long long key = 0ull;
#pragma unroll
                for (int q = 0; q < NP / 32; ++q) {
                    unsigned long long k = (unsigned long long)__double_as_longlong(ca[tj + 32 * q]);
                    k = (k & ~0xFFull) | (unsigned)(tj + 32 * q);
                    key = k > key ? k : key;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, o);
                    key = k2 > key ? k2 : key;
                }
                if ((key >> 8) == 0ull) { ok = false; break; }  // zero column: uniform over the team
                const int pr = (int)(key & 0xFFull);
                // NaN / Inf rank above every finite magnitude, so a non-finite entry in the column becomes the pivot:
                // refuse the system as the other solvers do (the value is read from shared memory by every thread)
                if (!isfinite(fc[pr])) { ok = false; break; }
                const int xpiv = (ti == pr % TR) ? pr / TR : -1;
                if (xpiv >= 0) {
                    const double inv = 1.0 / fc[pr];
                    switch (xpiv) {
                        PB_GJ_CASE(0) PB_GJ_CASE(1) PB_GJ_CASE(2) PB_GJ_CASE(3) PB_GJ_CASE(4)
                        PB_GJ_CASE(5) PB_GJ_CASE(6) PB_GJ_CASE(7) PB_GJ_CASE(8) PB_GJ_CASE(9)
                        PB_GJ_CASE(10) PB_GJ_CASE(11) PB_GJ_CASE(12) PB_GJ_CASE(13) PB_GJ_CASE(14)
                        PB_GJ_CASE(15) PB_GJ_CASE(16) PB_GJ_CASE(17)
                        default: break;
                    }
                    used |= 1u << xpiv;
                    if (tj == 0) rowidx[p] = pr;
                }
                t.sync();
                // C1: rank-1 update of the pivot's own 32-column block (holds column p+1 as well)
                double pv[CL];
#pragma unroll
                for (int y = py; y < CL; ++y) pv[y] = pw[tj + 32 * y];
                double fx[RL];
#pragma unroll
                for (int x = 0; x < RL; ++x) {
                    fx[x] = (x != xpiv) ? fc[ti + TR * x] : 0.0;
                    if (tj > pl) a[x][py] -= fx[x] * pv[py];
                }
                // A' (look-ahead): dump column p+1 for the next step when it is in this block
                const bool la = (pl < 31) && (p + 1 < n);
                double *fc2 = col + (buf ^ 1) * NP;
                double *ca2 = cab + (buf ^ 1) * NP;
                if (la && tj == pl + 1) {
#pragma unroll
                    for (int x = 0; x < RL; ++x) {
                        const double v = a[x][py];
                        fc2[ti + TR * x] = v;
                        ca2[ti + TR * x] = ((used >> x) & 1u) ? 0.0 : fabs(v);
                    }
                }
                // C2: the remaining column blocks
#pragma unroll
                for (int x = 0; x < RL; ++x) {
                    if (fx[x] != 0.0) {
#pragma unroll
                        for (int y = py + 1; y < CL; ++y) a[x][y] -= fx[x] * pv[y];
                    }
                }
                if (!la && p + 1 < n && tj == 0) {  // first column of the next block
#pragma unroll
                    for (int x = 0; x < RL; ++x) {
                        const double v = a[x][py + 1 < CL ? py + 1 : py];
                        fc2[ti + TR * x] = v;
                        ca2[ti + TR * x] = ((used >> x) & 1u) ? 0.0 : fabs(v);
                    }
                }
                if (TR == 1) t.sync();
            }
            if (!ok) break;
        }
        t.sync();
        if (!ok) return false;
#pragma unroll
        for (int x = 0; x < RL; ++x) {
            const int r = ti + TR * x;
            if (r < n) {
#pragma unroll
                for (int y = 0; y < CL; ++y) {
                    const int c = tj + 32 * y;
                    if (c >= n && c < wend) A[r * W + c] = a[x][y];
                }
            }
        }
        t.sync();
        return true;
    }
};
#endif

#if defined(__CUDACC__)
// Blocked Gauss-Jordan on FP64 tensor cores (DMMA, mma.sync.m8n8k4.f64 -- tcgen05 has no FP64
// kind).  The augmented matrix lives in registers as 8x8 accumulator tiles: warp w owns row
// tile w (8 rows) and all NCT column tiles (2 doubles per lane and tile).  Pivots are taken four
// at a time (a panel = half a column tile):
//   S1  every warp dumps its 8x4 slice of the panel to shared memory;            -- barrier --
//   S2  warp 0 runs partial pivoting on the n x 4 panel in registers (packed-key warp arg-max
//       per column), inverts the 4x4 pivot block A11 and publishes rows + A11^-1;  -- barrier --
//   S3  the owners post the four raw pivot rows;                                  -- barrier --
//   S4  all threads form R = A11^-1 * (pivot rows), one column each;              -- barrier --
//   S5  block update  A22 -= A21 * R : the A fragment (8x4 slice of the panel) comes from the
//       warp's own tile by two shuffles, the B fragment is one conflict-free shared load, one
//       DMMA per tile; the pivot rows are overwritten with R.
// Block Gauss-Jordan identity: [A11 A12; A21 A22] -> [I A11^-1 A12; 0 A22 - A21 A11^-1 A12].
// 4 barriers per 4 pivots instead of 8, and 256 FMAs per issued math instruction instead of 32.
__device__ __forceinline__ void pb_dmma(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1])
                 : "d"(a), "d"(b));
}

template <int NW, int RT, int NCT, int MINB>
struct TileGJ {
    // NW warps; warp w owns the row tiles {w + NW*rt, rt < RT} (8 rows each) and all NCT column
    // tiles.  (A variant with a dedicated panel warp factorizing panel q+1 during the block update
    // of panel q was measured no faster on B200 and is not kept: profiles/r01_notes.md.)
    static_assert(NCT % 2 == 0, "padded row stride must be 4 mod 16");
    static constexpr int team = NW * 32;
    static constexpr int min_blocks = MINB;
    static constexpr int NRT = NW * RT;
    static constexpr int max_n = NRT * 8;
    static constexpr int max_w = NCT * 8;
    static constexpr int NP = ((max_n + 31) / 32) * 32;  // rows of the panel buffer
    static constexpr int NI = NP / 32;
    static constexpr int WP = NCT * 8 + 4;               // stride of the pivot-row buffers
    static_assert(NP <= 256, "row index must fit the 8-bit key field");
    static_assert(NI <= 8, "extend the PB_PICK list");
    static __host__ __device__ constexpr int64_t scratch_doubles_c() {
        return NP * 4 + 2 * 4 * WP + 16 * (NW + 1) + (8 + NP) / 2 + 4;
    }
    static PB_HD int64_t scratch_doubles(int) { return scratch_doubles_c(); }

    // partial pivoting on the n x 4 panel held in P0 (one warp); publishes the pivot rows, the
    // inverse of the 4x4 pivot block and the bookkeeping
    // 4x4 inverse of the pivot block, one element per lane (lane = 4*row + col; lanes >= 16 mirror
    // lanes 0..15), Gauss-Jordan in the given row order, shuffles for the broadcasts.
    // Returns max |inverse entry| (inf / nan when the block is not invertible in that order).
    static __device__ __forceinline__ double invert_block(int l, double m, double &iv) {
        const int mj = (l >> 2) & 3, mi = l & 3;
        iv = (mi == mj) ? 1.0 : 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double inv = __drcp_rn(__shfl_sync(0xffffffffu, m, k * 4 + k));
            if (mj == k) { m *= inv; iv *= inv; }
            const double mk = __shfl_sync(0xffffffffu, m, k * 4 + mi);
            const double ik = __shfl_sync(0xffffffffu, iv, k * 4 + mi);
            const double f = __shfl_sync(0xffffffffu, m, mj * 4 + k);
            if (mj != k) { m -= f * mk; iv -= f * ik; }
        }
        // max |entry| through one redux.sync on the float-rounded magnitude (monotone bit pattern for
        // non-negative floats; inf and nan map above every finite value) instead of four rounds of
        // 64-bit shuffles: the result is only compared with the growth threshold
        const unsigned key = __reduce_max_sync(0xffffffffu, __float_as_uint(fabsf((float)iv)) & 0x7FFFFFFFu);
        return (key >= 0x7F800000u) ? __longlong_as_double(0x7FF0000000000000LL) : (double)__uint_as_float(key);
    }

    // Pivot choice for one panel (one warp).  Fast path: the panel's natural rows p0..p0+3 (the
    // "diagonal block") are accepted as pivot block when they are unused and the inverse of the
    // block is tame (max |entry| <= kGrowth; rows are scaled to unit 1-norm) -- threshold block
    // pivoting: no search, ~6x shorter dependent chain.  Otherwise: partial pivoting on the n x 4
    // panel (packed-key warp arg-max per column).  Publishes the pivot rows, A11^-1 and bookkeeping.
    static constexpr double kGrowth = 64.0;
    // fast-path test, executed by EVERY warp redundantly (same inputs -> same decision): no
    // serialized section and no extra barrier on the common path
    static __device__ __forceinline__ bool try_diagonal_block(int l, const double *P0, const int *usedf,
                                                              int p0, int pw, double &iv) {
        const int mj = (l >> 2) & 3, mi = l & 3;
        const double m = (mj < pw) ? ((mi < pw) ? P0[(p0 + mj) * 4 + mi] : 0.0) : (mi == mj ? 1.0 : 0.0);
        // a used row, or a non-finite entry (a block holding an Inf can have a finite, tame computed inverse)
        const bool bad = ((mj < pw) && (usedf[p0 + mj] != 0)) || !isfinite(m);
        const bool any_bad = __any_sync(0xffffffffu, bad);
        const double growth = invert_block(l, m, iv);
        return !any_bad && growth <= kGrowth;
    }

    template <bool TRY_FAST>
    static __device__ __forceinline__ void factor_panel(int l, const double *P0, int *usedf, int *prs,
                                                        double *Ainv, int *rowidx, int p0, int pw) {
        const int mj = (l >> 2) & 3, mi = l & 3;
        int mypr[4] = {-1, -1, -1, -1};
        bool sing = false;
        double iv;
        // ---- fast path
        if (TRY_FAST) {
            const bool bad = (mj < pw) && (usedf[p0 + mj] != 0);
            const bool any_used = __any_sync(0xffffffffu, bad);
            double m = (mj < pw) ? ((mi < pw) ? P0[(p0 + mj) * 4 + mi] : 0.0) : (mi == mj ? 1.0 : 0.0);
            const double growth = invert_block(l, m, iv);
            if (!any_used && growth <= kGrowth) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < pw) mypr[j] = p0 + j;
                if (l < 16) Ainv[l] = iv;
                if (l == 0) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        prs[j] = mypr[j];
                        if (mypr[j] >= 0) { usedf[mypr[j]] = 1; rowidx[p0 + j] = mypr[j]; }
                    }
                }
                return;
            }
        }
        // ---- partial pivoting on the panel
        double v[NI][4];
        bool us[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int rr = l + 32 * i;
#pragma unroll
            for (int j = 0; j < 4; ++j) v[i][j] = P0[rr * 4 + j];
            us[i] = usedf[rr] != 0;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < pw && !sing) {
                // pivot choice on the high word of |v| (sign, exponent and 20 mantissa bits; the low byte is
                // replaced by the row): one redux.sync instead of five 64-bit shuffle rounds.  The high word is
                // monotone over the whole double range; a float-rounded magnitude flushes everything below 1e-45
                // to zero, which refused regular systems with graded columns.  Zero only for |v| < 2^-1034.
                unsigned key = 0u;
#pragma unroll
                for (int i = 0; i < NI; ++i) {
                    unsigned k = ((unsigned)(__double_as_longlong(fabs(v[i][j])) >> 32) & 0x7FFFFF00u) |
                                 (unsigned)(l + 32 * i);
                    key = (!us[i] && k > key) ? k : key;
                }
                key = __reduce_max_sync(0xffffffffu, key);
                if ((key >> 8) == 0u) { sing = true; }
                else {
                    const int pr = (int)(key & 0xFFu);
                    mypr[j] = pr;
                    const int ol = pr & 31, os = pr >> 5;
                    double prow[4];
                    {
                        double x[4] = {0.0, 0.0, 0.0, 0.0};
                        switch (os) {  // warp-uniform: a jump instead of NI*4 predicated selects
#define PB_PICK(I)                                                        \
    case I:                                                               \
        if constexpr (I < NI) {                                           \
            x[0] = v[I][0]; x[1] = v[I][1]; x[2] = v[I][2]; x[3] = v[I][3]; \
        }                                                                 \
        break;
                            PB_PICK(0) PB_PICK(1) PB_PICK(2) PB_PICK(3) PB_PICK(4) PB_PICK(5) PB_PICK(6) PB_PICK(7)
#undef PB_PICK
                            default: break;
                        }
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) prow[jj] = __shfl_sync(0xffffffffu, x[jj], ol);
                    }
                    // elimination with the multiplier f / piv.  The panel copy is only used to CHOOSE the
                    // pivots (A11^-1 is formed from the original entries below); a fraction-free update
                    // (v * piv - f * prow) would save the reciprocal but multiplies the copy by a pivot per
                    // step, so a panel of columns of order s reaches s^8 after three steps and underflows
                    const double rp = 1.0 / prow[j];
#pragma unroll
                    for (int i = 0; i < NI; ++i) {
                        const bool me = (l == ol) && (i == os);
                        if (me) us[i] = true;
                        else {
                            const double f = v[i][j] * rp;
#pragma unroll
                            for (int jj = j + 1; jj < 4; ++jj) v[i][jj] -= f * prow[jj];
                        }
                    }
                }
            }
        }
        // A11 = original panel entries of the pivot rows (identity for missing pivots)
        int prj = -1;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j == mj) prj = mypr[j];
        const double m = (prj >= 0) ? ((mi < pw) ? P0[prj * 4 + mi] : 0.0) : (mi == mj ? 1.0 : 0.0);
        const double growth = invert_block(l, m, iv);
        // inf / nan inverse, or a non-finite pivot-block entry (1 / Inf = 0 can leave the computed inverse finite)
        if (!(growth < 1e300) || __any_sync(0xffffffffu, !isfinite(m))) sing = true;
        if (l < 16) Ainv[l] = iv;
        if (l == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                prs[j] = mypr[j];
                if (mypr[j] >= 0) { usedf[mypr[j]] = 1; rowidx[p0 + j] = mypr[j]; }
            }
            if (sing) prs[4] = 1;
        }
    }


    template <class Team>
    static __device__ __forceinline__ bool solve(Team &t, double *A, int n, int W, int nrhs,
                                                 int *rowidx, double *scratch) {
        const int ti = t.warp(), l = t.lane();
        const int gr = l >> 2, gc = (l & 3) * 2;
        const int wend = n + nrhs;
        double c[RT][NCT][2];
#pragma unroll
        for (int rt = 0; rt < RT; ++rt) {
            const int myrow = 8 * (ti + NW * rt) + gr;
#pragma unroll
            for (int tc = 0; tc < NCT; ++tc) {
                const int col = 8 * tc + gc;
                c[rt][tc][0] = (myrow < n && col < wend) ? A[myrow * W + col] : 0.0;
                c[rt][tc][1] = (myrow < n && col + 1 < wend) ? A[myrow * W + col + 1] : 0.0;
            }
        }
        double *P0 = scratch;              // [NP][4]  panel columns
        double *Raw = P0 + NP * 4;         // [4][WP]  raw pivot rows
        double *R = Raw + 4 * WP;          // [4][WP]  A11^-1 * pivot rows
        double *Ainv = R + 4 * WP;         // [NW+1][4][4]: copy 0 = slow-path result, copy 1+w = warp w's own
        int *prs = (int *)(Ainv + 16 * (NW + 1));  // [4] pivot rows of the panel, [4] = singular flag
        int *usedf = prs + 8;              // [NP]
        for (int i = t.tid(); i < NP; i += t.size()) usedf[i] = i < n ? 0 : 1;
        for (int i = t.tid(); i < NP * 4; i += t.size()) P0[i] = 0.0;
        if (t.tid() == 0) prs[4] = 0;
        t.sync();
        const int npanel = (n + 3) >> 2;
        bool ok = true;
#pragma unroll
        for (int tcp = 0; tcp < NRT && tcp < NCT; ++tcp) {
            for (int half = 0; half < 2; ++half) {
                const int q = 2 * tcp + half;
                if (q >= npanel || !ok) break;
                const int p0 = 4 * q;
                const int pw = (n - p0) < 4 ? (n - p0) : 4;
                // S1: dump my 8x4 slices of the panel; the owners of the panel's natural rows
                // p0..p0+3 post them as raw pivot rows right away (speculation for the fast path)
                if (((l & 3) >> 1) == half) {
                    const int j0 = 2 * (l & 1);
#pragma unroll
                    for (int rt = 0; rt < RT; ++rt) {
                        const int myrow = 8 * (ti + NW * rt) + gr;
                        P0[myrow * 4 + j0] = c[rt][tcp][0];
                        P0[myrow * 4 + j0 + 1] = c[rt][tcp][1];
                    }
                }
                int myp[RT];
#pragma unroll
                for (int rt = 0; rt < RT; ++rt) {
                    const int myrow = 8 * (ti + NW * rt) + gr;
                    const int j = myrow - p0;
                    myp[rt] = (j >= 0 && j < pw) ? j : -1;
                    if (myp[rt] >= 0) {
#pragma unroll
                        for (int tc = tcp; tc < NCT; ++tc) {
                            Raw[myp[rt] * WP + 8 * tc + gc] = c[rt][tc][0];
                            Raw[myp[rt] * WP + 8 * tc + gc + 1] = c[rt][tc][1];
                        }
                    }
                }
                t.sync();
                // S2: every warp tests the diagonal block (threshold block pivoting)
                double iv;
                const bool fast = try_diagonal_block(l, P0, usedf, p0, pw, iv);
                const double *ainv = Ainv;  // slow path: warp 0's result, published behind a barrier
                if (fast) {
                    double *mine = Ainv + 16 * (ti + 1);  // private copy: no cross-warp sharing
                    if (l < 16) mine[l] = iv;
                    __syncwarp();
                    ainv = mine;
                } else {
                    // rare: partial pivoting on the panel by warp 0, then the owners re-post the rows
                    t.sync();  // all warps have read usedf / P0 for the test
                    if (ti == 0) factor_panel<false>(l, P0, usedf, prs, Ainv, rowidx, p0, pw);
                    t.sync();
                    ok = prs[4] == 0;  // uniform over the team
                    if (!ok) break;
#pragma unroll
                    for (int rt = 0; rt < RT; ++rt) {
                        const int myrow = 8 * (ti + NW * rt) + gr;
                        myp[rt] = -1;
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (prs[j] == myrow) myp[rt] = j;
                        if (myp[rt] >= 0) {
#pragma unroll
                            for (int tc = tcp; tc < NCT; ++tc) {
                                Raw[myp[rt] * WP + 8 * tc + gc] = c[rt][tc][0];
                                Raw[myp[rt] * WP + 8 * tc + gc + 1] = c[rt][tc][1];
                            }
                        }
                    }
                    t.sync();
                }
                // S4: R = A11^-1 * Raw, one column per thread
                for (int col = 8 * tcp + t.tid(); col < NCT * 8; col += t.size()) {
                    double raw[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) raw[i] = (i < pw) ? Raw[i * WP + col] : 0.0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        double x = 0.0;
#pragma unroll
                        for (int i = 0; i < 4; ++i) x += ainv[j * 4 + i] * raw[i];
                        R[j * WP + col] = (j < pw) ? x : 0.0;
                    }
                }
                t.sync();
                // S5: A22 -= A21 * R  (one DMMA per tile), pivot rows <- R
                if (fast && t.tid() < pw) {  // bookkeeping of the fast path (after every warp's test)
                    usedf[p0 + t.tid()] = 1;
                    rowidx[p0 + t.tid()] = p0 + t.tid();
                }
                {
                    const int k = l & 3;
                    const int src = (l & ~3) | (2 * half + (k >> 1));
                    double af[RT];
#pragma unroll
                    for (int rt = 0; rt < RT; ++rt) {
                        const double v0 = __shfl_sync(0xffffffffu, c[rt][tcp][0], src);
                        const double v1 = __shfl_sync(0xffffffffu, c[rt][tcp][1], src);
                        af[rt] = (k < pw) ? -((k & 1) ? v1 : v0) : 0.0;
                    }
                    const double *rb = R + k * WP + (l >> 2);
#pragma unroll
                    for (int tc = tcp; tc < NCT; ++tc) {
                        const double bf = rb[8 * tc];
#pragma unroll
                        for (int rt = 0; rt < RT; ++rt) pb_dmma(c[rt][tc], af[rt], bf);
                    }
#pragma unroll
                    for (int rt = 0; rt < RT; ++rt)
                        if (myp[rt] >= 0) {
#pragma unroll
                            for (int tc = tcp; tc < NCT; ++tc) {
                                c[rt][tc][0] = R[myp[rt] * WP + 8 * tc + gc];
                                c[rt][tc][1] = R[myp[rt] * WP + 8 * tc + gc + 1];
                            }
                        }
                }
            }
        }
        t.sync();
        if (!ok) return false;
#pragma unroll
        for (int rt = 0; rt < RT; ++rt) {
            const int myrow = 8 * (ti + NW * rt) + gr;
#pragma unroll
            for (int tc = 0; tc < NCT; ++tc) {
                const int col = 8 * tc + gc;
                if (myrow < n) {
                    if (col >= n && col < wend) A[myrow * W + col] = c[rt][tc][0];
                    if (col + 1 >= n && col + 1 < wend) A[myrow * W + col + 1] = c[rt][tc][1];
                }
            }
        }
        t.sync();
        return true;
    }
};
#endif

// ------------------------------------------------------------------------------------
// small dense inverse of the nd x nd matrix of distance vectors (rows d_m)
// ------------------------------------------------------------------------------------
#if defined(__CUDACC__)
__device__ __forceinline__ void pb_prefetch_l2(const void *p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
#endif

template <int ND>
PB_HD bool invert_small(const double (&D)[ND][ND], double (&E)[ND][ND]);

template <>
PB_HD bool invert_small<2>(const double (&D)[2][2], double (&E)[2][2]) {
    double det = D[0][0] * D[1][1] - D[0][1] * D[1][0];
    if (det == 0.0 || !(det == det)) return false;
    double id = 1.0 / det;
    E[0][0] = D[1][1] * id; E[0][1] = -D[0][1] * id;
    E[1][0] = -D[1][0] * id; E[1][1] = D[0][0] * id;
    return true;
}

template <>
PB_HD bool invert_small<3>(const double (&D)[3][3], double (&E)[3][3]) {
    double c00 = D[1][1] * D[2][2] - D[1][2] * D[2][1];
    double c01 = D[1][2] * D[2][0] - D[1][0] * D[2][2];
    double c02 = D[1][0] * D[2][1] - D[1][1] * D[2][0];
    double det = D[0][0] * c00 + D[0][1] * c01 + D[0][2] * c02;
    if (det == 0.0 || !(det == det)) return false;
    double id = 1.0 / det;
    E[0][0] = c00 * id;
    E[1][0] = c01 * id;
    E[2][0] = c02 * id;
    E[0][1] = (D[0][2] * D[2][1] - D[0][1] * D[2][2]) * id;
    E[1][1] = (D[0][0] * D[2][2] - D[0][2] * D[2][0]) * id;
    E[2][1] = (D[0][1] * D[2][0] - D[0][0] * D[2][1]) * id;
    E[0][2] = (D[0][1] * D[1][2] - D[0][2] * D[1][1]) * id;
    E[1][2] = (D[0][2] * D[1][0] - D[0][0] * D[1][2]) * id;
    E[2][2] = (D[0][0] * D[1][1] - D[0][1] * D[1][0]) * id;
    return true;
}

// ------------------------------------------------------------------------------------
// MPFA
// ------------------------------------------------------------------------------------
// doubles of shared memory one team needs for a node with the given counts
PB_HD int mpfa_width(int nd, int nsf, int nsc, int nb) { return (nsf + nsc + nb + nd * nsc) | 1; }
PB_HD int64_t mpfa_A_doubles(int nd, int nsf, int nsc, int nb) {
    return (int64_t)nsf * mpfa_width(nd, nsf, nsc, nb);
}
// everything but A and the solver scratch
PB_HD int64_t mpfa_rest_doubles(int nd, int nsf, int nsc, int nb) {
    (void)nb;
    int64_t d = 2 * (int64_t)nsc * nd * nd + 2 * (int64_t)nsf;
    int64_t ints = nsc + 5 * (int64_t)nsf + (int64_t)nsc * nd;
    return d + (ints + 1) / 2 + 2;
}

template <int ND, class Solver, class Team>
PB_HD void mpfa_node(Team &t, const PlanView &P, const GeoView &G, const MpfaParams &prm,
                     const MpfaOut &o, int64_t s, double *A, double *smd, double *scratch, int *err) {
    const int sc0 = P.node_sc_ptr[s], nsc = P.node_sc_ptr[s + 1] - sc0;
    const int sf0 = P.node_sf_ptr[s], nsf = P.node_sf_ptr[s + 1] - sf0;
    const int nb = P.node_nb[s];
    if (nsf == 0) return;
    const int nrhs = nsc + nb + ND * nsc;
    const int W = (nsf + nrhs) | 1;
    const int64_t nf = P.nf, nc = P.nc, nn = P.nn;
    double *Tk = smd;
    double *Rk = Tk + nsc * ND * ND;
    double *invmf = Rk + nsc * ND * ND;
    double *robw = invmf + nsf;
    int *cell = (int *)(robw + nsf);
    int *face = cell + nsc;
    int *sides = face + nsf;
    int *bloc = sides + nsf;
    int *bcu = bloc + nsf;
    int *rowidx = bcu + nsf;
    int *slot = rowidx + nsf;

    // ---- phase 1: stage the node's index lists, zero the system
    for (int k = t.tid(); k < nsc; k += t.size()) cell[k] = P.sc_cell[sc0 + k];
    for (int i = t.tid(); i < nsc * ND; i += t.size()) slot[i] = P.slot_sf[(int64_t)sc0 * ND + i];
    for (int u = t.tid(); u < nsf; u += t.size()) {
        const int f = P.sf_face[sf0 + u];
        face[u] = f;
        sides[u] = (int)P.sf_sides[sf0 + u];
        const int bl = P.sf_bloc[sf0 + u];
        bloc[u] = (bl == 0xFFFF) ? -1 : bl;
        const double im = 1.0 / (double)(P.fn_indptr[f + 1] - P.fn_indptr[f]);
        invmf[u] = im;
        int code = 0;
        if (bl != 0xFFFF) {
            code = prm.bc[f];
            if (code == 0) code = 2;  // boundary face without a flag: Neumann (params/bc.py:130-140)
        }
        bcu[u] = code;
        robw[u] = (code == 3 && prm.robw) ? prm.robw[f] * G.farea[f] * im : 0.0;
        rowidx[u] = u;
    }
    for (int i = t.tid(); i < nsf * W; i += t.size()) A[i] = 0.0;
    t.sync();

    // ---- phase 2: per sub-cell  D (distance rows), r = (n/m)^T K,  T = R D^{-1}
    for (int k = t.tid(); k < nsc; k += t.size()) {
        const int64_t c = cell[k];
        double xc[ND], xs[ND], K[ND][ND], D[ND][ND], R[ND][ND], E[ND][ND];
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            xc[i] = G.ccent[i * G.cell_cs + c * G.cell_es];
            xs[i] = G.nodes[i * G.node_cs + s * G.node_es];
#pragma unroll
            for (int j = 0; j < ND; ++j) K[i][j] = prm.perm[(i * 3 + j) * prm.perm_cs + c * prm.perm_es];
        }
#pragma unroll
        for (int m = 0; m < ND; ++m) {
            const int u = slot[k * ND + m] >> 1;
            const int64_t f = face[u];
            const double e = (bloc[u] >= 0) ? 0.0 : prm.eta;  // eta = 0 on boundary faces (_fvutils.py:259-263)
            double nrm[ND];
#pragma unroll
            for (int i = 0; i < ND; ++i) {
                const double xf = G.fcent[i * G.face_cs + f * G.face_es];
                D[m][i] = xf + e * (xs[i] - xf) - xc[i];
                nrm[i] = G.fnorm[i * G.face_cs + f * G.face_es] * invmf[u];
            }
#pragma unroll
            for (int j = 0; j < ND; ++j) {
                double a = 0.0;
#pragma unroll
                for (int i = 0; i < ND; ++i) a += nrm[i] * K[i][j];
                R[m][j] = a;
            }
        }
        if (!invert_small<ND>(D, E)) flag_singular(err, s);
#pragma unroll
        for (int m = 0; m < ND; ++m)
#pragma unroll
            for (int m2 = 0; m2 < ND; ++m2) {
                double a = 0.0;
#pragma unroll
                for (int q = 0; q < ND; ++q) a += R[m][q] * E[q][m2];
                Tk[k * ND * ND + m * ND + m2] = a;
                Rk[k * ND * ND + m * ND + m2] = R[m][m2];
            }
    }
    t.sync();

    // ---- phase 3: one row per sub-face
    for (int u = t.tid(); u < nsf; u += t.size()) {
        double *row = A + (int64_t)u * W;
        const int code = bcu[u];
        if (code == 1) {  // Dirichlet: pbar_u = p_b   (mpfa.py:1547)
            row[u] = 1.0;
            row[nsf + nsc + bloc[u]] = 1.0;
            continue;
        }
        for (int sd = 0; sd < 2; ++sd) {
            const int side = sd == 0 ? (sides[u] & 0xFFFF) : ((sides[u] >> 16) & 0xFFFF);
            if (side == 0xFFFF) continue;
            const int k = side / ND, m = side - k * ND;
            const double sg = (slot[side] & 1) ? -1.0 : 1.0;
            double tau = 0.0;
#pragma unroll
            for (int m2 = 0; m2 < ND; ++m2) {
                const int u2 = slot[k * ND + m2] >> 1;
                const double tt = sg * Tk[k * ND * ND + m * ND + m2];
                row[u2] += tt;
                tau += tt;
            }
            row[nsf + k] += tau;
#pragma unroll
            for (int j = 0; j < ND; ++j) row[nsf + nsc + nb + k * ND + j] += sg * Rk[k * ND * ND + m * ND + j];
        }
        if (code == 2 || code == 3) row[nsf + nsc + bloc[u]] = -invmf[u];  // mpfa.py:1516-1526
        if (code == 3) row[u] -= robw[u];                                   // mpfa.py:869-887
        // row scaling (matrix_operations.py:1880-1906)
        double sum = 0.0;
        for (int c = 0; c < nsf; ++c) sum += fabs(row[c]);
        if (!(sum > 0.0)) { flag_singular(err, s); continue; }
        const double is = 1.0 / sum;
        for (int c = 0; c < nsf + nrhs; ++c) row[c] *= is;
    }
    t.sync();

    // ---- phase 4: solve for all right-hand sides
    if (!Solver::solve(t, A, nsf, W, nrhs, rowidx, scratch)) {
        if (t.tid() == 0) flag_singular(err, s);
        t.sync();
        return;
    }

    // ---- phase 5: sub-face rows -> CSR values.  Columns: [cells | boundary faces | (cell, j)]
    const int32_t *pfc = P.pos_fc + P.posfc_ptr[s];
    const int32_t *pfb = P.pos_fb + P.posfb_ptr[s];
    for (int u = t.warp(); u < nsf; u += t.nwarps()) {
        // The reference takes the flux from the side with the smaller cell index
        // (_fvutils.py:163).  Flux continuity makes both sides give the same number; in the
        // continuity-point formulation the side with the SMALLER transmissibilities is the
        // well-conditioned one (on the high-permeability side the gradient is a difference
        // of nearly equal pressures), so evaluate from that side.
        int side1 = sides[u] & 0xFFFF;
        {
            const int side2 = (sides[u] >> 16) & 0xFFFF;
            if (side2 != 0xFFFF) {
                double n1 = 0.0, n2 = 0.0;
#pragma unroll
                for (int m2 = 0; m2 < ND; ++m2) {
                    n1 += fabs(Tk[side1 * ND + m2]);
                    n2 += fabs(Tk[side2 * ND + m2]);
                }
                if (n2 < n1) side1 = side2;
            }
        }
        const int k1 = side1 / ND, m1 = side1 - k1 * ND;
        const double *T1 = Tk + k1 * ND * ND + m1 * ND;
        const double *R1 = Rk + k1 * ND * ND + m1 * ND;
        const double *xrow[ND];
        double tau1 = 0.0;
#pragma unroll
        for (int m2 = 0; m2 < ND; ++m2) {
            xrow[m2] = A + (int64_t)rowidx[slot[k1 * ND + m2] >> 1] * W + nsf;
            tau1 += T1[m2];
        }
        const double *xu = A + (int64_t)rowidx[u] * W + nsf;
        const double im = invmf[u];
        for (int c = t.lane(); c < nrhs; c += t.lanes()) {
            double fl = 0.0;
#pragma unroll
            for (int m2 = 0; m2 < ND; ++m2) fl -= T1[m2] * xrow[m2][c];
            const double tr = xu[c] * im;
            if (c < nsc) {
                if (c == k1) fl += tau1;
                const int64_t p = pfc[u * nsc + c];
                if (o.flux) red_add(o.flux + p, fl);
                if (o.bpc) red_add(o.bpc + p, tr);
            } else if (c < nsc + nb) {
                const int64_t p = pfb[u * nb + (c - nsc)];
                if (o.bflux) red_add(o.bflux + p, fl);
                if (o.bpf) red_add(o.bpf + p, tr);
            } else {
                const int cc = c - nsc - nb;
                const int k = cc / ND, j = cc - k * ND;
                if (k == k1) fl += R1[j];
                const int64_t p = (int64_t)pfc[u * nsc + k] * ND + j;
                if (o.vs) red_add(o.vs + p, fl);
                if (o.bpvs) red_add(o.bpvs + p, tr);
            }
        }
    }
    t.sync();
}

}  // namespace pb
