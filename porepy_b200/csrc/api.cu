// api.cu -- C ABI of libporeb200.so (see include/poreb200.h), device memory management and
// kernel launches.  sm_100a only; there is no CPU path in this library: every compute entry
// point needs a CUDA device and fails with PB_ECUDA otherwise.
#include <cuda_runtime.h>

#include <omp.h>

#include <atomic>
#include <chrono>
#include <thread>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "plan.hpp"
#include <nvtx3/nvToolsExt.h>

// NVTX range for the lifetime of a scope: one range per C-ABI phase (SURVEY.md 5: the reference logs per-phase times,
// models/solution_strategy.py:435-441; here the phases show up in nsys / ncu --nvtx timelines)
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// ------------------------------------------------------------------------------------
// error state
// ------------------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local int64_t g_err_node = -1;
static std::atomic<int64_t> g_launches{0};

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int pb_fail_(int code, const std::string &msg) { return fail(code, msg); }  // for spmv.cu
void pb_count_launch_() { g_launches++; }

DevPool &pb_dev_pool_() {
    static DevPool *pool = new DevPool;   // leaked on purpose: DevBufs of static lifetime may release after exit handlers
    return *pool;
}
extern "C" void pb_device_pool_trim(void) { pb_dev_pool_().trim(); }

extern "C" const char *pb_last_error(void) { return g_err.c_str(); }
// cudaMalloc / cudaFree calls that did not go through the block pool, and the time spent in them (diagnosis of
// the host-side variance of a re-discretization): out = {malloc calls, malloc seconds, free calls, free seconds}
static std::atomic<int64_t> g_alloc_calls[2];
static std::atomic<int64_t> g_alloc_ns[2];
void pb_alloc_stat_(int kind, double seconds) {
    g_alloc_calls[kind & 1]++;
    g_alloc_ns[kind & 1] += (int64_t)(seconds * 1e9);
}
extern "C" void pb_alloc_stats(double *out) {
    if (!out) return;
    out[0] = (double)g_alloc_calls[0].load(); out[1] = 1e-9 * (double)g_alloc_ns[0].load();
    out[2] = (double)g_alloc_calls[1].load(); out[3] = 1e-9 * (double)g_alloc_ns[1].load();
}
extern "C" int64_t pb_last_error_node(void) { return g_err_node; }
void pb_set_error_node_(int64_t node) { g_err_node = node; }
extern "C" int64_t pb_launch_count(void) { return g_launches.load(); }
extern "C" int pb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return -1;
    return n;
}
extern "C" int pb_set_device(int device) {
    CUDA_TRY(cudaSetDevice(device));
    return PB_OK;
}

extern "C" int pb_host_alloc(uint64_t bytes, void **out) {
    if (!out) return fail(PB_EINVAL, "null pointer");
    CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 8, cudaHostAllocDefault));
    return PB_OK;
}
extern "C" void pb_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// ------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------
static int64_t cfg_scratch(int cfg, int n) {
    switch (cfg) {
        case 0: return Cfg0::scratch_doubles_c();
        case 1: return Cfg1::scratch_doubles_c();
        case 2: return Cfg2::scratch_doubles_c();
        case 3: return Cfg3::scratch_doubles_c();
        case 4: return Cfg4::scratch_doubles_c();
        case 5: return Cfg5::scratch_doubles_c();
        case 7: return Cfg7::scratch_doubles_c();
        default: return n;
    }
}

// size_of(nsf, nsc, nb, &n, &w, &a_doubles, &rest_doubles)
template <class F>
static int build_classes(pb_plan *p, std::vector<NodeClass> &out, F size_of) {
    const HostPlan &H = p->H;
    const char *alt = getenv("POREB200_CFG4");
    const bool use7 = alt && strcmp(alt, "reg") == 0;
    // key: cfg*2 + a_global
    std::vector<int32_t> lists[2 * kNumCfg];
    int64_t amax[2 * kNumCfg] = {0}, rmax[2 * kNumCfg] = {0}, smax[2 * kNumCfg] = {0};
    for (int64_t s = 0; s < H.nn; ++s) {
        int nsc = H.node_sc_ptr[s + 1] - H.node_sc_ptr[s];
        int nsf = H.node_sf_ptr[s + 1] - H.node_sf_ptr[s];
        if (nsf == 0) continue;
        if (!p->active.empty() && !p->active[s]) continue;
        int n = 0, w = 0;
        int64_t a = 0, r = 0;
        size_of(nsf, nsc, H.node_nb[s], &n, &w, &a, &r);
        int cfg = 0;
        while (cfg < kCatchAll && (n > kCfg[cfg].max_n || w > kCfg[cfg].max_w)) ++cfg;
        if (cfg == 4 && use7 && n <= kCfg[7].max_n && w <= kCfg[7].max_w) cfg = 7;
        const int64_t scr = cfg_scratch(cfg, n);
        const int tpb = kCfg[cfg].team == 32 ? 4 : 1;
        bool glob = (size_t)(a + r + scr) * 8 * tpb > kMaxSmem;
        if (glob && (size_t)(r + scr) * 8 * tpb > kMaxSmem)
            return fail(PB_ENOTIMPL, "interaction region at node " + std::to_string(s) +
                                         " is too large for this build (" + std::to_string(nsf) +
                                         " sub-faces)");
        int key = cfg * 2 + (glob ? 1 : 0);
        lists[key].push_back((int32_t)s);
        amax[key] = std::max(amax[key], a);
        rmax[key] = std::max(rmax[key], r);
        smax[key] = std::max(smax[key], scr);
    }
    out.clear();
    for (int key = 0; key < 2 * kNumCfg; ++key) {
        if (lists[key].empty()) continue;
        out.emplace_back();
        NodeClass &c = out.back();
        c.cfg = key / 2;
        c.a_global = key & 1;
        c.team = kCfg[c.cfg].team;
        c.n = (int)lists[key].size();
        c.a_doubles = amax[key];
        c.rest_doubles = rmax[key];
        c.scr_doubles = smax[key];
        if (!c.a_global) {
            // the class maxima of A and of the rest may come from different nodes
            const int tpb = c.team == 32 ? 4 : 1;
            if ((size_t)(c.a_doubles + c.rest_doubles + c.scr_doubles) * 8 * tpb > kMaxSmem) c.a_global = true;
        }
        // Launch order = a space-filling (Morton) order of the node coordinates when the geometry is known: the <= m_f
        // nodes of a face are then processed close in time, so the scatter-adds into one face row meet in L2 instead
        // of each paying a DRAM read-modify-write (index order puts the neighbours in the 2nd / 3rd grid direction
        // thousands of regions apart; ncu: 2.9x the algorithmic DRAM traffic).  POREB200_NODE_ORDER=index disables it.
        if (!p->node_key.empty()) {
            const std::vector<uint32_t> &nk = p->node_key;
            std::stable_sort(lists[key].begin(), lists[key].end(), [&](int32_t x, int32_t y) { return nk[x] < nk[y]; });
        }
        if (c.nodes.upload(lists[key], p->stream) != cudaSuccess) return fail(PB_ECUDA, "upload of node list failed");
    }
    return PB_OK;
}

static int build_mpfa_classes(pb_plan *p) {
    const int nd = p->H.nd;
    return build_classes(p, p->mpfa_cls, [&](int nsf, int nsc, int nb, int *n, int *w, int64_t *a, int64_t *r) {
        *n = nsf;
        *w = mpfa_width(nd, nsf, nsc, nb);
        *a = mpfa_A_doubles(nd, nsf, nsc, nb);
        *r = mpfa_rest_doubles(nd, nsf, nsc, nb);
    });
}

// Structural patterns on the device: row r = sorted union over the nodes of row entity r of the
// node's column entities.  One warp per row: gather the (<= CAP) candidates into shared memory,
// bitonic sort, unique.  pass 0 writes the row length, pass 1 the indices.
template <int CAP>
__global__ void pattern_kernel(int64_t nrows, const int32_t *__restrict__ rn_ptr, const int32_t *__restrict__ rn,
                               const int32_t *__restrict__ col_ptr, const int32_t *__restrict__ col_idx,
                               int32_t *__restrict__ counts, const int32_t *__restrict__ indptr,
                               int32_t *__restrict__ indices, int pass, int *overflow) {
    __shared__ int32_t sbuf[8][CAP];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int32_t *buf = sbuf[wib];
    const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = warp; r < nrows; r += nwarps) {
        int total = 0;
        bool over = false;
        for (int q = rn_ptr[r]; q < rn_ptr[r + 1]; ++q) {
            const int s = rn[q];
            const int b = col_ptr[s], len = col_ptr[s + 1] - b;
            if (total + len > CAP) { over = true; break; }
            for (int i = lane; i < len; i += 32) buf[total + i] = col_idx[b + i];
            total += len;
        }
        if (over) {
            if (lane == 0) { atomicExch(overflow, 1); if (pass == 0) counts[r] = 0; }
            continue;
        }
        int P = 1;
        while (P < total) P <<= 1;
        for (int i = total + lane; i < P; i += 32) buf[i] = 0x7fffffff;
        __syncwarp();
        for (int k = 2; k <= P; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = lane; i < P; i += 32) {
                    const int l = i ^ j;
                    if (l > i) {
                        const int32_t a = buf[i], c = buf[l];
                        const bool asc = (i & k) == 0;
                        if ((a > c) == asc) { buf[i] = c; buf[l] = a; }
                    }
                }
                __syncwarp();
            }
        int off = 0;
        for (int i0 = 0; i0 < total; i0 += 32) {
            const int i = i0 + lane;
            const bool flag = i < total && (i == 0 || buf[i] != buf[i - 1]);
            const unsigned m = __ballot_sync(0xffffffffu, flag);
            if (pass == 1 && flag) indices[indptr[r] + off + __popc(m & ((1u << lane) - 1u))] = buf[i];
            off += __popc(m);
        }
        if (pass == 0 && lane == 0) counts[r] = off;
        __syncwarp();
    }
}

// exclusive scan of nrows+1 int32 counts (single block, serial over chunks: nrows <= ~10^7, a few ms)
__global__ void scan_kernel(int64_t n, const int32_t *__restrict__ counts, int32_t *__restrict__ indptr,
                            long long *total_out) {
    __shared__ long long wsum[32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int64_t base = 0; base < n; base += blockDim.x) {
        const int64_t i = base + threadIdx.x;
        long long v = i < n ? counts[i] : 0;
        long long x = v;
        for (int o = 1; o < 32; o <<= 1) {
            long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wsum[w] = x;
        __syncthreads();
        if (w == 0) {
            long long t = lane < (blockDim.x >> 5) ? wsum[lane] : 0;
            for (int o = 1; o < 32; o <<= 1) {
                long long y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            wsum[lane] = t;
        }
        __syncthreads();
        const long long excl = carry + (w ? wsum[w - 1] : 0) + x - v;
        if (i < n) indptr[i] = (int32_t)excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry += wsum[(blockDim.x >> 5) - 1];
        __syncthreads();
    }
    if (threadIdx.x == 0) { indptr[n] = (int32_t)carry; *total_out = carry; }
}

// Position maps: one warp per node, lanes over the node's (local row, local column) pairs;
// position = lower_bound of the column entity in the row of the structural pattern.
// (replaces 0.46 s of host binary searches + a 0.9 GB upload at 10^6 tetrahedra)
__global__ void posmap_kernel(int64_t nn, const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ row_ent,
                              const int32_t *__restrict__ col_ptr, const int32_t *__restrict__ col_ent,
                              const int32_t *__restrict__ ip, const int32_t *__restrict__ ix,
                              const int64_t *__restrict__ pos_ptr, int32_t *__restrict__ pos) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t s = warp; s < nn; s += nwarps) {
        const int r0 = row_ptr[s], nr = row_ptr[s + 1] - r0;
        const int c0 = col_ptr[s], ncl = col_ptr[s + 1] - c0;
        const int64_t base = pos_ptr[s];
        for (int e = lane; e < nr * ncl; e += 32) {
            const int i = e / ncl, j = e - i * ncl;
            const int r = row_ent[r0 + i], c = col_ent[c0 + j];
            int lo = ip[r], hi = ip[r + 1];
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (ix[mid] < c) lo = mid + 1; else hi = mid;
            }
            pos[base + e] = lo;
        }
    }
}

extern "C" int pb_plan_create(int nd, int64_t nc, int64_t nf, int64_t nn, const int32_t *cf_indptr,
                              const int32_t *cf_indices, const int8_t *cf_data,
                              const int32_t *fn_indptr, const int32_t *fn_indices, pb_plan **out) {
    NvtxRange nvtx_("pb_plan_create");
    if (!out || !cf_indptr || !cf_indices || !cf_data || !fn_indptr || !fn_indices)
        return fail(PB_EINVAL, "null pointer");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(PB_ECUDA, "no CUDA device: libporeb200 has no CPU path");
    pb_plan *p = new pb_plan;
    std::string err;
    {
        // torchrun exports OMP_NUM_THREADS=1; the plan builder is the one OpenMP user here, so give
        // it this rank's share of the cores (POREB200_PLAN_THREADS overrides) -- through a num_threads clause on
        // its parallel regions, not through the process-wide setter (numpy / torch keep their thread counts)
        int hw = (int)std::thread::hardware_concurrency();
        const char *lws = getenv("LOCAL_WORLD_SIZE");
        int share = hw / std::max(1, lws ? atoi(lws) : 1);
        const char *ov = getenv("POREB200_PLAN_THREADS");
        int nt = ov ? atoi(ov) : std::min(64, std::max(1, share));
        pb::g_plan_threads = std::max(1, nt);
    }
    auto tp0 = std::chrono::steady_clock::now();
    auto bail = [&](const char *what, cudaError_t e) {
        std::string m = std::string(what) + ": " + cudaGetErrorString(e);
        delete p;
        return fail(PB_ECUDA, m);
    };
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
    if ((e = cudaEventCreate(&p->e0)) != cudaSuccess) return bail("event", e);
    if ((e = cudaEventCreate(&p->e1)) != cudaSuccess) return bail("event", e);
    HostPlan &H = p->H;
    cudaStream_t st = p->stream;
    DevBuf fn_idx_dev;
    // ---- sub-cell topology: on the device (plan_device.cu); the host construction (plan_host.hpp) is the fallback
    // for interaction regions beyond the shared-memory sort capacity, and can be forced with POREB200_HOST_PLAN=1
    int rc = getenv("POREB200_HOST_PLAN") ? -1
             : pb_build_device_topology_(p, nd, nc, nf, nn, cf_indptr, cf_indices, cf_data, fn_indptr, fn_indices,
                                         fn_idx_dev, err);
    if (rc > 0) { delete p; return fail(rc, err); }
    const bool device_topology = rc == 0;
    if (getenv("POREB200_PLAN_TIMING")) {
        cudaStreamSynchronize(st);
        fprintf(stderr, "[plan] topology on the %s        %8.1f ms (since start)\n", device_topology ? "device" : "host  ",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count());
    }
    if (!device_topology) {
        p->H = HostPlan{};
        rc = build_host_plan(nd, nc, nf, nn, cf_indptr, cf_indices, cf_data, fn_indptr, fn_indices,
                             p->H, err, /*build_pos_maps=*/false, /*build_patterns=*/false);
        if (rc) {
            delete p;
            return fail(rc, err);
        }
#define UP(field, vec)                                                      \
    if ((e = p->field.upload(vec, st)) != cudaSuccess) return bail(#field, e);
        UP(fn_indptr, H.fn_indptr) UP(node_sc_ptr, H.node_sc_ptr) UP(sc_cell, H.sc_cell)
        UP(node_sf_ptr, H.node_sf_ptr) UP(sf_face, H.sf_face) UP(sf_sides, H.sf_sides)
        UP(sf_bloc, H.sf_bloc) UP(slot_sf, H.slot_sf) UP(node_nb, H.node_nb) UP(sc_ncn, H.sc_ncn)
        UP(posfc_ptr, H.posfc_ptr) UP(posfb_ptr, H.posfb_ptr) UP(poscc_ptr, H.poscc_ptr)
        UP(poscb_ptr, H.poscb_ptr) UP(nbf_ptr, H.nbf_ptr) UP(nbf_idx, H.nbf_idx) UP(cn_ptr, H.cn_ptr)
        UP(cn_idx, H.cn_idx) UP(face_cells, H.face_cells)
#undef UP
        if ((e = fn_idx_dev.upload(fn_indices, (size_t)fn_indptr[nf], st)) != cudaSuccess) return bail("fn_indices", e);
    }
    {
        // ---- structural patterns on the device (host fallback when a row has > 256 candidates)
        struct PJob { int which; int64_t nrows, ncols; DevBuf *rnp, *rn, *cp, *ci, *ip; };
        PJob pj[4] = {{0, nf, nc, &p->fn_indptr, &fn_idx_dev, &p->node_sc_ptr, &p->sc_cell, &p->fc_indptr},
                      {1, nf, nf, &p->fn_indptr, &fn_idx_dev, &p->nbf_ptr, &p->nbf_idx, &p->fb_indptr},
                      {2, nc, nc, &p->cn_ptr, &p->cn_idx, &p->node_sc_ptr, &p->sc_cell, &p->cc_indptr},
                      {3, nc, nf, &p->cn_ptr, &p->cn_idx, &p->nbf_ptr, &p->nbf_idx, &p->cb_indptr}};
        DevBuf counts, flag, total;
        if ((e = flag.ensure(sizeof(int))) != cudaSuccess) return bail("flag", e);
        if ((e = total.ensure(sizeof(long long))) != cudaSuccess) return bail("total", e);
        if ((e = cudaMemsetAsync(flag.p, 0, sizeof(int), st)) != cudaSuccess) return bail("memset", e);
        bool host_fallback = false;
        for (auto &j : pj) {
            if ((e = counts.ensure((size_t)(j.nrows + 1) * sizeof(int32_t))) != cudaSuccess) return bail("counts", e);
            if ((e = j.ip->ensure((size_t)(j.nrows + 1) * sizeof(int32_t))) != cudaSuccess) return bail("indptr", e);
            const int block = 256;
            int grid = (int)std::max<int64_t>(1, std::min<int64_t>((j.nrows + 7) / 8, (int64_t)kSMs * 8));
            pattern_kernel<256><<<grid, block, 0, st>>>(j.nrows, j.rnp->as<int32_t>(), j.rn->as<int32_t>(),
                                                        j.cp->as<int32_t>(), j.ci->as<int32_t>(),
                                                        counts.as<int32_t>(), nullptr, nullptr, 0, flag.as<int>());
            scan_kernel<<<1, 1024, 0, st>>>(j.nrows, counts.as<int32_t>(), j.ip->as<int32_t>(),
                                            total.as<long long>());
            long long tot = 0;
            int ov = 0;
            if ((e = cudaMemcpyAsync(&tot, total.p, sizeof(tot), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return bail("copy", e);
            if ((e = cudaMemcpyAsync(&ov, flag.p, sizeof(ov), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return bail("copy", e);
            if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail("pattern pass 0", e);
            g_launches += 2;
            if (ov) { host_fallback = true; break; }
            if (tot > 0x7FFFFFFFll) { delete p; return fail(PB_EINVAL, "pattern exceeds 2^31 entries; split the grid"); }
            if ((e = p->pat_idx[j.which].ensure((size_t)std::max<long long>(1, tot) * sizeof(int32_t))) != cudaSuccess) return bail("indices", e);
            pattern_kernel<256><<<grid, block, 0, st>>>(j.nrows, j.rnp->as<int32_t>(), j.rn->as<int32_t>(),
                                                        j.cp->as<int32_t>(), j.ci->as<int32_t>(), nullptr,
                                                        j.ip->as<int32_t>(), p->pat_idx[j.which].as<int32_t>(), 1,
                                                        flag.as<int>());
            g_launches++;
            p->pat_rows[j.which] = j.nrows; p->pat_cols[j.which] = j.ncols; p->pat_nnz[j.which] = tot;
        }
        if (host_fallback) {
            // rare: Delaunay-type nodes with > 256 candidates per row -> rebuild everything on the host
            std::string err2;
            HostPlan H2;
            int rc2 = build_host_plan(nd, nc, nf, nn, cf_indptr, cf_indices, cf_data, fn_indptr, fn_indices,
                                      H2, err2, false, true);
            if (rc2) { delete p; return fail(rc2, err2); }
            for (int w = 0; w < 4; ++w) {
                DevBuf *ip = w == 0 ? &p->fc_indptr : w == 1 ? &p->fb_indptr : w == 2 ? &p->cc_indptr : &p->cb_indptr;
                if ((e = ip->upload(H2.pat[w].indptr, st)) != cudaSuccess) return bail("indptr", e);
                if ((e = p->pat_idx[w].upload(H2.pat[w].indices, st)) != cudaSuccess) return bail("indices", e);
                p->pat_rows[w] = H2.pat[w].nrows; p->pat_cols[w] = H2.pat[w].ncols; p->pat_nnz[w] = H2.pat[w].nnz();
            }
            if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail("sync", e);
        }
        if (getenv("POREB200_PLAN_TIMING")) {
            cudaStreamSynchronize(st);
            fprintf(stderr, "[plan] patterns on device done     %8.1f ms (since start)\n",
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count());
        }
    }
    {
        struct Job { DevBuf *pos; const std::vector<int64_t> *ptr; DevBuf *pptr; int pat;
                     DevBuf *rp, *re, *cp, *ce; DevBuf *ip; };
        Job jobs[4] = {
            {&p->pos_fc, &H.posfc_ptr, &p->posfc_ptr, 0, &p->node_sf_ptr, &p->sf_face, &p->node_sc_ptr, &p->sc_cell, &p->fc_indptr},
            {&p->pos_fb, &H.posfb_ptr, &p->posfb_ptr, 1, &p->node_sf_ptr, &p->sf_face, &p->nbf_ptr, &p->nbf_idx, &p->fb_indptr},
            {&p->pos_cc, &H.poscc_ptr, &p->poscc_ptr, 2, &p->node_sc_ptr, &p->sc_cell, &p->node_sc_ptr, &p->sc_cell, &p->cc_indptr},
            {&p->pos_cb, &H.poscb_ptr, &p->poscb_ptr, 3, &p->node_sc_ptr, &p->sc_cell, &p->nbf_ptr, &p->nbf_idx, &p->cb_indptr},
        };
        for (auto &j : jobs) {
            // + 32 bytes: a 16-byte widened bulk copy of the last node's block may read past the end (PB_EXP_TMA)
            if ((e = j.pos->ensure((size_t)std::max<int64_t>(1, j.ptr->back()) * sizeof(int32_t) + 32)) != cudaSuccess)
                return bail("pos map", e);
            const int block = 256;
            int64_t need = (nn * 32 + block - 1) / block;
            int grid = (int)std::max<int64_t>(1, std::min<int64_t>(need, (int64_t)kSMs * 16));
            posmap_kernel<<<grid, block, 0, st>>>(nn, j.rp->as<int32_t>(), j.re->as<int32_t>(),
                                                  j.cp->as<int32_t>(), j.ce->as<int32_t>(),
                                                  j.ip->as<int32_t>(), p->pat_idx[j.pat].as<int32_t>(),
                                                  j.pptr->as<int64_t>(), j.pos->as<int32_t>());
            g_launches++;
            if ((e = cudaGetLastError()) != cudaSuccess) return bail("posmap_kernel", e);
        }
    }
    if ((e = p->err.ensure(sizeof(int))) != cudaSuccess) return bail("err", e);
    PlanView &v = p->view;
    v.nd = nd; v.nc = nc; v.nf = nf; v.nn = nn;
    v.fn_indptr = p->fn_indptr.as<int32_t>();
    v.node_sc_ptr = p->node_sc_ptr.as<int32_t>(); v.sc_cell = p->sc_cell.as<int32_t>();
    v.node_sf_ptr = p->node_sf_ptr.as<int32_t>(); v.sf_face = p->sf_face.as<int32_t>();
    v.sf_sides = p->sf_sides.as<uint32_t>(); v.sf_bloc = p->sf_bloc.as<uint16_t>();
    v.slot_sf = p->slot_sf.as<uint16_t>(); v.node_nb = p->node_nb.as<int32_t>();
    v.sc_ncn = p->sc_ncn.as<int32_t>();
    v.posfc_ptr = p->posfc_ptr.as<int64_t>(); v.posfb_ptr = p->posfb_ptr.as<int64_t>();
    v.poscc_ptr = p->poscc_ptr.as<int64_t>(); v.poscb_ptr = p->poscb_ptr.as<int64_t>();
    v.pos_fc = p->pos_fc.as<int32_t>(); v.pos_fb = p->pos_fb.as<int32_t>();
    v.pos_cc = p->pos_cc.as<int32_t>(); v.pos_cb = p->pos_cb.as<int32_t>();
    v.fc_indptr = p->fc_indptr.as<int32_t>(); v.fb_indptr = p->fb_indptr.as<int32_t>();
    v.cc_indptr = p->cc_indptr.as<int32_t>(); v.cb_indptr = p->cb_indptr.as<int32_t>();
    rc = build_mpfa_classes(p);
    if (rc) { delete p; return rc; }
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail("sync", e);
    // the host copies of the node-major lists are only needed for the uploads above
    {
        auto drop = [](auto &v) { v.clear(); v.shrink_to_fit(); };
        drop(H.sc_cell); drop(H.sf_face); drop(H.sf_sides); drop(H.sf_bloc); drop(H.slot_sf); drop(H.sc_ncn);
        drop(H.posfc_ptr); drop(H.posfb_ptr); drop(H.poscc_ptr); drop(H.poscb_ptr);
        drop(H.nbf_ptr); drop(H.nbf_idx); drop(H.cn_ptr); drop(H.cn_idx); drop(H.face_cells); drop(H.fn_indptr);
    }
    if (getenv("POREB200_PLAN_TIMING"))
        fprintf(stderr, "[plan] total incl. upload          %8.1f ms\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count());
    *out = p;
    return PB_OK;
}

extern "C" void pb_plan_destroy(pb_plan *p) {
    if (!p) return;
    if (p->stream) cudaStreamSynchronize(p->stream);
    if (p->e0) cudaEventDestroy(p->e0);
    if (p->e1) cudaEventDestroy(p->e1);
    if (p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

extern "C" int pb_plan_sizes(const pb_plan *p, int64_t *num_subcells, int64_t *num_subfaces,
                             int64_t *num_subhalffaces, int32_t *max_sf, int32_t *max_sc) {
    if (!p) return fail(PB_EINVAL, "null plan");
    if (num_subcells) *num_subcells = p->H.S;
    if (num_subfaces) *num_subfaces = p->H.U;
    if (num_subhalffaces) *num_subhalffaces = p->H.H;
    if (max_sf) *max_sf = p->H.max_nsf;
    if (max_sc) *max_sc = p->H.max_nsc;
    return PB_OK;
}

extern "C" int pb_plan_node_classes(const pb_plan *p, int kind, int cap, int32_t *cfg, uint8_t *a_global,
                                    int64_t *nodes, int *count) {
    if (!p || !count || cap < 0 || (kind != 0 && kind != 1)) return fail(PB_EINVAL, "bad arguments");
    const std::vector<NodeClass> &cls = kind == 0 ? p->mpfa_cls : p->mpsa_cls;
    *count = (int)cls.size();
    for (int i = 0; i < (int)cls.size() && i < cap; ++i) {
        if (cfg) cfg[i] = cls[i].cfg;
        if (a_global) a_global[i] = cls[i].a_global ? 1 : 0;
        if (nodes) nodes[i] = cls[i].n;
    }
    return PB_OK;
}

extern "C" int pb_plan_set_active_nodes(pb_plan *p, const uint8_t *mask) {
    if (!p) return pb_fail_(PB_EINVAL, "null plan");
    if (mask) p->active.assign(mask, mask + p->H.nn); else p->active.clear();
    p->mpsa_cls_nalpha = -1;  // the MPSA / Biot node classes are rebuilt at the next upload
    int rc = build_mpfa_classes(p);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    return PB_OK;
}

extern "C" int pb_plan_pattern_size(const pb_plan *p, int which, int64_t *nrows, int64_t *nnz) {
    if (!p || which < 0 || which > 3) return fail(PB_EINVAL, "bad pattern id");
    *nrows = p->pat_rows[which];
    *nnz = p->pat_nnz[which];
    return PB_OK;
}

extern "C" int pb_plan_pattern_get(const pb_plan *p, int which, int32_t *indptr, int32_t *indices) {
    if (!p || which < 0 || which > 3) return fail(PB_EINVAL, "bad pattern id");
    const DevBuf *ip = which == 0 ? &p->fc_indptr : which == 1 ? &p->fb_indptr : which == 2 ? &p->cc_indptr : &p->cb_indptr;
    CUDA_TRY(cudaMemcpyAsync(indptr, ip->p, (p->pat_rows[which] + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, p->stream));
    if (p->pat_nnz[which])
        CUDA_TRY(cudaMemcpyAsync(indices, p->pat_idx[which].p, p->pat_nnz[which] * sizeof(int32_t),
                                 cudaMemcpyDeviceToHost, p->stream));
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    return PB_OK;
}

// one warp per base row; lanes run over the row's expanded entries (coalesced stores)
__global__ void expand_pattern_kernel(int64_t nrows, const int32_t *__restrict__ ip,
                                      const int32_t *__restrict__ ix, int br, int bc,
                                      int32_t *__restrict__ nip, int32_t *__restrict__ nix) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < nrows; r += nwarps) {
        const int64_t b = ip[r], len = ip[r + 1] - b;
        const int64_t base = (int64_t)br * bc * b, rowlen = len * bc;
        for (int i = 0; i < br; ++i) {
            if (lane == 0) nip[r * br + i] = (int32_t)(base + i * rowlen);
            for (int64_t t = lane; t < rowlen; t += 32) {
                const int64_t q = t / bc;
                const int j = (int)(t - q * bc);
                nix[base + i * rowlen + t] = ix[b + q] * bc + j;
            }
        }
    }
    if (warp == 0 && lane == 0) nip[nrows * br] = (int32_t)((int64_t)br * bc * ip[nrows]);
}

extern "C" int pb_plan_pattern_expanded(pb_plan *p, int which, int br, int bc, int32_t *indptr,
                                        int32_t *indices) {
    if (!p || which < 0 || which > 3 || br < 1 || bc < 1 || !indptr || !indices)
        return fail(PB_EINVAL, "bad arguments");
    struct { int64_t nrows, ncols; } c{p->pat_rows[which], p->pat_cols[which]};
    const int64_t nnz = p->pat_nnz[which] * br * bc;
    if (nnz >= 0x7FFFFFFFll || c.ncols * bc >= 0x7FFFFFFFll)
        return fail(PB_ENOTIMPL, "expanded pattern does not fit int32 indices");
    DevBuf *bip = which == 0 ? &p->fc_indptr : which == 1 ? &p->fb_indptr : which == 2 ? &p->cc_indptr : &p->cb_indptr;
    DevBuf nip, nix;
    DevBuf &dix = p->pat_idx[which];
    cudaStream_t st = p->stream;
    CUDA_TRY(nip.ensure((c.nrows * br + 1) * sizeof(int32_t)));
    CUDA_TRY(nix.ensure((nnz ? nnz : 1) * sizeof(int32_t)));
    const int block = 256;
    int64_t need = (c.nrows * 32 + block - 1) / block;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>(need, (int64_t)kSMs * 16));
    expand_pattern_kernel<<<grid, block, 0, st>>>(c.nrows, bip->as<int32_t>(), dix.as<int32_t>(), br, bc,
                                                  nip.as<int32_t>(), nix.as<int32_t>());
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(indptr, nip.p, (c.nrows * br + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (nnz) CUDA_TRY(cudaMemcpyAsync(indices, nix.p, nnz * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return PB_OK;
}

// (ncomp, n) row-major -> (n, ncomp): one contiguous record per entity for the per-sub-cell gathers
__global__ void repack_kernel(const double *__restrict__ in, double *__restrict__ out, int ncomp, int64_t n) {
    const int64_t total = (int64_t)ncomp * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i / ncomp;
        const int comp = (int)(i - e * ncomp);
        out[i] = in[(int64_t)comp * n + e];
    }
}

int pb_upload_repacked_(cudaStream_t st, DevBuf &tmp, DevBuf &dst, const double *host, int ncomp, int64_t n) {
    CUDA_TRY(tmp.upload(host, (size_t)ncomp * n, st));
    CUDA_TRY(dst.ensure((size_t)ncomp * n * sizeof(double)));
    const int64_t total = (int64_t)ncomp * n;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, (int64_t)kSMs * 32));
    repack_kernel<<<grid, 256, 0, st>>>(tmp.as<double>(), dst.as<double>(), ncomp, n);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return PB_OK;
}

// the same with a gather: the host array holds the cells of a LARGER (global) grid, (ncomp, n_src) row-major, and
// entity e of this plan is cell map[e] of it (a shard uploads the global tensor and restricts it on the device)
__global__ void repack_gather_kernel(const double *__restrict__ in, double *__restrict__ out, int ncomp, int64_t n,
                                     int64_t n_src, const int64_t *__restrict__ map) {
    const int64_t total = (int64_t)ncomp * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i / ncomp;
        const int comp = (int)(i - e * ncomp);
        out[i] = in[(int64_t)comp * n_src + map[e]];
    }
}

static int upload_repacked(pb_plan *p, DevBuf &dst, const double *host, int ncomp, int64_t n) {
    return pb_upload_repacked_(p->stream, p->repack_tmp, dst, host, ncomp, n);
}

// cell tensors: through the cell map when one is set (pb_plan_set_cell_map)
static int upload_cell_tensor(pb_plan *p, DevBuf &dst, const double *host, int ncomp) {
    const int64_t n = p->H.nc;
    if (!p->cell_map.p) return upload_repacked(p, dst, host, ncomp, n);
    cudaStream_t st = p->stream;
    CUDA_TRY(p->repack_tmp.upload(host, (size_t)ncomp * p->cell_map_src, st));
    CUDA_TRY(dst.ensure((size_t)ncomp * n * sizeof(double)));
    const int64_t total = (int64_t)ncomp * n;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, (int64_t)kSMs * 32));
    repack_gather_kernel<<<grid, 256, 0, st>>>(p->repack_tmp.as<double>(), dst.as<double>(), ncomp, n, p->cell_map_src,
                                               p->cell_map.as<int64_t>());
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return PB_OK;
}

extern "C" int pb_plan_set_cell_map(pb_plan *p, const int64_t *cells, int64_t n_source_cells) {
    if (!p) return fail(PB_EINVAL, "null plan");
    if (!cells) { p->cell_map.release(); p->cell_map_src = 0; return PB_OK; }
    if (n_source_cells < 1) return fail(PB_EINVAL, "bad source size");
    for (int64_t e = 0; e < p->H.nc; ++e)
        if (cells[e] < 0 || cells[e] >= n_source_cells) return fail(PB_EINVAL, "cell map entry out of range");
    CUDA_TRY(p->cell_map.upload(cells, (size_t)p->H.nc, p->stream));
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    p->cell_map_src = n_source_cells;
    return PB_OK;
}

extern "C" int pb_plan_set_geometry(pb_plan *p, const double *nodes, const double *face_normals,
                                    const double *face_centers, const double *face_areas,
                                    const double *cell_centers, const double *cell_volumes) {
    NvtxRange nvtx_("pb_plan_set_geometry");
    if (!p || !nodes || !face_normals || !face_centers || !face_areas || !cell_centers || !cell_volumes)
        return fail(PB_EINVAL, "null pointer");
    const HostPlan &H = p->H;
    cudaStream_t st = p->stream;
    int rc;
    {   // Morton keys of the nodes (10 bits per axis over the bounding box) and re-ordered class lists
        const char *ord = getenv("POREB200_NODE_ORDER");
        const bool morton = !(ord && strcmp(ord, "index") == 0);
        const bool had = !p->node_key.empty();
        double sig = 0.0;   // cheap signature of the coordinates: unchanged geometry keeps the keys and the lists
        for (int64_t i = 0; i < 3 * H.nn; i += 7) sig += nodes[i] * (double)((i % 13) + 1);
        const bool same = had && morton && sig == p->node_key_sig;
        p->node_key_sig = sig;
        if (!same) p->node_key.clear();
        if (morton && !same) {
            double lo[3], hi[3];
            for (int d = 0; d < 3; ++d) {
                lo[d] = 1e300; hi[d] = -1e300;
                for (int64_t s = 0; s < H.nn; ++s) { const double v = nodes[d * H.nn + s]; lo[d] = std::min(lo[d], v); hi[d] = std::max(hi[d], v); }
            }
            auto spread = [](uint32_t v) {   // 10 bits -> every third bit
                v &= 0x3ff;
                v = (v | (v << 16)) & 0x30000ff; v = (v | (v << 8)) & 0x300f00f;
                v = (v | (v << 4)) & 0x30c30c3;  v = (v | (v << 2)) & 0x9249249;
                return v;
            };
            p->node_key.resize(H.nn);
            for (int64_t s = 0; s < H.nn; ++s) {
                uint32_t q[3];
                for (int d = 0; d < 3; ++d) {
                    const double ext = hi[d] - lo[d];
                    q[d] = ext > 0 ? (uint32_t)std::min(1023.0, (nodes[d * H.nn + s] - lo[d]) / ext * 1024.0) : 0u;
                }
                p->node_key[s] = spread(q[0]) | (spread(q[1]) << 1) | (spread(q[2]) << 2);
            }
        }
        if (!same && (morton || had)) {
            if ((rc = build_mpfa_classes(p))) return rc;
            p->mpsa_cls_nalpha = -1;   // MPSA / Biot classes are rebuilt (and ordered) at the next upload
        }
    }
    if ((rc = upload_repacked(p, p->nodes, nodes, 3, H.nn))) return rc;
    if ((rc = upload_repacked(p, p->fnorm, face_normals, 3, H.nf))) return rc;
    if ((rc = upload_repacked(p, p->fcent, face_centers, 3, H.nf))) return rc;
    if ((rc = upload_repacked(p, p->ccent, cell_centers, 3, H.nc))) return rc;
    CUDA_TRY(p->farea.upload(face_areas, H.nf, st));
    CUDA_TRY(p->cvol.upload(cell_volumes, H.nc, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    p->geo = GeoView{p->nodes.as<double>(), p->fnorm.as<double>(), p->fcent.as<double>(),
                     p->farea.as<double>(), p->ccent.as<double>(), p->cvol.as<double>(),
                     1, 3, 1, 3, 1, 3};
    p->have_geo = true;
    return PB_OK;
}

// ------------------------------------------------------------------------------------
// error flag helpers
// ------------------------------------------------------------------------------------
static int check_singular(pb_plan *p) {
    int h = INT_MAX;
    CUDA_TRY(cudaMemcpyAsync(&h, p->err.p, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    if (h != INT_MAX) {
        g_err_node = h;
        return fail(PB_ESINGULAR, "singular local system at node " + std::to_string(h));
    }
    return PB_OK;
}

// ------------------------------------------------------------------------------------
// MPFA
// ------------------------------------------------------------------------------------
extern "C" int pb_mpfa_upload(pb_plan *p, const double *perm, const uint8_t *bc,
                              const double *robin_weight, double eta) {
    NvtxRange nvtx_("pb_mpfa_upload");
    if (!p || !perm || !bc) return fail(PB_EINVAL, "null pointer");
    if (!p->have_geo) return fail(PB_EINVAL, "pb_plan_set_geometry has not been called");
    const HostPlan &H = p->H;
    cudaStream_t st = p->stream;
    { int rcp = upload_cell_tensor(p, p->perm, perm, 9); if (rcp) return rcp; }
    CUDA_TRY(p->bc.upload(bc, H.nf, st));
    p->have_robw = robin_weight != nullptr;
    if (robin_weight) CUDA_TRY(p->robw.upload(robin_weight, H.nf, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    p->eta = eta;
    p->mpfa_ready = true;
    return PB_OK;
}

extern "C" int pb_mpfa_assemble(pb_plan *p, int want_flux, int want_trace, int want_vs, float *ms) {
    NvtxRange nvtx_("pb_mpfa_assemble");
    if (!p) return fail(PB_EINVAL, "null plan");
    if (!p->mpfa_ready) return fail(PB_EINVAL, "pb_mpfa_upload has not been called");
    const HostPlan &H = p->H;
    const int nd = H.nd;
    cudaStream_t st = p->stream;
    const size_t nfc = (size_t)p->pat_nnz[0], nfb = (size_t)p->pat_nnz[1];
    MpfaOut o{};
    struct Req { DevBuf *b; double **slot; size_t n; bool want; };
    Req reqs[6] = {{&p->o_flux, &o.flux, nfc, want_flux != 0},
                   {&p->o_bflux, &o.bflux, nfb, want_flux != 0},
                   {&p->o_bpc, &o.bpc, nfc, want_trace != 0},
                   {&p->o_bpf, &o.bpf, nfb, want_trace != 0},
                   {&p->o_vs, &o.vs, nfc * nd, want_vs != 0 && want_flux != 0},
                   {&p->o_bpvs, &o.bpvs, nfc * nd, want_vs != 0 && want_trace != 0}};
    for (auto &r : reqs)
        if (r.want) CUDA_TRY(r.b->ensure(r.n * sizeof(double)));
    CUDA_TRY(cudaEventRecord(p->e0, st));
    for (auto &r : reqs) {
        if (!r.want) { *r.slot = nullptr; continue; }
        CUDA_TRY(cudaMemsetAsync(r.b->p, 0, r.n * sizeof(double), st));
        *r.slot = r.b->as<double>();
    }
    int init = INT_MAX;
    CUDA_TRY(cudaMemcpyAsync(p->err.p, &init, sizeof(int), cudaMemcpyHostToDevice, st));
    MpfaParams prm{p->perm.as<double>(), p->bc.as<uint8_t>(),
                   p->have_robw ? p->robw.as<double>() : nullptr, p->eta, 1, 9};
    { int rc = pb_launch_mpfa_(p, prm, o); if (rc) return rc; }
    CUDA_TRY(cudaEventRecord(p->e1, st));
    CUDA_TRY(cudaEventSynchronize(p->e1));
    if (ms) CUDA_TRY(cudaEventElapsedTime(ms, p->e0, p->e1));
    return check_singular(p);
}

static int dl(pb_plan *p, DevBuf &b, double *h, size_t n) {
    if (!h) return PB_OK;
    if (!b.p || b.bytes < n * sizeof(double)) return fail(PB_EINVAL, "output was not assembled");
    CUDA_TRY(cudaMemcpyAsync(h, b.p, n * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    return PB_OK;
}

extern "C" int pb_mpfa_download(pb_plan *p, double *flux, double *bound_flux, double *bpc,
                                double *bpf, double *vs, double *bpvs) {
    if (!p) return fail(PB_EINVAL, "null plan");
    const HostPlan &H = p->H;
    const size_t nfc = (size_t)p->pat_nnz[0], nfb = (size_t)p->pat_nnz[1];
    int rc;
    if ((rc = dl(p, p->o_flux, flux, nfc))) return rc;
    if ((rc = dl(p, p->o_bflux, bound_flux, nfb))) return rc;
    if ((rc = dl(p, p->o_bpc, bpc, nfc))) return rc;
    if ((rc = dl(p, p->o_bpf, bpf, nfb))) return rc;
    if ((rc = dl(p, p->o_vs, vs, nfc * H.nd))) return rc;
    if ((rc = dl(p, p->o_bpvs, bpvs, nfc * H.nd))) return rc;
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    return PB_OK;
}

// ------------------------------------------------------------------------------------
// detached output value arrays (device resident; the lazily downloaded matrices of the Python layer)
// ------------------------------------------------------------------------------------
struct pb_values {
    DevBuf buf;
    int64_t n = 0;
    cudaStream_t stream = nullptr;  // the plan's stream (kernels that wrote the values were ordered on it)
};

static DevBuf *output_slot(pb_plan *p, int key, int64_t *n) {
    const int64_t nd = p->H.nd, nd2 = nd * nd;
    const int64_t nfc = p->pat_nnz[0], nfb = p->pat_nnz[1], ncc = p->pat_nnz[2], ncb = p->pat_nnz[3];
    switch (key) {
        case PB_OUT_FLUX: *n = nfc; return &p->o_flux;
        case PB_OUT_BOUND_FLUX: *n = nfb; return &p->o_bflux;
        case PB_OUT_BOUND_PRESSURE_CELL: *n = nfc; return &p->o_bpc;
        case PB_OUT_BOUND_PRESSURE_FACE: *n = nfb; return &p->o_bpf;
        case PB_OUT_VECTOR_SOURCE: *n = nfc * nd; return &p->o_vs;
        case PB_OUT_BOUND_PRESSURE_VECTOR_SOURCE: *n = nfc * nd; return &p->o_bpvs;
        case PB_OUT_STRESS: *n = nfc * nd2; return &p->o_stress;
        case PB_OUT_BOUND_STRESS: *n = nfb * nd2; return &p->o_bstress;
        case PB_OUT_BOUND_DISPLACEMENT_CELL: *n = nfc * nd2; return &p->o_bdc;
        case PB_OUT_BOUND_DISPLACEMENT_FACE: *n = nfb * nd2; return &p->o_bdf;
        default: break;
    }
    if (key >= PB_OUT_BIOT && key < PB_OUT_BIOT + 5 * PB_MAX_ALPHA) {
        const int q = (key - PB_OUT_BIOT) / 5, t = (key - PB_OUT_BIOT) % 5;
        if (q >= p->n_alpha) return nullptr;
        switch (t) {
            case 0: *n = ncc * nd; return &p->o_dd[q];
            case 1: *n = ncb * nd; return &p->o_bdd[q];
            case 2: *n = nfc * nd; return &p->o_sg[q];
            case 3: *n = ncc; return &p->o_cons[q];
            default: *n = nfc * nd; return &p->o_bdp[q];
        }
    }
    return nullptr;
}

extern "C" int pb_plan_take_output(pb_plan *p, int key, pb_values **out) {
    if (!p || !out) return fail(PB_EINVAL, "null pointer");
    int64_t n = 0;
    DevBuf *slot = output_slot(p, key, &n);
    if (!slot) return fail(PB_EINVAL, "unknown output key");
    if (!slot->p || slot->bytes < (size_t)n * sizeof(double)) return fail(PB_EINVAL, "output was not assembled");
    pb_values *v = new pb_values;
    v->buf = std::move(*slot);   // the plan allocates a fresh array at its next assemble
    v->n = n;
    v->stream = p->stream;
    *out = v;
    return PB_OK;
}
extern "C" int64_t pb_values_size(const pb_values *v) { return v ? v->n : -1; }
extern "C" void pb_values_destroy(pb_values *v) { delete v; }
extern "C" int pb_values_download(pb_values *v, double *host) {
    if (!v || !host) return fail(PB_EINVAL, "null pointer");
    if (v->n) CUDA_TRY(cudaMemcpy(host, v->buf.p, (size_t)v->n * sizeof(double), cudaMemcpyDeviceToHost));
    return PB_OK;
}
// sum and sum of squares of the values (device reduction; a 16-byte read that proves the values exist)
__global__ void values_checksum_kernel(int64_t n, const double *__restrict__ v, double *out) {
    double s = 0.0, q = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double x = v[i];
        s += x; q += x * x;
    }
    for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
    if ((threadIdx.x & 31) == 0) { atomicAdd(out, s); atomicAdd(out + 1, q); }
}
int pb_checksum_dev_(const double *v, int64_t n, double *sum, double *sumsq) {
    DevBuf o;
    CUDA_TRY(o.ensure(16));
    CUDA_TRY(cudaMemset(o.p, 0, 16));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)kSMs * 8));
    values_checksum_kernel<<<grid, 256>>>(n, v, o.as<double>());
    g_launches++;
    double h[2];
    CUDA_TRY(cudaMemcpy(h, o.p, 16, cudaMemcpyDeviceToHost));
    if (sum) *sum = h[0];
    if (sumsq) *sumsq = h[1];
    return PB_OK;
}
extern "C" int pb_values_checksum(pb_values *v, double *sum, double *sumsq) {
    if (!v) return fail(PB_EINVAL, "null pointer");
    CUDA_TRY(cudaStreamSynchronize(v->stream));
    return pb_checksum_dev_(v->buf.as<double>(), v->n, sum, sumsq);
}

// ------------------------------------------------------------------------------------
// device-side flow system  A = div @ flux,  b = -div @ (bound_flux @ bc [+ vector_source @ v])
// ------------------------------------------------------------------------------------
struct pb_csr;
int pb_csr_from_device_pattern_(int64_t nrows, int64_t ncols, int64_t nnz, const int32_t *indptr_dev,
                                const int32_t *indices_dev, pb_csr **out);  // spmv.cu
double *pb_csr_data_(pb_csr *a);

// one warp per face: every entry (f, k) of the flux row goes to row c of A for the one or two
// cells c of the face, with the sign of cell_faces[f, c] (= div[c, f]); position by binary search
// in the CELL_CELL row (the flux row's columns are a subset of it)
__global__ void div_flux_kernel(int64_t nf, const int32_t *__restrict__ fc_ip, const int32_t *__restrict__ fc_ix,
                                const double *__restrict__ flux, const int32_t *__restrict__ face_cells,
                                const int32_t *__restrict__ cc_ip, const int32_t *__restrict__ cc_ix,
                                double *__restrict__ a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t f = warp; f < nf; f += nwarps) {
        for (int sd = 0; sd < 2; ++sd) {
            const int32_t enc = face_cells[2 * f + sd];  // (cell << 1) | (sign < 0), -1 = none
            if (enc < 0) continue;
            const int c = enc >> 1;
            const double sg = (enc & 1) ? -1.0 : 1.0;
            const int b = cc_ip[c], e = cc_ip[c + 1];
            for (int q = fc_ip[f] + lane; q < fc_ip[f + 1]; q += 32) {
                const int k = fc_ix[q];
                int lo = b, hi = e;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (cc_ix[mid] < k) lo = mid + 1; else hi = mid;
                }
                atomicAdd(a + lo, sg * flux[q]);
            }
        }
    }
}

// y[f] = sum_q vals[q*blk + j] * x[cols[q]*blk + j]   (blk = 1: bound_flux @ bc; blk = nd: vector_source @ v)
__global__ void face_row_dot_kernel(int64_t nf, const int32_t *__restrict__ ip, const int32_t *__restrict__ ix,
                                    const double *__restrict__ vals, int blk, const double *__restrict__ x,
                                    double *__restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t f = warp; f < nf; f += nwarps) {
        double acc = 0.0;
        const int64_t b = ip[f], e = ip[f + 1];
        for (int64_t t = b * blk + lane; t < e * blk; t += 32) {
            const int64_t q = t / blk;
            const int j = (int)(t - q * blk);
            acc += vals[t] * x[(int64_t)ix[q] * blk + j];
        }
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) y[f] += acc;
    }
}

// rhs[c] = - sum_{f of c} sign * w[f]
__global__ void neg_div_kernel(int64_t nf, const int32_t *__restrict__ face_cells, const double *__restrict__ w,
                               double *__restrict__ rhs) {
    for (int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; f < nf; f += (int64_t)gridDim.x * blockDim.x)
        for (int sd = 0; sd < 2; ++sd) {
            const int32_t enc = face_cells[2 * f + sd];
            if (enc >= 0) atomicAdd(rhs + (enc >> 1), ((enc & 1) ? 1.0 : -1.0) * w[f]);
        }
}

static int ensure_face_cells(pb_plan *p) {
    if (p->face_cells.p) return PB_OK;  // uploaded by pb_plan_create
    return fail(PB_EINVAL, "plan has no face->cell table");
}

int pb_csr_alloc_(int64_t nrows, int64_t ncols, int64_t nnz, pb_csr **out);  // spmv.cu
int32_t *pb_csr_indptr_(pb_csr *a);
int32_t *pb_csr_indices_(pb_csr *a);

// One output matrix as a device CSR (the block-expanded pattern + a copy of the values): the operand form of the
// device-side AD chain (sparse_ops.cu).  which / br / bc as in pb_plan_pattern_expanded.
extern "C" int pb_plan_output_csr(pb_plan *p, const pb_values *v, int which, int br, int bc, pb_csr **out) {
    if (!p || !v || !out || which < 0 || which > 3 || br < 1 || bc < 1) return fail(PB_EINVAL, "bad arguments");
    const int64_t nrows = p->pat_rows[which], nnz = p->pat_nnz[which] * br * bc;
    if (v->n != nnz) return fail(PB_EINVAL, "values do not match this pattern / block size");
    if (nnz >= 0x7FFFFFFFll || p->pat_cols[which] * bc >= 0x7FFFFFFFll) return fail(PB_ENOTIMPL, "matrix does not fit int32 indices");
    pb_csr *a = nullptr;
    int rc = pb_csr_alloc_(nrows * br, p->pat_cols[which] * bc, nnz, &a);
    if (rc) return rc;
    DevBuf *bip = which == 0 ? &p->fc_indptr : which == 1 ? &p->fb_indptr : which == 2 ? &p->cc_indptr : &p->cb_indptr;
    const int block = 256;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((nrows * 32 + block - 1) / block, (int64_t)kSMs * 16));
    expand_pattern_kernel<<<grid, block, 0, p->stream>>>(nrows, bip->as<int32_t>(), p->pat_idx[which].as<int32_t>(), br, bc,
                                                         pb_csr_indptr_(a), pb_csr_indices_(a));
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    if (nnz) CUDA_TRY(cudaMemcpyAsync(pb_csr_data_(a), v->buf.p, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToDevice, p->stream));
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    *out = a;
    return PB_OK;
}

extern "C" int pb_mpfa_system(pb_plan *p, const pb_values *flux, pb_csr **out) {
    NvtxRange nvtx_("pb_mpfa_system");
    if (!p || !out) return fail(PB_EINVAL, "null pointer");
    const double *flux_dev = flux ? flux->buf.as<double>() : p->o_flux.as<double>();
    if (flux && flux->n != p->pat_nnz[0]) return fail(PB_EINVAL, "flux values do not belong to this plan");
    if (!flux_dev) return fail(PB_EINVAL, "pb_mpfa_assemble (flux terms) has not been called");
    const HostPlan &H = p->H;
    int rc = ensure_face_cells(p);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    pb_csr *a = nullptr;
    rc = pb_csr_from_device_pattern_(H.nc, H.nc, p->pat_nnz[2], p->cc_indptr.as<int32_t>(),
                                     p->pat_idx[2].as<int32_t>(), &a);
    if (rc) return rc;
    const int block = 256;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((H.nf * 32 + block - 1) / block, (int64_t)kSMs * 16));
    div_flux_kernel<<<grid, block, 0, p->stream>>>(H.nf, p->fc_indptr.as<int32_t>(), p->pat_idx[0].as<int32_t>(),
                                                   flux_dev, p->face_cells.as<int32_t>(),
                                                   p->cc_indptr.as<int32_t>(), p->pat_idx[2].as<int32_t>(),
                                                   pb_csr_data_(a));
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    *out = a;
    return PB_OK;
}

extern "C" int pb_mpfa_rhs(pb_plan *p, const pb_values *bound_flux, const pb_values *vector_source_discr,
                           const double *bc_values, const double *vector_source, double *rhs) {
    NvtxRange nvtx_("pb_mpfa_rhs");
    if (!p || !bc_values || !rhs) return fail(PB_EINVAL, "null pointer");
    const double *bflux_dev = bound_flux ? bound_flux->buf.as<double>() : p->o_bflux.as<double>();
    const double *vs_dev = vector_source_discr ? vector_source_discr->buf.as<double>() : p->o_vs.as<double>();
    if (bound_flux && bound_flux->n != p->pat_nnz[1]) return fail(PB_EINVAL, "bound_flux values do not belong to this plan");
    if (vector_source_discr && vector_source_discr->n != p->pat_nnz[0] * p->H.nd)
        return fail(PB_EINVAL, "vector_source values do not belong to this plan");
    if (!bflux_dev) return fail(PB_EINVAL, "pb_mpfa_assemble (flux terms) has not been called");
    if (vector_source && !vs_dev) return fail(PB_EINVAL, "vector source terms were not assembled");
    const HostPlan &H = p->H;
    cudaStream_t st = p->stream;
    int rc = ensure_face_cells(p);
    if (rc) return rc;
    DevBuf bc, vs, w, r;
    CUDA_TRY(bc.upload(bc_values, (size_t)H.nf, st));
    CUDA_TRY(w.ensure((size_t)H.nf * sizeof(double)));
    CUDA_TRY(r.ensure((size_t)H.nc * sizeof(double)));
    CUDA_TRY(cudaMemsetAsync(w.p, 0, (size_t)H.nf * sizeof(double), st));
    CUDA_TRY(cudaMemsetAsync(r.p, 0, (size_t)H.nc * sizeof(double), st));
    const int block = 256;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((H.nf * 32 + block - 1) / block, (int64_t)kSMs * 16));
    face_row_dot_kernel<<<grid, block, 0, st>>>(H.nf, p->fb_indptr.as<int32_t>(), p->pat_idx[1].as<int32_t>(),
                                                bflux_dev, 1, bc.as<double>(), w.as<double>());
    g_launches++;
    if (vector_source) {
        CUDA_TRY(vs.upload(vector_source, (size_t)H.nc * H.nd, st));
        face_row_dot_kernel<<<grid, block, 0, st>>>(H.nf, p->fc_indptr.as<int32_t>(), p->pat_idx[0].as<int32_t>(),
                                                    vs_dev, H.nd, vs.as<double>(), w.as<double>());
        g_launches++;
    }
    int grid2 = (int)std::max<int64_t>(1, std::min<int64_t>((H.nf + block - 1) / block, (int64_t)kSMs * 16));
    neg_div_kernel<<<grid2, block, 0, st>>>(H.nf, p->face_cells.as<int32_t>(), w.as<double>(), r.as<double>());
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(rhs, r.p, (size_t)H.nc * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return PB_OK;
}

// ------------------------------------------------------------------------------------
// device-side mechanics system  A = div_nd @ stress,  b = -div_nd @ (bound_stress @ bc) + source
// ------------------------------------------------------------------------------------
// one warp per face; block layouts as documented at pb_plan_pattern_expanded
__global__ void div_stress_kernel(int64_t nf, int nd, const int32_t *__restrict__ fc_ip,
                                  const int32_t *__restrict__ fc_ix, const double *__restrict__ stress,
                                  const int32_t *__restrict__ face_cells, const int32_t *__restrict__ cc_ip,
                                  const int32_t *__restrict__ cc_ix, double *__restrict__ a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nd2 = nd * nd;
    for (int64_t f = warp; f < nf; f += nwarps) {
        const int64_t fb = fc_ip[f], flen = fc_ip[f + 1] - fb;
        for (int sd = 0; sd < 2; ++sd) {
            const int32_t enc = face_cells[2 * f + sd];
            if (enc < 0) continue;
            const int c = enc >> 1;
            const double sg = (enc & 1) ? -1.0 : 1.0;
            const int64_t cb = cc_ip[c], clen = cc_ip[c + 1] - cb;
            for (int64_t t = lane; t < flen * nd2; t += 32) {
                const int64_t q = t / nd2;
                const int ij = (int)(t - q * nd2);
                const int i = ij / nd, j = ij - i * nd;
                const int k = fc_ix[fb + q];
                int64_t lo = cb, hi = cb + clen;
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (cc_ix[mid] < k) lo = mid + 1; else hi = mid;
                }
                const double v = stress[nd2 * fb + (int64_t)i * nd * flen + q * nd + j];
                atomicAdd(a + nd2 * cb + (int64_t)i * nd * clen + (lo - cb) * nd + j, sg * v);
            }
        }
    }
}

// Gather form of the same product, used when the plan holds the cell -> faces lists (device topology build): one warp per
// cell sums the rows of its faces into the cell's block row in shared memory -- no atomics, one coalesced store of the
// nd*nd*clen values (the scatter form above issues nd*nd atomics and binary searches per stress entry and side: 20 ms at
// 10^6 tetrahedra against ~13 GB = 2 ms of compulsory traffic).  Rows longer than `cap` block columns accumulate in place.
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
    div_stress_gather_kernel(int64_t nc, int nd, const int32_t *__restrict__ cf_ip, const int32_t *__restrict__ cf_ix,
                             const int8_t *__restrict__ cf_sg, const int32_t *__restrict__ fc_ip,
                             const int32_t *__restrict__ fc_ix, const double *__restrict__ stress,
                             const int32_t *__restrict__ cc_ip, const int32_t *__restrict__ cc_ix, double *a, int cap) {
    extern __shared__ double gather_sm[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nd2 = nd * nd;
    double *acc = gather_sm + (size_t)w * cap * nd2;
    for (int64_t c = (int64_t)blockIdx.x * WARPS + w; c < nc; c += (int64_t)gridDim.x * WARPS) {
        const int64_t cb = cc_ip[c];
        const int clen = (int)(cc_ip[c + 1] - cb);
        const bool staged = clen <= cap;
        double *dst = staged ? acc : a + nd2 * cb;     // [i][position in the row][j]
        const int tot = clen * nd2;
        for (int t = lane; t < tot; t += 32) dst[t] = 0.0;
        __syncwarp();
        for (int s = cf_ip[c]; s < cf_ip[c + 1]; ++s) {
            const int f = cf_ix[s];
            const double sg = (double)cf_sg[s];        // div[c, f] = cell_faces[f, c]
            const int64_t fb = fc_ip[f];
            const int flen = (int)(fc_ip[f + 1] - fb);
            for (int t = lane; t < flen * nd; t += 32) {
                const int q = t / nd, j = t - q * nd;
                const int k = fc_ix[fb + q];
                int lo = 0, hi = clen;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (cc_ix[cb + mid] < k) lo = mid + 1; else hi = mid;
                }
                for (int i = 0; i < nd; ++i)
                    dst[i * nd * clen + lo * nd + j] += sg * stress[nd2 * fb + (int64_t)i * nd * flen + t];
            }
            __syncwarp();                               // the next face may touch the same entries from other lanes
        }
        if (staged) {
            for (int t = lane; t < tot; t += 32) a[nd2 * cb + t] = acc[t];
            __syncwarp();
        }
    }
}

// w[f*nd+i] = sum over block entries of bound_stress row (f,i) times bc
__global__ void bound_stress_dot_kernel(int64_t nf, int nd, const int32_t *__restrict__ ip,
                                        const int32_t *__restrict__ ix, const double *__restrict__ vals,
                                        const double *__restrict__ x, double *__restrict__ w) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nd2 = nd * nd;
    for (int64_t r = warp; r < nf * nd; r += nwarps) {
        const int64_t f = r / nd;
        const int i = (int)(r - f * nd);
        const int64_t b = ip[f], len = ip[f + 1] - b;
        double acc = 0.0;
        for (int64_t t = lane; t < len * nd; t += 32) {
            const int64_t q = t / nd;
            const int j = (int)(t - q * nd);
            acc += vals[nd2 * b + (int64_t)i * nd * len + t] * x[(int64_t)ix[b + q] * nd + j];
        }
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) w[r] = acc;
    }
}

__global__ void neg_div_nd_kernel(int64_t nf, int nd, const int32_t *__restrict__ face_cells,
                                  const double *__restrict__ w, double *__restrict__ rhs) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nf * nd; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = r / nd;
        const int i = (int)(r - f * nd);
        for (int sd = 0; sd < 2; ++sd) {
            const int32_t enc = face_cells[2 * f + sd];
            if (enc >= 0) atomicAdd(rhs + (int64_t)(enc >> 1) * nd + i, ((enc & 1) ? 1.0 : -1.0) * w[r]);
        }
    }
}

extern "C" int pb_mpsa_system(pb_plan *p, const pb_values *stress, pb_csr **out) {
    NvtxRange nvtx_("pb_mpsa_system");
    if (!p || !out) return fail(PB_EINVAL, "null pointer");
    const double *stress_dev = stress ? stress->buf.as<double>() : p->o_stress.as<double>();
    if (stress && stress->n != p->pat_nnz[0] * p->H.nd * p->H.nd) return fail(PB_EINVAL, "stress values do not belong to this plan");
    if (!stress_dev) return fail(PB_EINVAL, "pb_mpsa_assemble has not been called");
    const HostPlan &H = p->H;
    const int nd = H.nd, nd2 = nd * nd;
    if ((int64_t)p->pat_nnz[2] * nd2 >= 0x7FFFFFFFll) return fail(PB_ENOTIMPL, "system matrix does not fit int32 indices");
    int rc = ensure_face_cells(p);
    if (rc) return rc;
    cudaStream_t st = p->stream;
    // block-expanded CELL_CELL pattern on the device
    DevBuf nip, nix;
    CUDA_TRY(nip.ensure((size_t)(H.nc * nd + 1) * sizeof(int32_t)));
    CUDA_TRY(nix.ensure((size_t)std::max<int64_t>(1, p->pat_nnz[2] * nd2) * sizeof(int32_t)));
    const int block = 256;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((H.nc * 32 + block - 1) / block, (int64_t)kSMs * 16));
    expand_pattern_kernel<<<grid, block, 0, st>>>(H.nc, p->cc_indptr.as<int32_t>(), p->pat_idx[2].as<int32_t>(), nd, nd,
                                                  nip.as<int32_t>(), nix.as<int32_t>());
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    pb_csr *a = nullptr;
    rc = pb_csr_from_device_pattern_(H.nc * nd, H.nc * nd, p->pat_nnz[2] * nd2, nip.as<int32_t>(), nix.as<int32_t>(), &a);
    if (rc) return rc;
    if (p->cf_ip.p && !getenv("POREB200_DIV_SCATTER")) {
        constexpr int kWarps = 4, kCap = 128;           // 4 x 128 x 9 doubles = 36 KB of shared memory per block
        int gridg = (int)std::max<int64_t>(1, std::min<int64_t>((H.nc + kWarps - 1) / kWarps, (int64_t)kSMs * 24));
        div_stress_gather_kernel<kWarps><<<gridg, kWarps * 32, (size_t)kWarps * kCap * nd2 * sizeof(double), st>>>(
            H.nc, nd, p->cf_ip.as<int32_t>(), p->cf_ix.as<int32_t>(), p->cf_sg.as<int8_t>(), p->fc_indptr.as<int32_t>(),
            p->pat_idx[0].as<int32_t>(), stress_dev, p->cc_indptr.as<int32_t>(), p->pat_idx[2].as<int32_t>(),
            pb_csr_data_(a), kCap);
    } else {
        int grid2 = (int)std::max<int64_t>(1, std::min<int64_t>((H.nf * 32 + block - 1) / block, (int64_t)kSMs * 16));
        div_stress_kernel<<<grid2, block, 0, st>>>(H.nf, nd, p->fc_indptr.as<int32_t>(), p->pat_idx[0].as<int32_t>(),
                                                   stress_dev, p->face_cells.as<int32_t>(),
                                                   p->cc_indptr.as<int32_t>(), p->pat_idx[2].as<int32_t>(), pb_csr_data_(a));
    }
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    *out = a;
    return PB_OK;
}

extern "C" int pb_mpsa_rhs(pb_plan *p, const pb_values *bound_stress, const double *bc_values, const double *source,
                           double *rhs) {
    NvtxRange nvtx_("pb_mpsa_rhs");
    if (!p || !bc_values || !rhs) return fail(PB_EINVAL, "null pointer");
    const double *bstress_dev = bound_stress ? bound_stress->buf.as<double>() : p->o_bstress.as<double>();
    if (bound_stress && bound_stress->n != p->pat_nnz[1] * p->H.nd * p->H.nd)
        return fail(PB_EINVAL, "bound_stress values do not belong to this plan");
    if (!bstress_dev) return fail(PB_EINVAL, "pb_mpsa_assemble has not been called");
    const HostPlan &H = p->H;
    const int nd = H.nd;
    cudaStream_t st = p->stream;
    int rc = ensure_face_cells(p);
    if (rc) return rc;
    DevBuf bc, w, r;
    CUDA_TRY(bc.upload(bc_values, (size_t)H.nf * nd, st));
    CUDA_TRY(w.ensure((size_t)H.nf * nd * sizeof(double)));
    CUDA_TRY(r.ensure((size_t)H.nc * nd * sizeof(double)));
    if (source) CUDA_TRY(cudaMemcpyAsync(r.p, source, (size_t)H.nc * nd * sizeof(double), cudaMemcpyHostToDevice, st));
    else CUDA_TRY(cudaMemsetAsync(r.p, 0, (size_t)H.nc * nd * sizeof(double), st));
    const int block = 256;
    int grid = (int)std::max<int64_t>(1, std::min<int64_t>((H.nf * nd * 32 + block - 1) / block, (int64_t)kSMs * 16));
    bound_stress_dot_kernel<<<grid, block, 0, st>>>(H.nf, nd, p->fb_indptr.as<int32_t>(), p->pat_idx[1].as<int32_t>(),
                                                    bstress_dev, bc.as<double>(), w.as<double>());
    int grid2 = (int)std::max<int64_t>(1, std::min<int64_t>((H.nf * nd + block - 1) / block, (int64_t)kSMs * 16));
    neg_div_nd_kernel<<<grid2, block, 0, st>>>(H.nf, nd, p->face_cells.as<int32_t>(), w.as<double>(), r.as<double>());
    g_launches += 2;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(rhs, r.p, (size_t)H.nc * nd * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return PB_OK;
}

// ------------------------------------------------------------------------------------
// MPSA / Biot
// ------------------------------------------------------------------------------------
extern "C" int pb_mpsa_upload(pb_plan *p, const double *stiffness, const uint8_t *bc,
                              const double *robin_weight, double eta, int n_alpha,
                              const double *alpha) {
    NvtxRange nvtx_("pb_mpsa_upload");
    if (!p || !stiffness || !bc) return fail(PB_EINVAL, "null pointer");
    if (!p->have_geo) return fail(PB_EINVAL, "pb_plan_set_geometry has not been called");
    if (n_alpha < 0 || n_alpha > PB_MAX_ALPHA) return fail(PB_EINVAL, "0 <= n_alpha <= 4");
    if (n_alpha > 0 && !alpha) return fail(PB_EINVAL, "null alpha");
    const HostPlan &H = p->H;
    const int nd = H.nd;
    cudaStream_t st = p->stream;
    { int rcs = upload_cell_tensor(p, p->stiff, stiffness, 81); if (rcs) return rcs; }
    CUDA_TRY(p->vbc.upload(bc, (size_t)nd * H.nf, st));
    p->have_vrobw = robin_weight != nullptr;
    p->have_vbasis = false;  // set again by pb_mpsa_set_basis after every upload
    if (robin_weight) CUDA_TRY(p->vrobw.upload(robin_weight, (size_t)nd * nd * H.nf, st));
    if (n_alpha) {
        CUDA_TRY(p->alpha.ensure((size_t)n_alpha * 9 * H.nc * sizeof(double)));
        for (int q = 0; q < n_alpha; ++q) {
            DevBuf one;
            int rca = upload_cell_tensor(p, one, alpha + (size_t)q * 9 * (p->cell_map.p ? p->cell_map_src : H.nc), 9);
            if (rca) return rca;
            CUDA_TRY(cudaMemcpyAsync(p->alpha.as<double>() + (size_t)q * 9 * H.nc, one.p,
                                     (size_t)9 * H.nc * sizeof(double), cudaMemcpyDeviceToDevice, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
    }
    p->n_alpha = n_alpha;
    p->veta = eta;
    if (p->mpsa_cls_nalpha != n_alpha) {
        int rc = build_classes(p, p->mpsa_cls, [&](int nsf, int nsc, int nb, int *n, int *w, int64_t *a,
                                                   int64_t *r) {
            *n = nsf * nd;
            *w = mpsa_width(nd, nsf, nsc, nb, n_alpha);
            *a = mpsa_A_doubles(nd, nsf, nsc, nb, n_alpha);
            *r = mpsa_rest_doubles(nd, nsf, nsc, nb, n_alpha);
        });
        if (rc) return rc;
        p->mpsa_cls_nalpha = n_alpha;
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    p->mpsa_ready = true;
    return PB_OK;
}

extern "C" int pb_mpsa_set_basis(pb_plan *p, const double *basis) {
    if (!p) return fail(PB_EINVAL, "null plan");
    if (!p->mpsa_ready) return fail(PB_EINVAL, "pb_mpsa_upload has not been called");
    p->have_vbasis = basis != nullptr;
    if (basis) {
        const HostPlan &H = p->H;
        CUDA_TRY(p->vbasis.upload(basis, (size_t)H.nd * H.nd * H.nf, p->stream));
        CUDA_TRY(cudaStreamSynchronize(p->stream));
    }
    return PB_OK;
}

extern "C" int pb_mpsa_assemble(pb_plan *p, float *ms) {
    NvtxRange nvtx_("pb_mpsa_assemble");
    if (!p) return fail(PB_EINVAL, "null plan");
    if (!p->mpsa_ready) return fail(PB_EINVAL, "pb_mpsa_upload has not been called");
    const HostPlan &H = p->H;
    const int nd = H.nd;
    cudaStream_t st = p->stream;
    const size_t nfc = (size_t)p->pat_nnz[0], nfb = (size_t)p->pat_nnz[1], ncc = (size_t)p->pat_nnz[2], ncb = (size_t)p->pat_nnz[3];
    MpsaOut o{};
    struct Req { DevBuf *b; double **slot; size_t n; };
    std::vector<Req> reqs = {{&p->o_stress, &o.stress, nfc * nd * nd},
                             {&p->o_bstress, &o.bstress, nfb * nd * nd},
                             {&p->o_bdc, &o.bdc, nfc * nd * nd},
                             {&p->o_bdf, &o.bdf, nfb * nd * nd}};
    for (int a = 0; a < p->n_alpha; ++a) {
        reqs.push_back({&p->o_dd[a], &o.dd[a], ncc * nd});
        reqs.push_back({&p->o_bdd[a], &o.bdd[a], ncb * nd});
        reqs.push_back({&p->o_sg[a], &o.sg[a], nfc * nd});
        reqs.push_back({&p->o_cons[a], &o.cons[a], ncc});
        reqs.push_back({&p->o_bdp[a], &o.bdp[a], nfc * nd});
    }
    for (auto &r : reqs) CUDA_TRY(r.b->ensure(r.n * sizeof(double)));
    CUDA_TRY(cudaEventRecord(p->e0, st));
    for (auto &r : reqs) {
        CUDA_TRY(cudaMemsetAsync(r.b->p, 0, r.n * sizeof(double), st));
        *r.slot = r.b->as<double>();
    }
    int init = INT_MAX;
    CUDA_TRY(cudaMemcpyAsync(p->err.p, &init, sizeof(int), cudaMemcpyHostToDevice, st));
    MpsaParams prm{p->stiff.as<double>(), p->vbc.as<uint8_t>(),
                   p->have_vrobw ? p->vrobw.as<double>() : nullptr,
                   p->have_vbasis ? p->vbasis.as<double>() : nullptr, p->veta, p->n_alpha,
                   p->n_alpha ? p->alpha.as<double>() : nullptr, 1, 81, 1, 9, 9 * H.nc};
    { int rc = nd == 3 ? pb_launch_mpsa3_(p, prm, o) : pb_launch_mpsa2_(p, prm, o); if (rc) return rc; }
    CUDA_TRY(cudaEventRecord(p->e1, st));
    CUDA_TRY(cudaEventSynchronize(p->e1));
    if (ms) CUDA_TRY(cudaEventElapsedTime(ms, p->e0, p->e1));
    return check_singular(p);
}

extern "C" int pb_mpsa_download(pb_plan *p, double *stress, double *bound_stress, double *bdc,
                                double *bdf) {
    if (!p) return fail(PB_EINVAL, "null plan");
    const HostPlan &H = p->H;
    const size_t nd2 = (size_t)H.nd * H.nd;
    int rc;
    if ((rc = dl(p, p->o_stress, stress, (size_t)p->pat_nnz[0] * nd2))) return rc;
    if ((rc = dl(p, p->o_bstress, bound_stress, (size_t)p->pat_nnz[1] * nd2))) return rc;
    if ((rc = dl(p, p->o_bdc, bdc, (size_t)p->pat_nnz[0] * nd2))) return rc;
    if ((rc = dl(p, p->o_bdf, bdf, (size_t)p->pat_nnz[1] * nd2))) return rc;
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    return PB_OK;
}

extern "C" int pb_biot_download(pb_plan *p, int a, double *dd, double *bdd, double *sg, double *cons,
                                double *bdp) {
    if (!p) return fail(PB_EINVAL, "null plan");
    if (a < 0 || a >= p->n_alpha) return fail(PB_EINVAL, "coupling tensor index out of range");
    const HostPlan &H = p->H;
    const size_t nd = H.nd;
    int rc;
    if ((rc = dl(p, p->o_dd[a], dd, (size_t)p->pat_nnz[2] * nd))) return rc;
    if ((rc = dl(p, p->o_bdd[a], bdd, (size_t)p->pat_nnz[3] * nd))) return rc;
    if ((rc = dl(p, p->o_sg[a], sg, (size_t)p->pat_nnz[0] * nd))) return rc;
    if ((rc = dl(p, p->o_cons[a], cons, (size_t)p->pat_nnz[2]))) return rc;
    if ((rc = dl(p, p->o_bdp[a], bdp, (size_t)p->pat_nnz[0] * nd))) return rc;
    CUDA_TRY(cudaStreamSynchronize(p->stream));
    return PB_OK;
}

