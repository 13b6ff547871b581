/*
 * bsp_api.cu -- C-ABI of libbspatom.so (see include/bspatom.h).
 *
 * Host side of the B200 path: groups the caller's (instance, l) problems by
 * (k, nfun, nkp, ka), de-duplicates instances (all l of one potential share
 * S, H0, Q -- the reference recomputes Uij(:,:,0:lmax), matrices.f90:148-153,
 * we keep one Q and form H_l = H0 + c_l Q on the fly), runs the assembly
 * kernel once per instance and the banded eigensolver chunk by chunk.
 * There is no CPU compute path in this file: without a device every entry
 * point returns BSPATOM_ENODEVICE.
 */
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <cmath>
#include <chrono>
#include <mutex>
#include <map>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/bspatom.h"
#include "bsp_assembly.cuh"
#include "bsp_core.h"
#include "bsp_driver.h"
#include "bsp_gemm.cuh"
#include "bsp_kernels.cuh"
#include "bsp_plan.h"

#define BSP_KMIN 3
#define BSP_KMAX 10

static_assert(BSP_PLAN_THREADS == BSP_EIG_THREADS, "the chunk plan sizes a wave in eigen-stage blocks");

namespace {

/* f(std::integral_constant<int, v>{}) for the one v in LO..HI that equals x: the kernels templated on that axis are
 * instantiated for exactly these values; BSPATOM_EUNSUPPORTED for any other x */
template <int LO, int HI, class F>
int dispatch(int x, F &&f)
{
    if constexpr (LO > HI) return BSPATOM_EUNSUPPORTED;
    else return x == LO ? f(std::integral_constant<int, LO>{}) : dispatch<LO + 1, HI>(x, f);
}
template <class F> int with_half_band(int B, F &&f) { return dispatch<BSP_KMIN - 1, BSP_KMAX - 1>(B, f); }
template <class F> int with_order(int k, F &&f) { return dispatch<BSP_KMIN, BSP_KMAX>(k, f); }

struct Options {
    double tau = 1e-4;
    double delta_rel = 1e-6;  /* 1e-4 in round 1: a correction pass then only gains 1e-4 per pass and left |C^T S C - I| ~ 1e-10..1e-9
                                  on a few pairs per batch (found by bspatom_batch_verify over all 408 pencils) */
    double conv_tol = 1e-11;
    double res_tol = 1e-9;
    int max_rounds = 90;      /* cap used when a chunk has to be redone */
    int rounds_enqueued = 26; /* bracketing rounds enqueued up front (surplus ones return at once) */
    int sign_rule = 0;        /* 0: first significant coefficient positive; 1: then the literal CHKPHS of matrices.f90:398-449 */
    int ckpt = 0;             /* check-pointed full-width solves: 0 never (default: measured break-even, DESIGN.md section 12), 1 always, -1 for half bandwidth <= 6 */
    double vec_tol = 1e-12;   /* ||r||_2 / gap above which an eigenpair gets the correction pass after its second solve */
    int min_iters = 2;        /* solves every eigenpair gets (3 = round-1 schedule: everybody gets the correction pass) */
    int trace = 0;        /* diagnostics: print the chunk / copy timeline of every run to stderr */
    int max_iters = 12;
    int chunk = 0; /* 0 = auto */
    long long shifted_chunk = 0; /* systems per chunk of a shifted solve (0: as many as the workspace budget allows) */
    int workers = 2; /* concurrent chunk streams (1..4) */
    int stream_chunks = 6; /* chunks per group when results stream to the host */
    int stream_workers = 2; /* chunk streams when results stream to the host */
#define BSP_MAX_STREAMS 8
#define BSP_MAIL_INTS (1 << 18)
#define BSP_MAIL_REPORT_INTS (1 << 14)
};

struct Group {
    int k = 0, B = 0, n = 0, nkp = 0, ka = 0, npad = 0, nrows = 0, xrows = 0, ldw = 0, FS = 0;
    int ninst = 0, npencil = 0;
    bool any_vtab = false;
    bool band = false; /* ingested from caller-supplied bands (bspatom_band_upload): no knots, nothing to assemble */
    bool rows_built = false; /* S, H0, Q rows hold the assembly (a band group's from the upload); a shifted solve
                                before the first batch_run assembles once, batch_run assembles every time as before */
    int budget_pencils = 0; /* pencils whose workspaces fit the memory budget (decided on the first run) */
    std::vector<int> prob_index; /* pencil -> caller's problem index */
    std::vector<int> inst, nvec;
    std::vector<double> cl;
    std::vector<long long> coff; /* offset of pencil block inside group C  */
    long long c_elems = 0;
    /* device */
    double *d_rt = nullptr, *d_xgwg = nullptr, *d_vtab = nullptr;
    BspInstParams *d_par = nullptr;
    double *d_fbS = nullptr, *d_fbH0 = nullptr, *d_fbQ = nullptr;
    int *d_inst = nullptr, *d_nvec = nullptr, *d_pdinfo = nullptr, *d_bad = nullptr;
    /* device-side state selection (bsp_problem.sel_mode): per pencil rule, the nvec the bracketing sees (0 where
     * the selection needs every eigenvalue to rounding first) and the nvec the refinement sees (written by the
     * selection kernel); sel_off = offset of this group's counts in the handle's mapped selection mailbox */
    bool any_sel = false;
    std::vector<BspSelect> sel;
    BspSelect *d_sel = nullptr;
    int *d_nvec_br = nullptr, *d_nvec_eff = nullptr;
    size_t sel_off = 0;
    double *d_cl = nullptr, *d_E = nullptr, *d_C = nullptr;
    long long *d_coff = nullptr;
    std::vector<int> pdinfo, bad;
};

struct Workspace {
    size_t bytes = 0;
    char *base = nullptr;
};

} // namespace

struct bspatom_handle_s {
    int dev = 0;
    cudaStream_t st = nullptr;
    cudaStream_t st_copy = nullptr; /* D2H of finished chunks overlaps the next chunk's kernels */
    std::vector<cudaEvent_t> chunk_done;
    std::string err;
    Options opt;
    std::vector<Group> groups;
    int nprob = 0;
    std::vector<long long> e_off, c_off; /* per caller problem: offsets in E and C */
    std::vector<int> p_n, p_nvec;
    bool uploaded = false, ran = false;
    bool band = false;                      /* the batch came from bspatom_band_upload */
    std::vector<std::pair<int, int>> outside; /* (problem, info) of band pencils in no group: n = 0, or B not PD */
    double *h_stage = nullptr;              /* pinned staging of bspatom_band_upload, h_stage_cap doubles */
    size_t h_stage_cap = 0;
    Workspace ws;
    /* freed device buffers by byte size: a sweep re-submits batches of identical shape, and
     * cudaMalloc/cudaFree of the multi-GB result buffers costs tens of ms per call */
    std::multimap<size_t, void *> pool;
    size_t pool_bytes = 0;
    /* mailbox: pinned host memory mapped into the device.  Kernels write the small per-run outputs (chunk
     * reports, info flags) straight into it, so the host reads them after a stream synchronise without a
     * D2H transfer -- which would queue behind the bulk eigenvector copies of this or another handle. */
    int *h_counter = nullptr;     /* pinned + mapped, BSP_MAIL_INTS ints */
    int *h_counter_dev = nullptr; /* device view of h_counter */
    int *h_sel = nullptr, *h_sel_dev = nullptr;   /* pinned + mapped: eigenvectors selected per pencil (device-written) */
    size_t h_sel_cap = 0;
    long long c_bytes_copied = 0; /* eigenvector bytes the last run sent to the host */
    size_t budget_bytes = 0;      /* workspace budget of this handle (decided on the first run) */
    bool mail_info = false;       /* the mailbox holds pdinfo / bad of the last run (see run_internal) */
    double stats[27] = {0};
    long long launches = 0;
    /* further chunk streams: auxiliary contexts (own stream, workspace, event pool) that the same host
     * thread enqueues on, so several chunks are in flight and the GPU back-fills the tail waves and the
     * latency-bound kernels of one with blocks of the others */
    std::vector<bspatom_handle_s *> aux; /* helper contexts 1..workers-1 */
    std::mutex mu;
    /* per-kernel-class device timing (CUDA events on the launching stream) */
    std::vector<cudaEvent_t> ev_pool;
    std::vector<int> ev_class; /* class of the pair starting at 2*i */
    size_t ev_used = 0;
    double k_ms[4] = {0, 0, 0, 0};   /* 0 round, 1 factor, 2 back, 3 assembly */
    long long k_cnt[4] = {0, 0, 0, 0};
};

namespace {

#define CU(call)                                                                               \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess) {                                                               \
            char b_[512];                                                                      \
            snprintf(b_, sizeof b_, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            h->err = b_;                                                                       \
            return BSPATOM_ECUDA;                                                              \
        }                                                                                      \
    } while (0)

void pool_flush(bspatom_handle h)
{
    for (auto &kv : h->pool) cudaFree(kv.second);
    h->pool.clear();
    h->pool_bytes = 0;
}

size_t pool_round(size_t bytes) { return (bytes + 511) & ~(size_t)511; }

template <class T>
int dev_alloc(bspatom_handle h, T **p, size_t count)
{
    *p = nullptr;
    if (count == 0) count = 1;
    const size_t bytes = pool_round(count * sizeof(T));
    auto it = h->pool.find(bytes);
    if (it != h->pool.end()) {
        *p = (T *)it->second;
        h->pool_bytes -= bytes;
        h->pool.erase(it);
        return 0;
    }
    cudaError_t e = cudaMalloc((void **)p, bytes);
    if (e != cudaSuccess) {          /* give the pooled memory back and retry once */
        cudaGetLastError();
        pool_flush(h);
        CU(cudaMalloc((void **)p, bytes));
    }
    return 0;
}

template <class T>
void dev_free(bspatom_handle h, T *p, size_t count)
{
    if (!p) return;
    if (count == 0) count = 1;
    const size_t bytes = pool_round(count * sizeof(T));
    h->pool.insert({bytes, (void *)p});
    h->pool_bytes += bytes;
}

void free_group(bspatom_handle h, Group &g)
{
    const size_t per_mat = (size_t)g.nrows * g.FS;
    dev_free(h, g.d_rt, (size_t)g.ninst * g.nkp);
    dev_free(h, g.d_xgwg, (size_t)g.ninst * 64);
    dev_free(h, g.d_vtab, (size_t)g.ninst * (size_t)(g.nkp - 1) * g.ka);
    dev_free(h, g.d_par, (size_t)g.ninst);
    dev_free(h, g.d_fbS, per_mat * g.ninst);
    dev_free(h, g.d_fbH0, per_mat * g.ninst);
    dev_free(h, g.d_fbQ, per_mat * g.ninst);
    dev_free(h, g.d_inst, (size_t)g.npencil);
    dev_free(h, g.d_nvec, (size_t)g.npencil);
    dev_free(h, g.d_sel, (size_t)g.npencil);
    dev_free(h, g.d_nvec_br, (size_t)g.npencil);
    dev_free(h, g.d_nvec_eff, (size_t)g.npencil);
    dev_free(h, g.d_pdinfo, (size_t)g.ninst);
    dev_free(h, g.d_bad, (size_t)g.npencil);
    dev_free(h, g.d_cl, (size_t)g.npencil);
    dev_free(h, g.d_E, (size_t)g.npencil * g.n);
    dev_free(h, g.d_C, (size_t)g.c_elems);
    dev_free(h, g.d_coff, (size_t)g.npencil);
    g = Group();
}

/* row layout of a group's pencils: order n, half bandwidth B */
void set_geometry(Group &G, int n, int B)
{
    G.n = n; G.B = B; G.FS = 2 * B + 2;
    G.npad = BSP_NPAD(n, B);
    G.nrows = BSP_NROWS(G.npad, B);
    G.xrows = G.npad + B + 1;
    G.ldw = ((n + 31) / 32) * 32;
}

/* S, H0 and Q rows of every instance of a group and their positive-definiteness info */
int alloc_group_rows(bspatom_handle h, Group &G)
{
    const size_t per_mat = (size_t)G.nrows * G.FS;
    int rc;
    if ((rc = dev_alloc(h, &G.d_fbS, per_mat * G.ninst))) return rc;
    if ((rc = dev_alloc(h, &G.d_fbH0, per_mat * G.ninst))) return rc;
    if ((rc = dev_alloc(h, &G.d_fbQ, per_mat * G.ninst))) return rc;
    return dev_alloc(h, &G.d_pdinfo, G.ninst);
}

void free_batch(bspatom_handle h)
{
    for (auto &g : h->groups) free_group(h, g);
    h->groups.clear();
    h->uploaded = h->ran = false;
    h->band = false;
    h->outside.clear();
}

/* Gauss-Legendre nodes/weights on [-1,1] by Newton iteration on P_n with the
 * start values and stopping rule the host program uses (gauleg,
 * Modules.f90:112-153: z0 = cos(pi (i-1/4)/(n+1/2)), stop at 10 eps), so that a
 * caller who passes xg = wg = NULL gets the nodes GRID would have produced. */
void gauss_legendre(int n, double *x, double *w)
{
    const double pi = acos(-1.0), tol = 10.0 * BSP_EPS;
    /* dp deliberately outlives the loop body: for odd n the reference skips the
     * Newton loop at the middle node (start value cos(pi/2) ~ 6e-17 is within
     * tol of its initial zold = 0) and forms that weight with the derivative
     * left over from the previous node.  Kept, because a host that lets the
     * library compute the nodes must get what GRID would have handed over;
     * callers wanting exact Gauss-Legendre weights pass xg/wg themselves. */
    double dp = 1.0;
    for (int i = 1; i <= (n + 1) / 2; ++i) {
        double z = cos(pi * (i - 0.25) / (n + 0.5)), zold = 0.0;
        while (fabs(z - zold) > tol) {
            double pa = 1.0, pb = 0.0;
            for (int j = 1; j <= n; ++j) {
                const double pc = pb;
                pb = pa;
                pa = ((2.0 * j - 1.0) * z * pb - (j - 1.0) * pc) / j;
            }
            dp = n * (z * pa - pb) / (z * z - 1.0);
            zold = z;
            z = zold - pa / dp;
        }
        x[i - 1] = -z;
        x[n - i] = z;
        w[i - 1] = 2.0 / ((1.0 - z * z) * dp * dp);
        w[n - i] = w[i - 1];
    }
}

int validate_problem(const bsp_problem &p)
{
    if (p.k < BSP_KMIN || p.k > BSP_KMAX) return BSPATOM_EUNSUPPORTED;
    if (p.nfun < 1) return -3;
    if (p.nkp != p.nfun + p.k) return -3;
    if (p.ka < 1 || p.ka > 32) return -3;
    if (!p.rt) return -3;
    if ((p.xg == nullptr) != (p.wg == nullptr)) return -3;
    if (p.pot_kind == BSPATOM_POT_TABLE && !p.v_tab) return -3;
    if (p.nvec < 0 || p.nvec > p.nfun) return -3;
    if (p.l < 0) return -3;
    if (p.sel_mode != 0 && p.sel_mode != 1) return -3;
    if (p.sel_mode == 1 && (p.sel_extra < 0 || !(p.sel_ecut_a == p.sel_ecut_a) || !(p.sel_ecut_b == p.sel_ecut_b))) return -3;
    return 0;
}

bool same_instance(const bsp_problem &a, const bsp_problem &b)
{
    if (a.pot_kind != b.pot_kind) return false;
    if (a.pot_kind == BSPATOM_POT_TABLE) {
        if (a.v_tab != b.v_tab &&
            memcmp(a.v_tab, b.v_tab, sizeof(double) * (size_t)(a.nkp - 1) * a.ka) != 0)
            return false;
    } else if (memcmp(a.pot_par, b.pot_par, sizeof a.pot_par) != 0) {
        return false;
    }
    if (a.rt != b.rt && memcmp(a.rt, b.rt, sizeof(double) * a.nkp) != 0) return false;
    if ((a.xg == nullptr) != (b.xg == nullptr)) return false;
    if (a.xg && a.xg != b.xg && memcmp(a.xg, b.xg, sizeof(double) * a.ka) != 0) return false;
    if (a.wg && a.wg != b.wg && memcmp(a.wg, b.wg, sizeof(double) * a.ka) != 0) return false;
    return true;
}

uint64_t hash_bytes(const void *p, size_t n, uint64_t h)
{
    const unsigned char *c = (const unsigned char *)p;
    for (size_t i = 0; i < n; ++i) { h ^= c[i]; h *= 1099511628211ull; }
    return h;
}

uint64_t instance_hash(const bsp_problem &p)
{
    uint64_t h = 1469598103934665603ull;
    h = hash_bytes(&p.pot_kind, sizeof p.pot_kind, h);
    if (p.pot_kind == BSPATOM_POT_TABLE) h = hash_bytes(p.v_tab, sizeof(double) * (size_t)(p.nkp - 1) * p.ka, h);
    else h = hash_bytes(p.pot_par, sizeof p.pot_par, h);
    h = hash_bytes(p.rt, sizeof(double) * p.nkp, h);
    if (p.xg) h = hash_bytes(p.xg, sizeof(double) * p.ka, h);
    return h;
}

/* ---- per-kernel timing ---------------------------------------------------- */
int timed_begin(bspatom_handle h, int cls)
{
    if (h->ev_used + 2 > h->ev_pool.size()) {
        for (int i = 0; i < 2; ++i) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return -1;
            h->ev_pool.push_back(e);
        }
        h->ev_class.push_back(cls);
    }
    h->ev_class[h->ev_used / 2] = cls;
    cudaEventRecord(h->ev_pool[h->ev_used], h->st);
    return (int)h->ev_used;
}
void timed_end(bspatom_handle h, int slot)
{
    if (slot < 0) return;
    cudaEventRecord(h->ev_pool[slot + 1], h->st);
    h->ev_used = slot + 2;
}
/* call after the stream has been synchronised */
void timed_collect(bspatom_handle h)
{
    for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]) == cudaSuccess) {
            h->k_ms[h->ev_class[i / 2]] += ms;
            h->k_cnt[h->ev_class[i / 2]] += 1;
        }
    }
    h->ev_used = 0;
}

/* ---- assembly launch ---------------------------------------------------- */
int launch_assembly(bspatom_handle h, int k, const BspAsmArgs &a)
{
    return with_order(k, [&](auto K) {
        constexpr int PK = K * (K + 1) / 2;
        const int per_int = (a.want_pi ? 6 : 4) * PK + (a.want_pi ? K * K : 0);
        const size_t smem = (size_t)(BSP_ASM_TR + K - 1) * per_int * sizeof(double);
        dim3 grid((a.nrows + BSP_ASM_TR - 1) / BSP_ASM_TR, a.ninst);
        if (a.ka <= 16) {
            CU(cudaFuncSetAttribute(bsp_assemble_kernel<K, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            bsp_assemble_kernel<K, 16><<<grid, BSP_ASM_THREADS, smem, h->st>>>(a);
        } else {
            CU(cudaFuncSetAttribute(bsp_assemble_kernel<K, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            bsp_assemble_kernel<K, 32><<<grid, BSP_ASM_THREADS, smem, h->st>>>(a);
        }
        h->launches++;
        CU(cudaGetLastError());
        return 0;
    });
}

/* ---- eigen stage executor ------------------------------------------------ */
template <int B>
struct GpuExec {
    bspatom_handle h;
    BspEigChunk g;
    double *cand_s;
    int *cand_c;
    int open_ok = 0;
    bool ckpt = false;   /* iterations 0 and 1 run check-pointed (no stored factor) */
    cudaEvent_t ev_refine = nullptr; /* recorded between the bracketing and the refinement */
    cudaError_t first_err = cudaSuccess;
    dim3 grid() const { return dim3((g.n + BSP_EIG_THREADS - 1) / BSP_EIG_THREADS, g.npencil); }
    /* compacted passes: a pencil lists 10-17 % of its eigenpairs (64-thread blocks were measured: factor +0.25 ms,
     * no gain overall) */
#ifndef BSP_LISTED_THREADS
#define BSP_LISTED_THREADS 128
#endif
    static constexpr int LISTED_THREADS = BSP_LISTED_THREADS;
    dim3 grid_listed() const { return dim3((g.n + LISTED_THREADS - 1) / LISTED_THREADS, g.npencil); }
    void note() {
        h->launches++;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess && first_err == cudaSuccess) first_err = e;
    }
    void bounds() {
        bsp_bounds_kernel<B><<<g.npencil, BSP_NCAND, 0, h->st>>>(g, cand_s, cand_c); note();
        bsp_bounds_pick_kernel<<<(g.npencil + 127) / 128, 128, 0, h->st>>>(g, cand_s, cand_c); note();
    }
    void round(int r, int max_rounds) {
        const int s = timed_begin(h, 0);
        bsp_round_kernel<B><<<grid(), BSP_EIG_THREADS, 0, h->st>>>(g, r, max_rounds, open_ok); note();
        timed_end(h, s);
    }
    const BspSelect *d_sel = nullptr;   /* selection rules of the chunk's pencils, or null */
    int *d_nvec_eff = nullptr, *sel_report = nullptr;
    cudaEvent_t ev_selected = nullptr;  /* recorded behind the selection kernel: the host sizes the copies with its counts */
    void select() {
        if (!d_sel) return;
        bsp_select_kernel<<<1, 1, 0, h->st>>>(g, d_sel, d_nvec_eff, sel_report); note();
        if (ev_selected) cudaEventRecord(ev_selected, h->st);
    }
    void prepare() {
        if (ev_refine) cudaEventRecord(ev_refine, h->st);
        bsp_prepare_kernel<<<grid(), BSP_EIG_THREADS, 0, h->st>>>(g); note();
    }
    /* iteration 0 solves for the hashed start vector, 1 for S x, later ones for (H - rho S) x */
    template <int RHS>
    void factor_rhs(int it, int optional) {
        if constexpr (RHS != BSP_RHS_RESID) {
            if (ckpt && !optional) { bsp_factor_ckpt_kernel<B, RHS><<<grid(), BSP_EIG_THREADS, 0, h->st>>>(g); return; }
        }
        if (optional) bsp_factor_kernel<B, RHS><<<grid_listed(), LISTED_THREADS, 0, h->st>>>(g, it, optional);
        else bsp_factor_kernel<B, RHS><<<grid(), BSP_EIG_THREADS, 0, h->st>>>(g, it, optional);
    }
    void factor(int it, int optional) {
        const int s = timed_begin(h, 1);
        if (it == 0) factor_rhs<BSP_RHS_START>(it, optional);
        else if (it == 1) factor_rhs<BSP_RHS_SX>(it, optional);
        else factor_rhs<BSP_RHS_RESID>(it, optional);
        note();
        timed_end(h, s);
    }
    void back(int it, int cn, int cx, int optional) {
        const int s = timed_begin(h, 2);
        if (ckpt && it < 2 && !optional) {
            const size_t smem = bsp_back_ckpt_smem<B>(BSP_CKB_THREADS);
            cudaFuncSetAttribute(bsp_back_ckpt_kernel<B>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            dim3 gr((g.n + BSP_CKB_THREADS - 1) / BSP_CKB_THREADS, g.npencil);
            bsp_back_ckpt_kernel<B><<<gr, BSP_CKB_THREADS, smem, h->st>>>(g, it, cx);
        } else if (optional) {
            bsp_back_kernel<B><<<grid_listed(), LISTED_THREADS, 0, h->st>>>(g, it, cn, cx, optional);
        } else {
            bsp_back_kernel<B><<<grid(), BSP_EIG_THREADS, 0, h->st>>>(g, it, cn, cx, optional);
        }
        note();
        timed_end(h, s);
    }
    void check(int it, int select) { bsp_check_kernel<<<grid(), BSP_EIG_THREADS, 0, h->st>>>(g, it, select); note(); }
};

/* one chunk of a run: pencils [p0, p0 + np) of a group, enqueued on chunk stream w; its events are the caller's */
struct ChunkRec {
    int p0 = 0, np = 0, w = 0;
    cudaEvent_t ev[4];                /* start, refinement, finalize, end */
    cudaEvent_t selected = nullptr;   /* null when the group has no selection */
    int *sel_report = nullptr;        /* device view of the selection mailbox slots of this chunk's pencils */
    /* results streaming to the host: `done` is recorded on the chunk's stream behind its last kernel (timed only with
     * the `trace` option, which also times the copy from c0 to c1) and the copy of its results waits for it */
    cudaEvent_t done = nullptr, c0 = nullptr, c1 = nullptr;
};

/* carve the chunk workspace out of one allocation */
struct Carver {
    char *p;
    size_t used = 0;
    template <class T> T *take(size_t count) {
        size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
        T *r = (T *)(p ? p + used : nullptr);
        used += bytes;
        return r;
    }
};

struct ChunkPtrs {
    double *fbH, *pbound, *lo, *hi, *samp_s, *gap, *sigma, *rho, *rho_prev, *scale, *res, *L, *X, *cand_s, *fac;
    double *samp_fm, *flm, *fhm, *beta, *xmax, *res2, *CK;
    int *clo, *chi, *samp_c, *done, *status, *counters, *cand_c, *samp_fe, *fle, *fhe, *side, *olist, *ocount, *rlist, *rcount;
};

size_t carve_chunk(const Group &G, int np, char *base, ChunkPtrs &c, bool ckpt)
{
    Carver cv{base};
    const size_t per = (size_t)np * G.ldw;
    c.fbH = cv.take<double>((size_t)np * G.nrows * G.FS);
    c.pbound = cv.take<double>((size_t)np * 4);
    c.lo = cv.take<double>(2 * per); c.hi = cv.take<double>(2 * per);
    c.clo = cv.take<int>(2 * per); c.chi = cv.take<int>(2 * per);
    c.samp_s = cv.take<double>(2 * per); c.samp_c = cv.take<int>(2 * per);
    c.samp_fm = cv.take<double>(2 * per); c.samp_fe = cv.take<int>(2 * per);
    c.flm = cv.take<double>(per); c.fhm = cv.take<double>(per); c.beta = cv.take<double>(per);
    c.fle = cv.take<int>(per); c.fhe = cv.take<int>(per); c.side = cv.take<int>(per);
    c.gap = cv.take<double>(per); c.done = cv.take<int>(per);
    c.sigma = cv.take<double>(per); c.rho = cv.take<double>(per); c.rho_prev = cv.take<double>(per);
    c.scale = cv.take<double>(per); c.res = cv.take<double>(per); c.status = cv.take<int>(per);
    c.xmax = cv.take<double>(per); c.res2 = cv.take<double>(per);
    c.fac = cv.take<double>(per);
    c.counters = cv.take<int>(64);
    c.olist = cv.take<int>(2 * per); c.ocount = cv.take<int>(4 * (size_t)np);
    c.rlist = cv.take<int>(2 * per); c.rcount = cv.take<int>(2 * (size_t)np);
    c.cand_s = cv.take<double>((size_t)np * BSP_NCAND); c.cand_c = cv.take<int>((size_t)np * BSP_NCAND);
    c.L = cv.take<double>((size_t)np * G.npad * (G.B + 1) * G.ldw);
    c.CK = ckpt ? cv.take<double>((size_t)np * (G.npad / BSP_CK_STEPS(G.B)) * BSP_CK_DOUBLES(G.B) * G.ldw) : nullptr;
    c.X = cv.take<double>((size_t)np * G.xrows * G.ldw);
    return cv.used;
}

bool use_ckpt(bspatom_handle h, const Group &G) { return h->opt.ckpt > 0 || (h->opt.ckpt < 0 && G.B <= 6); }

/* Enqueue the whole stage schedule of pencils [p0, p0+np) of G on h's stream: no host read-back.
 * report: BSP_C_WORDS ints on the device that receive the chunk's control block at the end. */
template <int B>
int enqueue_chunk_b(bspatom_handle h, Group &G, int p0, int np, const ChunkPtrs &c, const BspSchedule &sch,
                    ChunkRec &tm, int *report)
{
    const size_t per_mat = (size_t)G.nrows * G.FS;
    CU(cudaEventRecord(tm.ev[0], h->st));
    {
        dim3 grid((unsigned)((per_mat + 255) / 256), np);
        bsp_combine_kernel<<<grid, 256, 0, h->st>>>(c.fbH, G.d_fbH0, G.d_fbQ, G.d_inst + p0, G.d_cl + p0, per_mat);
        h->launches++;
        CU(cudaGetLastError());
    }
    BspEigChunk g;
    memset(&g, 0, sizeof g);
    g.n = G.n; g.npad = G.npad; g.nrows = G.nrows; g.xrows = G.xrows; g.ldw = G.ldw; g.npencil = np;
    g.fbH = c.fbH; g.fbS = G.d_fbS; g.inst = G.d_inst + p0;
    g.nvec = (G.any_sel ? G.d_nvec_eff : G.d_nvec) + p0;
    g.nvec_br = (G.any_sel ? G.d_nvec_br : G.d_nvec) + p0;
    g.pbound = c.pbound; g.lo = c.lo; g.hi = c.hi; g.clo = c.clo; g.chi = c.chi;
    g.samp_s = c.samp_s; g.samp_c = c.samp_c; g.gap = c.gap; g.done = c.done;
    g.samp_fm = c.samp_fm; g.samp_fe = c.samp_fe; g.flm = c.flm; g.fhm = c.fhm; g.fle = c.fle; g.fhe = c.fhe; g.side = c.side; g.beta = c.beta;
    g.sigma = c.sigma; g.rho = c.rho; g.rho_prev = c.rho_prev; g.scale = c.scale; g.res = c.res; g.xmax = c.xmax;
    g.status = c.status; g.L = c.L; g.CK = c.CK; g.X = c.X; g.counters = c.counters;
    g.olist = c.olist; g.ocount = c.ocount; g.res2 = c.res2; g.rlist = c.rlist; g.rcount = c.rcount;
    g.tau = h->opt.tau; g.delta_rel = h->opt.delta_rel; g.conv_tol = h->opt.conv_tol; g.vec_tol = h->opt.vec_tol;

    GpuExec<B> ex;
    ex.h = h; ex.g = g; ex.cand_s = c.cand_s; ex.cand_c = c.cand_c; ex.ev_refine = tm.ev[1];
    ex.ckpt = (c.CK != nullptr);
    if (G.any_sel) {
        ex.d_sel = G.d_sel + p0; ex.d_nvec_eff = G.d_nvec_eff + p0;
        ex.sel_report = tm.sel_report;
        ex.ev_selected = tm.selected;
    }
    /* every bracket is closed to tau x gap before the hand-over.  Round 1 handed a few stragglers per hundred thousand
     * eigenpairs over open (cheaper by two or three compacted rounds, ~0.3 ms): their first solve then starts from the
     * midpoint of a wide bracket, they pass conv_tol one iteration late with |C^T S C - I| up to 7e-7 (found by
     * bspatom_batch_verify on cfg3), and -- the count being per chunk -- results depended on how a batch was chunked. */
    ex.open_ok = 0;
    bsp_zero_words_kernel<<<1, 32, 0, h->st>>>(c.counters, BSP_C_WORDS);
    h->launches++;
    CU(cudaMemsetAsync(c.ocount, 0, sizeof(int) * 4 * (size_t)np, h->st));
    CU(cudaMemsetAsync(c.rcount, 0, sizeof(int) * 2 * (size_t)np, h->st));
    bsp_enqueue_chunk(ex, sch);
    if (ex.first_err != cudaSuccess) {
        h->err = std::string("eigen stage: ") + cudaGetErrorString(ex.first_err);
        return BSPATOM_ECUDA;
    }
    CU(cudaEventRecord(tm.ev[2], h->st));
    {
        dim3 grid((G.n + BSP_EIG_THREADS - 1) / BSP_EIG_THREADS, np);
        bsp_finalize_kernel<<<grid, BSP_EIG_THREADS, 0, h->st>>>(g, G.d_E + (size_t)p0 * G.n, c.fac, G.d_bad + p0, h->opt.res_tol);
        h->launches++;
        CU(cudaGetLastError());
        int maxnv = 0;
        for (int p = 0; p < np; ++p) maxnv = std::max(maxnv, G.nvec[p0 + p]);
        if (maxnv > 0 && h->opt.sign_rule == 1 && G.d_rt) {
            with_order(G.k, [&](auto K) { bsp_chkphs_kernel<K><<<grid, BSP_EIG_THREADS, 0, h->st>>>(g, G.d_rt, G.nkp, c.fac); return 0; });
            h->launches++;
            CU(cudaGetLastError());
        }
        if (maxnv > 0) {
            dim3 tg((maxnv + 31) / 32, (G.n + 32 * BSP_TR_TILES - 1) / (32 * BSP_TR_TILES), np), tb(32, 8);
            bsp_transpose_kernel<<<tg, tb, 0, h->st>>>(g, c.fac, G.d_C, G.d_coff + p0);
            h->launches++;
            CU(cudaGetLastError());
        }
        bsp_report_kernel<<<1, 32, 0, h->st>>>(g, report);
        h->launches++;
        CU(cudaGetLastError());
    }
    CU(cudaEventRecord(tm.ev[3], h->st));
    return 0;
}

int enqueue_chunk(bspatom_handle h, Group &G, int p0, int np, const ChunkPtrs &c, const BspSchedule &sch,
                  ChunkRec &tm, int *report)
{
    return with_half_band(G.B, [&](auto B) { return enqueue_chunk_b<B>(h, G, p0, np, c, sch, tm, report); });
}

int ensure_workspace(bspatom_handle h, size_t bytes, bspatom_handle pool_owner = nullptr)
{
    if (!pool_owner) pool_owner = h;
    if (h->ws.bytes >= bytes) return 0;
    if (h->ws.base) cudaFree(h->ws.base);
    h->ws.base = nullptr;
    h->ws.bytes = 0;
    if (cudaMalloc((void **)&h->ws.base, bytes) != cudaSuccess) {
        cudaGetLastError();
        pool_flush(pool_owner);
        CU(cudaMalloc((void **)&h->ws.base, bytes));
    }
    h->ws.bytes = bytes;
    return 0;
}

int upload_group_instances(bspatom_handle h, Group &G, const std::vector<const bsp_problem *> &insts)
{
    const int ni = (int)insts.size();
    std::vector<double> rt((size_t)ni * G.nkp), xgwg((size_t)ni * 64, 0.0);
    std::vector<BspInstParams> par(ni);
    std::vector<double> vtab;
    G.any_vtab = false;
    for (int i = 0; i < ni; ++i)
        if (insts[i]->pot_kind == BSPATOM_POT_TABLE) G.any_vtab = true;
    const size_t vt = (size_t)(G.nkp - 1) * G.ka;
    if (G.any_vtab) vtab.assign((size_t)ni * vt, 0.0);
    for (int i = 0; i < ni; ++i) {
        const bsp_problem &p = *insts[i];
        memcpy(&rt[(size_t)i * G.nkp], p.rt, sizeof(double) * G.nkp);
        if (p.xg) {
            memcpy(&xgwg[(size_t)i * 64], p.xg, sizeof(double) * G.ka);
            memcpy(&xgwg[(size_t)i * 64 + 32], p.wg, sizeof(double) * G.ka);
        } else {
            gauss_legendre(G.ka, &xgwg[(size_t)i * 64], &xgwg[(size_t)i * 64 + 32]);
        }
        par[i].pot_kind = p.pot_kind;
        par[i].has_vtab = (p.pot_kind == BSPATOM_POT_TABLE);
        memcpy(par[i].par, p.pot_par, sizeof p.pot_par);
        if (par[i].has_vtab) memcpy(&vtab[(size_t)i * vt], p.v_tab, sizeof(double) * vt);
    }
    int rc;
    if ((rc = dev_alloc(h, &G.d_rt, rt.size()))) return rc;
    if ((rc = dev_alloc(h, &G.d_xgwg, xgwg.size()))) return rc;
    if ((rc = dev_alloc(h, &G.d_par, par.size()))) return rc;
    CU(cudaMemcpyAsync(G.d_rt, rt.data(), rt.size() * sizeof(double), cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(G.d_xgwg, xgwg.data(), xgwg.size() * sizeof(double), cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(G.d_par, par.data(), par.size() * sizeof(BspInstParams), cudaMemcpyHostToDevice, h->st));
    if (G.any_vtab) {
        if ((rc = dev_alloc(h, &G.d_vtab, vtab.size()))) return rc;
        CU(cudaMemcpyAsync(G.d_vtab, vtab.data(), vtab.size() * sizeof(double), cudaMemcpyHostToDevice, h->st));
    }
    CU(cudaStreamSynchronize(h->st)); /* staging vectors die here */
    return 0;
}

/* per-pencil tables of a group (instance, nvec, c_l, C offset, selection rule) and its result buffers */
int upload_group_pencils(bspatom_handle h, Group &G)
{
    int rc;
    if ((rc = dev_alloc(h, &G.d_inst, G.npencil))) return rc;
    if ((rc = dev_alloc(h, &G.d_nvec, G.npencil))) return rc;
    if ((rc = dev_alloc(h, &G.d_cl, G.npencil))) return rc;
    if ((rc = dev_alloc(h, &G.d_coff, G.npencil))) return rc;
    if ((rc = dev_alloc(h, &G.d_bad, G.npencil))) return rc;
    if ((rc = dev_alloc(h, &G.d_E, (size_t)G.npencil * G.n))) return rc;
    if ((rc = dev_alloc(h, &G.d_C, (size_t)G.c_elems))) return rc;
    CU(cudaMemcpyAsync(G.d_inst, G.inst.data(), sizeof(int) * G.npencil, cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(G.d_nvec, G.nvec.data(), sizeof(int) * G.npencil, cudaMemcpyHostToDevice, h->st));
    std::vector<int> nvec_br(G.nvec);
    if (G.any_sel) {
        for (int p = 0; p < G.npencil; ++p) if (G.sel[p].mode) nvec_br[p] = 0;
        if ((rc = dev_alloc(h, &G.d_sel, G.npencil))) return rc;
        if ((rc = dev_alloc(h, &G.d_nvec_br, G.npencil))) return rc;
        if ((rc = dev_alloc(h, &G.d_nvec_eff, G.npencil))) return rc;
        CU(cudaMemcpyAsync(G.d_sel, G.sel.data(), sizeof(BspSelect) * G.npencil, cudaMemcpyHostToDevice, h->st));
        CU(cudaMemcpyAsync(G.d_nvec_br, nvec_br.data(), sizeof(int) * G.npencil, cudaMemcpyHostToDevice, h->st));
        CU(cudaMemcpyAsync(G.d_nvec_eff, G.nvec.data(), sizeof(int) * G.npencil, cudaMemcpyHostToDevice, h->st));
    }
    CU(cudaMemcpyAsync(G.d_cl, G.cl.data(), sizeof(double) * G.npencil, cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(G.d_coff, G.coff.data(), sizeof(long long) * G.npencil, cudaMemcpyHostToDevice, h->st));
    CU(cudaStreamSynchronize(h->st));
    return 0;
}

bspatom_handle new_context(int device_id)
{
    bspatom_handle h = new bspatom_handle_s();
    h->dev = device_id;
    if (cudaSetDevice(device_id) != cudaSuccess || cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->st_copy, cudaStreamNonBlocking) != cudaSuccess ||
        cudaHostAlloc((void **)&h->h_counter, sizeof(int) * BSP_MAIL_INTS, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void **)&h->h_counter_dev, h->h_counter, 0) != cudaSuccess) {
        cudaGetLastError();
        delete h;
        return nullptr;
    }
    return h;
}

void free_context(bspatom_handle h)
{
    if (!h) return;
    for (auto x : h->aux) free_context(x);
    free_batch(h);
    pool_flush(h);
    if (h->ws.base) cudaFree(h->ws.base);
    for (auto e : h->ev_pool) cudaEventDestroy(e);
    if (h->h_counter) cudaFreeHost(h->h_counter);
    if (h->h_sel) cudaFreeHost(h->h_sel);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    for (auto e : h->chunk_done) cudaEventDestroy(e);
    if (h->st_copy) cudaStreamDestroy(h->st_copy);
    if (h->st) cudaStreamDestroy(h->st);
    delete h;
}

int check_device(bspatom_handle h)
{
    if (!h) return -1;
    CU(cudaSetDevice(h->dev));
    return 0;
}

} // namespace

/* ========================================================================= */
extern "C" {

int bspatom_version(void) { return BSPATOM_VERSION; }

void *bspatom_alloc_host(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void bspatom_free_host(void *p)
{
    if (p) cudaFreeHost(p);
}

int bspatom_create(bspatom_handle *out, int device_id)
{
    if (!out) return -1;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return BSPATOM_ENODEVICE;
    if (device_id < 0 || device_id >= ndev) return -2;
    bspatom_handle h = new_context(device_id);
    if (!h) return BSPATOM_ECUDA;
    *out = h;
    return 0;
}

int bspatom_destroy(bspatom_handle h)
{
    if (!h) return 0;
    cudaSetDevice(h->dev);
    free_context(h);
    return 0;
}

const char *bspatom_last_error(bspatom_handle h) { return h ? h->err.c_str() : "null handle"; }

int bspatom_set_option(bspatom_handle h, const char *name, double v)
{
    if (!h) return -1;
    if (!name) return -2;
    std::string s(name);
    if (s == "tau") h->opt.tau = v;
    else if (s == "delta_rel") h->opt.delta_rel = v;
    else if (s == "conv_tol") h->opt.conv_tol = v;
    else if (s == "res_tol") h->opt.res_tol = v;
    else if (s == "max_rounds") h->opt.max_rounds = (int)v;
    else if (s == "trace") h->opt.trace = (int)v;
    else if (s == "min_iters") h->opt.min_iters = std::max(2, (int)v);
    else if (s == "max_iters") h->opt.max_iters = std::max(3, (int)v);
    else if (s == "rounds_enqueued") h->opt.rounds_enqueued = std::max(1, (int)v);
    else if (s == "first_check_round" || s == "check_every") { /* accepted and ignored: the schedule is static */ }
    else if (s == "chunk") h->opt.chunk = (int)v;
    else if (s == "vec_tol") h->opt.vec_tol = v;
    else if (s == "shifted_chunk") h->opt.shifted_chunk = (long long)std::max(0.0, v);
    else if (s == "sign_rule") h->opt.sign_rule = (int)v;
    else if (s == "gemm_variant") bsp_gemm_force = (int)v;   /* process-wide: A/B runs of the contraction kernel only */
    else if (s == "ckpt") { h->opt.ckpt = (int)v; h->budget_bytes = 0; }
    else if (s == "stream_chunks") h->opt.stream_chunks = std::max(1, (int)v);
    else if (s == "stream_workers") h->opt.stream_workers = std::min(BSP_MAX_STREAMS, std::max(1, (int)v));
    else if (s == "workers") h->opt.workers = std::min(BSP_MAX_STREAMS, std::max(1, (int)v));
    else return -2;
    return 0;
}

int bspatom_get_stats(bspatom_handle h, double *out, int nout)
{
    if (!h) return -1;
    if (!out) return -2;
    for (int i = 0; i < nout && i < 27; ++i) out[i] = h->stats[i];
    return 0;
}

/* ------------------------------------------------------------------------- */
int bspatom_batch_upload(bspatom_handle h, int nprob, const bsp_problem *probs)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (nprob < 0) return -2;
    if (nprob > 0 && !probs) return -3;
    free_batch(h);
    h->nprob = nprob;
    h->e_off.assign(nprob + 1, 0);
    h->c_off.assign(nprob + 1, 0);
    h->p_n.assign(nprob, 0);
    h->p_nvec.assign(nprob, 0);
    for (int i = 0; i < nprob; ++i) {
        rc = validate_problem(probs[i]);
        if (rc) { h->err = "invalid bsp_problem at index " + std::to_string(i); return rc; }
        h->p_n[i] = probs[i].nfun;
        h->p_nvec[i] = probs[i].nvec;
        h->e_off[i + 1] = h->e_off[i] + probs[i].nfun;
        h->c_off[i + 1] = h->c_off[i] + (long long)probs[i].nfun * probs[i].nvec;
    }
    /* group by shape */
    std::map<std::vector<int>, int> gid;
    std::vector<std::vector<const bsp_problem *>> ginsts;
    std::vector<std::multimap<uint64_t, int>> ghash;
    std::multimap<uint64_t, int> quick;
    for (int i = 0; i < nprob; ++i) {
        const bsp_problem &p = probs[i];
        std::vector<int> key = {p.k, p.nfun, p.nkp, p.ka};
        auto it = gid.find(key);
        int gi;
        if (it == gid.end()) {
            gi = (int)h->groups.size();
            gid[key] = gi;
            h->groups.emplace_back();
            ginsts.emplace_back();
            ghash.emplace_back();
            Group &G = h->groups.back();
            G.k = p.k; G.nkp = p.nkp; G.ka = p.ka;
            set_geometry(G, p.nfun, p.k - 1);
        } else {
            gi = it->second;
        }
        Group &G = h->groups[gi];
        /* level 1: same pointers and parameters as an earlier problem (all l of one potential) */
        uint64_t qk = 1469598103934665603ull;
        qk = hash_bytes(&p.rt, sizeof p.rt, qk);
        qk = hash_bytes(&p.xg, sizeof p.xg, qk);
        qk = hash_bytes(&p.v_tab, sizeof p.v_tab, qk);
        qk = hash_bytes(&p.pot_kind, sizeof p.pot_kind, qk);
        qk = hash_bytes(p.pot_par, sizeof p.pot_par, qk);
        qk = hash_bytes(&gi, sizeof gi, qk);
        int inst = -1;
        {
            auto range = quick.equal_range(qk);
            for (auto r = range.first; r != range.second; ++r) {
                const bsp_problem &o = *ginsts[gi][r->second];
                if (o.rt == p.rt && o.xg == p.xg && o.wg == p.wg && o.v_tab == p.v_tab && o.pot_kind == p.pot_kind &&
                    memcmp(o.pot_par, p.pot_par, sizeof p.pot_par) == 0) { inst = r->second; break; }
            }
        }
        if (inst < 0) {   /* level 2: equal contents behind different pointers */
            const uint64_t hv = instance_hash(p);
            auto range = ghash[gi].equal_range(hv);
            for (auto r = range.first; r != range.second; ++r)
                if (same_instance(*ginsts[gi][r->second], p)) { inst = r->second; break; }
            if (inst < 0) {
                inst = (int)ginsts[gi].size();
                ginsts[gi].push_back(&p);
                ghash[gi].insert({hv, inst});
            }
            quick.insert({qk, inst});
        }
        G.prob_index.push_back(i);
        G.inst.push_back(inst);
        G.nvec.push_back(p.nvec);
        {
            BspSelect sl;
            sl.mode = p.sel_mode; sl.extra = p.sel_extra; sl.group = p.sel_mode ? p.sel_group : -1; sl.cap = p.nvec;
            sl.ecut_a = p.sel_ecut_a; sl.ecut_b = p.sel_ecut_b;
            G.sel.push_back(sl);
            if (p.sel_mode) G.any_sel = true;
        }
        G.cl.push_back((double)p.l * (double)(p.l + 1) + 2.0 * p.ul_extra);
        G.coff.push_back(G.c_elems);
        G.c_elems += (long long)p.nfun * p.nvec;
    }
    for (size_t gi = 0; gi < h->groups.size(); ++gi) {
        Group &G = h->groups[gi];
        G.ninst = (int)ginsts[gi].size();
        G.npencil = (int)G.prob_index.size();
        if ((rc = upload_group_instances(h, G, ginsts[gi]))) return rc;
        if ((rc = alloc_group_rows(h, G))) return rc;
        if ((rc = upload_group_pencils(h, G))) return rc;
    }
    {
        size_t need = 0;
        for (auto &G : h->groups) { G.sel_off = need; if (G.any_sel) need += (size_t)G.npencil; }
        if (need > h->h_sel_cap) {
            if (h->h_sel) cudaFreeHost(h->h_sel);
            h->h_sel = nullptr; h->h_sel_cap = 0;
            CU(cudaHostAlloc((void **)&h->h_sel, sizeof(int) * need, cudaHostAllocMapped));
            CU(cudaHostGetDevicePointer((void **)&h->h_sel_dev, h->h_sel, 0));
            h->h_sel_cap = need;
        }
    }
    h->uploaded = true;
    return 0;
}

} /* extern "C" */

namespace {

bool is_pinned(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

/* One result-copy stream per device, shared by every handle of the process.  The D2H of the eigenvectors is
 * the longest leg of an end-to-end batch (PCIe), so the order in which batches reach the copy engine decides
 * how well consecutive batches overlap: with one FIFO stream the copies of batch i (all enqueued when batch i
 * was submitted) run before those of batch i+1, batch i returns as early as it can and its handle's next
 * batch computes while batch i+1 is being copied.  Per-handle copy streams would share the link instead and
 * let both batches finish late and together. */
struct CopyQueue {
    std::mutex mu;          /* held while one batch enqueues its chunks: keeps its copies contiguous */
    /* "compute turn": held by a streaming batch from its submission until all but its last small chunks are
     * final.  Two batches computing at the same time only share the SMs -- both become final later, and the
     * copy engine, which works through them in order, waits.  Taking turns, batch i+1 computes at full speed
     * while batch i is being copied, and starts exactly when batch i's tail leaves SMs idle. */
    std::mutex turn;
    cudaStream_t st = nullptr;
};
CopyQueue *copy_queue(int dev)
{
    static std::mutex g_mu;
    static CopyQueue *g_q[128] = {nullptr};
    std::lock_guard<std::mutex> lk(g_mu);
    if (dev < 0 || dev >= 128) return nullptr;
    if (!g_q[dev]) {
        CopyQueue *q = new CopyQueue();
        if (cudaStreamCreateWithFlags(&q->st, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); delete q; return nullptr; }
        g_q[dev] = q;   /* lives as long as the process */
    }
    return g_q[dev];
}

/* enqueue on `cs` the D2H of pencils [p0, p0+np) of group G into the caller's E / C; c_bytes receives the bytes of
 * eigenvectors enqueued */
int copy_chunk_out(bspatom_handle h, Group &G, int p0, int np, double *E, double *C, cudaStream_t cs, const int *nsel,
                   long long &c_bytes)
{
    c_bytes = 0;
    if (nsel) {
        /* device-side selection: E in merged runs, C problem by problem, the selected columns only (a prefix of the
         * problem's column-major block) */
        int rc = copy_chunk_out(h, G, p0, np, E, nullptr, cs, nullptr, c_bytes);
        if (rc) return rc;
        if (C)
            for (int p = p0; p < p0 + np; ++p) {
                const long long nel = (long long)G.n * std::min(nsel[p - p0], G.nvec[p]);
                if (nel > 0) {
                    CU(cudaMemcpyAsync(C + h->c_off[G.prob_index[p]], G.d_C + G.coff[p], sizeof(double) * (size_t)nel, cudaMemcpyDefault, cs));
                    c_bytes += 8 * nel;
                }
            }
        return 0;
    }
    /* pencils of a group are usually contiguous in the caller's order: merge runs */
    int p = p0;
    while (p < p0 + np) {
        int q = p;
        while (q + 1 < p0 + np && G.prob_index[q + 1] == G.prob_index[q] + 1) ++q;
        const int i0 = G.prob_index[p];
        const int cnt = q - p + 1;
        if (E) CU(cudaMemcpyAsync(E + h->e_off[i0], G.d_E + (size_t)p * G.n, sizeof(double) * (size_t)cnt * G.n,
                                  cudaMemcpyDefault, cs));
        if (C) {
            const long long nel = (q + 1 < G.npencil ? G.coff[q + 1] : G.c_elems) - G.coff[p];
            if (nel > 0) CU(cudaMemcpyAsync(C + h->c_off[i0], G.d_C + G.coff[p], sizeof(double) * (size_t)nel,
                                            cudaMemcpyDefault, cs));
            c_bytes += 8 * nel;
        }
        p = q + 1;
    }
    return 0;
}

int run_internal(bspatom_handle h, double *E_out, double *C_out);

} // namespace

extern "C" int bspatom_batch_run(bspatom_handle h)
{
    int rc = check_device(h);
    if (rc) return rc;
    return run_internal(h, nullptr, nullptr);
}

namespace {

int launch_pdcheck(bspatom_handle h, Group &G, cudaStream_t st)
{
    return with_half_band(G.B, [&](auto B) {
        bsp_pdcheck_fast_kernel<B><<<(G.ninst + 31) / 32, 32, 0, st>>>(G.d_fbS, G.n, G.npad, G.nrows, G.ninst, G.d_pdinfo);
        h->launches++;
        CU(cudaGetLastError());
        return 0;
    });
}

/* S, H0 and Q rows of every instance of an assembled group */
int assemble_group(bspatom_handle h, Group &G)
{
    BspAsmArgs a;
    memset(&a, 0, sizeof a);
    a.n = G.n; a.nkp = G.nkp; a.ka = G.ka; a.nrows = G.nrows; a.ninst = G.ninst; a.want_pi = 0;
    a.rt = G.d_rt; a.xgwg = G.d_xgwg; a.par = G.d_par; a.vtab = G.d_vtab;
    a.fb[BSP_MAT_S] = G.d_fbS; a.fb[BSP_MAT_H0] = G.d_fbH0; a.fb[BSP_MAT_Q] = G.d_fbQ;
    const int rc = launch_assembly(h, G.k, a);
    if (!rc) G.rows_built = true;
    return rc;
}

BspRunStats stats_from_report(const int *r)
{
    BspRunStats st = {r[BSP_C_ROUNDS], r[BSP_C_ITERS], r[BSP_C_OPEN_END], r[BSP_C_CROWDED_END], r[BSP_C_UNCONV_END]};
    return st;
}

/* where a run streams its results: the caller's pinned E / C, through the device's copy queue */
struct Delivery {
    double *E, *C;
    CopyQueue *cq;             /* null when nothing streams */
    cudaEvent_t copies_done;   /* recorded behind the run's last copy */
};

/* enqueue on the copy stream, once the chunk is final, the D2H of its results (the selected columns with a
 * device-side selection, whose counts must be in the mailbox by now); the caller holds the queue's lock */
int copy_chunk(bspatom_handle h, Group &G, const ChunkRec &r, const Delivery &out)
{
    CU(cudaStreamWaitEvent(out.cq->st, r.done, 0));
    if (r.c0) CU(cudaEventRecord(r.c0, out.cq->st));
    long long bytes = 0;
    const int rc = copy_chunk_out(h, G, r.p0, r.np, out.E, out.C, out.cq->st, G.any_sel ? h->h_sel + G.sel_off + r.p0 : nullptr, bytes);
    if (rc) return rc;
    h->c_bytes_copied += bytes;
    if (r.c1) CU(cudaEventRecord(r.c1, out.cq->st));
    return 0;
}

int copy_chunk_locked(bspatom_handle h, Group &G, const ChunkRec &r, const Delivery &out)
{
    std::lock_guard<std::mutex> lk(out.cq->mu);
    const int rc = copy_chunk(h, G, r, out);
    if (rc) return rc;
    CU(cudaEventRecord(out.copies_done, out.cq->st));
    return 0;
}

/* the control blocks of chunks [c0, c0 + count) into report: from the mailbox, or from the device */
int read_reports(bspatom_handle h, const int *d_report, int c0, int count, int *report)
{
    const size_t off = (size_t)c0 * BSP_C_WORDS, bytes = (size_t)count * BSP_C_WORDS * sizeof(int);
    if (d_report == h->h_counter_dev) memcpy(report + off, h->h_counter + off, bytes);
    else CU(cudaMemcpy(report + off, d_report + off, bytes, cudaMemcpyDeviceToHost));
    return 0;
}

/* chunk ci ran out of rounds or iterations: run it again with the full limits on h's own stream, copy its results
 * again and re-read its report */
int redo_chunk(bspatom_handle h, Group &G, int largest, ChunkRec &r, const BspSchedule &sch, int *d_report, int ci,
               const Delivery &out, int *report)
{
    int rc;
    ChunkPtrs cc;
    carve_chunk(G, largest, h->ws.base, cc, use_ckpt(h, G));
    CU(cudaMemsetAsync(G.d_bad + r.p0, 0, sizeof(int) * r.np, h->st));
    if ((rc = enqueue_chunk(h, G, r.p0, r.np, cc, sch, r, d_report + (size_t)ci * BSP_C_WORDS))) return rc;
    if (out.cq && !G.any_sel) {
        CU(cudaEventRecord(r.done, h->st));
        if ((rc = copy_chunk_locked(h, G, r, out))) return rc;
    }
    CU(cudaStreamSynchronize(h->st));
    if (out.cq && G.any_sel && (rc = copy_chunk_locked(h, G, r, out))) return rc;   /* sized by the new counts */
    return read_reports(h, d_report, ci, 1, report);
}

/* info flags of every group -> mailbox, on h's stream (all chunk streams are drained at this point) */
int mail_info_flags(bspatom_handle h)
{
    size_t need = 0;
    for (auto &G : h->groups) need += (size_t)G.ninst + (size_t)G.npencil;
    h->mail_info = need <= (size_t)(BSP_MAIL_INTS - BSP_MAIL_REPORT_INTS);
    if (!h->mail_info) return 0;
    size_t off = BSP_MAIL_REPORT_INTS;
    for (auto &G : h->groups) {
        bsp_copy_ints_kernel<<<(G.ninst + 255) / 256, 256, 0, h->st>>>(h->h_counter_dev + off, G.d_pdinfo, G.ninst);
        off += (size_t)G.ninst;
        bsp_copy_ints_kernel<<<(G.npencil + 255) / 256, 256, 0, h->st>>>(h->h_counter_dev + off, G.d_bad, G.npencil);
        off += (size_t)G.npencil;
        h->launches += 2;
    }
    CU(cudaGetLastError());
    return 0;
}

/* `workers` chunk streams with a workspace of `need` bytes each: h and helper contexts, which wait for `after` */
int ready_streams(bspatom_handle h, int workers, size_t need, cudaEvent_t after, std::vector<bspatom_handle> &ctx)
{
    int rc;
    if ((rc = ensure_workspace(h, need))) return rc;
    while ((int)h->aux.size() < workers - 1) {
        bspatom_handle x = new_context(h->dev);
        if (!x) { h->err = "cannot create a helper chunk stream"; return BSPATOM_ECUDA; }
        h->aux.push_back(x);
    }
    ctx.assign(1, h);
    for (int w = 1; w < workers; ++w) {
        h->aux[w - 1]->opt = h->opt;
        if ((rc = ensure_workspace(h->aux[w - 1], need, h))) { h->err = h->aux[w - 1]->err; return rc; }
        CU(cudaStreamWaitEvent(h->aux[w - 1]->st, after, 0));
        ctx.push_back(h->aux[w - 1]);
    }
    return 0;
}

/* diagnostics (option trace): when each chunk was final and when its copy ran, in ms after e0 */
void print_trace(bspatom_handle h, cudaEvent_t e0, const std::vector<ChunkRec> &recs)
{
    for (size_t ci = 0; ci < recs.size(); ++ci) {
        float a = 0, b = 0, c = 0;
        cudaEventElapsedTime(&a, e0, recs[ci].done); cudaEventElapsedTime(&b, e0, recs[ci].c0); cudaEventElapsedTime(&c, e0, recs[ci].c1);
        fprintf(stderr, "[bspatom trace %p] chunk %d stream %d pencils %d final at %.2f ms, copy %.2f -> %.2f ms\n", (void *)h,
                (int)ci, recs[ci].w, recs[ci].np, a, b, c);
    }
}

/* events of a run, released on every exit (there are many CU(...) returns in run_internal) */
struct EventGuard {
    std::vector<cudaEvent_t> ev;
    cudaEvent_t make(unsigned flags, cudaError_t &err) {
        cudaEvent_t e = nullptr;
        err = cudaEventCreateWithFlags(&e, flags);
        if (err == cudaSuccess) ev.push_back(e);
        return e;
    }
    ~EventGuard() { for (auto e : ev) cudaEventDestroy(e); }
};

/* E_out / C_out: pinned host buffers (or NULL).  Every chunk's whole schedule is enqueued up front on one
 * of `workers` streams (each with its own workspace) -- the host reads nothing back while the batch runs,
 * so the GPU never waits for it and the chunk streams back-fill each other's tail waves.  When E_out / C_out
 * are given, each chunk's results are copied out on the device's copy queue as soon as the chunk is final. */
static double host_ms()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

int run_internal(bspatom_handle h, double *E_out, double *C_out)
{
    int rc = 0;
    const double t_run0 = host_ms();
    if (!h->uploaded) { h->err = "batch_run before batch_upload"; return BSPATOM_ESTATE; }
    auto aux_launches = [&] { long long s = 0; for (auto x : h->aux) s += x->launches; return s; };
    const long long launches0 = h->launches + aux_launches();
    for (int i = 0; i < 4; ++i) { h->k_ms[i] = 0; h->k_cnt[i] = 0; }
    h->ev_used = 0;
    for (auto x : h->aux) { for (int i = 0; i < 4; ++i) { x->k_ms[i] = 0; x->k_cnt[i] = 0; } x->ev_used = 0; }
    for (auto e : h->chunk_done) cudaEventDestroy(e);
    h->chunk_done.clear();
    double t_asm = 0, t_val = 0, t_vec = 0, t_fin = 0;
    int rounds = 0, iters = 0, redone = 0;
    long long selected = 0;
    h->c_bytes_copied = 0;
    EventGuard events;
    cudaError_t ev_err = cudaSuccess;
    cudaEvent_t e0 = events.make(cudaEventDefault, ev_err); CU(ev_err);
    cudaEvent_t e1 = events.make(cudaEventDefault, ev_err); CU(ev_err);
    cudaEvent_t e2 = events.make(cudaEventDefault, ev_err); CU(ev_err);
    cudaEvent_t copies_done = events.make(cudaEventDisableTiming, ev_err); CU(ev_err);
    cudaEvent_t pd_done = events.make(cudaEventDisableTiming, ev_err); CU(ev_err);
    CU(cudaEventRecord(pd_done, h->st_copy));
    const bool streaming = (E_out || C_out);
    const Delivery out = {E_out, C_out, streaming ? copy_queue(h->dev) : nullptr, copies_done};
    if (streaming && !out.cq) { h->err = "cannot create the result-copy stream"; return BSPATOM_ECUDA; }
    std::unique_lock<std::mutex> turn;
    if (streaming) turn = std::unique_lock<std::mutex>(out.cq->turn);
    if (streaming) CU(cudaEventRecord(copies_done, out.cq->st));
    CU(cudaEventRecord(e0, h->st));
    const BspSchedule sch_vec = {std::min(h->opt.rounds_enqueued, h->opt.max_rounds), h->opt.min_iters,
                                 std::min(h->opt.max_iters, h->opt.min_iters + 3)};
    /* eigen indices without a vector (nvec < nfun, device-side selection) close their brackets to rounding inside the
     * bracketing: a tail of ~25 cheap (compacted) rounds beyond the 13 of the hand-over; surplus launches are no-ops */
    const BspSchedule sch_val = {std::min(std::max(h->opt.rounds_enqueued, 64), h->opt.max_rounds), sch_vec.min_iters, sch_vec.max_iters};
    const BspSchedule sch_redo = {h->opt.max_rounds, h->opt.min_iters, h->opt.max_iters};
    for (auto &G : h->groups) {
        bool values_only = G.any_sel;
        for (int p = 0; p < G.npencil && !values_only; ++p) values_only = G.nvec[p] < G.n;
        const BspSchedule sch = values_only ? sch_val : sch_vec;
        /* ---- assembly, once per instance ---- */
        CU(cudaEventRecord(e1, h->st));
        if (!G.band) {   /* a band group's rows were written by bspatom_band_upload */
            const int s = timed_begin(h, 3);
            rc = assemble_group(h, G);
            timed_end(h, s);
            if (rc) return rc;
        }
        CU(cudaMemsetAsync(G.d_bad, 0, sizeof(int) * G.npencil, h->st));
        CU(cudaEventRecord(e2, h->st));
        /* positive definiteness of S: one thread per instance walks a whole Cholesky-like sweep (~0.7 ms of pure
         * latency), needed only when the info flags are assembled -- on the side stream, off the critical path */
        CU(cudaStreamWaitEvent(h->st_copy, e2, 0));
        if ((rc = launch_pdcheck(h, G, h->st_copy))) return rc;
        CU(cudaEventRecord(pd_done, h->st_copy));
        /* ---- chunking (bsp_plan.h) ---- */
        ChunkPtrs c;
        const size_t per_pencil = carve_chunk(G, 1, nullptr, c, use_ckpt(h, G));
        if (h->budget_bytes == 0) {
            /* once per handle: cudaMemGetInfo takes milliseconds and stalls behind whatever else the device is
             * doing (another handle's batch), which would delay every submission */
            size_t free_b = 0, total_b = 0;
            CU(cudaMemGetInfo(&free_b, &total_b));
            size_t have = h->ws.bytes + h->pool_bytes;
            for (auto x : h->aux) have += x->ws.bytes;
            h->budget_bytes = std::max<size_t>(std::min<size_t>((free_b + have) / 2, (size_t)64 << 30), 1);
        }
        G.budget_pencils = (int)std::max<size_t>(1, std::min<size_t>(h->budget_bytes / per_pencil, 1 << 24));
        BspPlanInput in;
        in.npencil = G.npencil; in.n = G.n; in.budget_pencils = G.budget_pencils; in.streaming = streaming; in.chunk = h->opt.chunk;
        in.workers = h->opt.workers; in.stream_workers = h->opt.stream_workers; in.stream_chunks = h->opt.stream_chunks;
        if (G.any_sel) for (auto &sl : G.sel) in.sel.push_back({sl.mode, sl.group});
        const BspChunkPlan plan = bsp_plan_chunks(in);
        if (plan.group_too_large) {
            h->err = "a selection group (sel_group) has more pencils than fit one chunk of the workspace";
            return BSPATOM_ENOMEM;
        }
        const int nchunks = plan.nchunks(), workers = plan.streams;
        std::vector<bspatom_handle> ctx;   /* the chunk streams' contexts; helpers start after the assembly */
        if ((rc = ready_streams(h, workers, carve_chunk(G, plan.largest, nullptr, c, use_ckpt(h, G)), e2, ctx))) return rc;
        /* ---- enqueue every chunk; no host read-back in here ---- */
        const bool report_mail = (size_t)nchunks * BSP_C_WORDS <= BSP_MAIL_REPORT_INTS;
        int *d_report = nullptr;
        struct ReportGuard {      /* gives the report buffer back to the handle's pool on every exit */
            bspatom_handle h; int *p = nullptr; size_t count = 0;
            ~ReportGuard() { if (p) dev_free(h, p, count); }
        } report_guard{h};
        if (report_mail) d_report = h->h_counter_dev;
        else {
            if ((rc = dev_alloc(h, &d_report, (size_t)nchunks * BSP_C_WORDS))) return rc;
            report_guard.p = d_report; report_guard.count = (size_t)nchunks * BSP_C_WORDS;
        }
        std::vector<ChunkRec> recs(nchunks);
        for (int ci = 0; ci < nchunks; ++ci) {
            ChunkRec &r = recs[ci];
            r.p0 = plan.bounds[ci]; r.np = plan.bounds[ci + 1] - r.p0;
            for (int i = 0; i < 4; ++i) { r.ev[i] = events.make(cudaEventDefault, ev_err); CU(ev_err); }
            if (G.any_sel) {
                r.selected = events.make(cudaEventDisableTiming, ev_err); CU(ev_err);
                r.sel_report = h->h_sel_dev + G.sel_off + r.p0;
            }
            if (streaming && h->opt.trace) {   /* diagnostics: when was the chunk final, when did its copy run */
                r.c0 = events.make(cudaEventDefault, ev_err); CU(ev_err);
                r.c1 = events.make(cudaEventDefault, ev_err); CU(ev_err);
            }
        }
        std::vector<long long> load(workers, 0);      /* pencils assigned to each stream so far */
        std::unique_lock<std::mutex> copy_lock;
        const double t_lock0 = host_ms();
        if (streaming) copy_lock = std::unique_lock<std::mutex>(out.cq->mu);
        const double t_lock1 = host_ms();
        for (int ci = 0; ci < nchunks; ++ci) {
            ChunkRec &r = recs[ci];
            for (int w = 1; w < workers; ++w) if (load[w] < load[r.w]) r.w = w;
            load[r.w] += r.np;
            bspatom_handle x = ctx[r.w];
            ChunkPtrs cc;
            carve_chunk(G, plan.largest, x->ws.base, cc, use_ckpt(h, G));
            if ((rc = enqueue_chunk(x, G, r.p0, r.np, cc, sch, r, d_report + (size_t)ci * BSP_C_WORDS))) {
                if (x != h) h->err = x->err;
                return rc;
            }
            if (!streaming) continue;
            CU(cudaEventCreateWithFlags(&r.done, h->opt.trace ? cudaEventDefault : cudaEventDisableTiming));
            h->chunk_done.push_back(r.done);
            CU(cudaEventRecord(r.done, x->st));
            /* copies sized by a device-side selection are enqueued below, once the chunk's counts are in the mailbox */
            if (!G.any_sel && (rc = copy_chunk(h, G, r, out))) return rc;
        }
        if (streaming && G.any_sel)
            for (auto &r : recs) {
                /* the selection kernel of the chunk ran right after its bracketing: its counts are in the mapped
                 * mailbox long before the vectors are final */
                CU(cudaEventSynchronize(r.selected));
                if ((rc = copy_chunk(h, G, r, out))) return rc;
            }
        if (streaming) {
            CU(cudaEventRecord(copies_done, out.cq->st));   /* behind this batch's last copy */
            copy_lock.unlock();
        }
        const double t_enq = host_ms();
        if (streaming && &G == &h->groups.back()) {
            /* pass the compute turn on once only the last (small) chunks are left */
            CU(cudaEventSynchronize(recs[nchunks >= 4 ? nchunks - 3 : nchunks - 1].done));
            turn.unlock();
        }
        for (auto x : ctx) CU(cudaStreamSynchronize(x->st));
        if (h->opt.trace)
            fprintf(stderr, "[bspatom trace %p] host clock %.1f ms: entered run; +%.1f lock wait %.1f; +%.1f enqueued; +%.1f kernels done\n",
                    (void *)h, t_run0, t_lock0 - t_run0, t_lock1 - t_lock0, t_enq - t_run0, host_ms() - t_run0);
        if (streaming && h->opt.trace) {
            CU(cudaEventSynchronize(copies_done));
            print_trace(h, e0, recs);
        }
        /* ---- reports; chunks that ran out of rounds / iterations are redone with the full limits ---- */
        std::vector<int> report((size_t)nchunks * BSP_C_WORDS);
        if ((rc = read_reports(h, d_report, 0, nchunks, report.data()))) return rc;
        for (int ci = 0; ci < nchunks; ++ci) {
            BspRunStats st = stats_from_report(&report[(size_t)ci * BSP_C_WORDS]);
            const bool again = (st.brackets_crowded > 0 || st.unconverged > 0) &&
                               (sch.rounds < sch_redo.rounds || sch.max_iters < sch_redo.max_iters);
            if (again) {
                ++redone;
                if ((rc = redo_chunk(h, G, plan.largest, recs[ci], sch_redo, d_report, ci, out, report.data()))) return rc;
                st = stats_from_report(&report[(size_t)ci * BSP_C_WORDS]);
            }
            rounds = std::max(rounds, st.rounds);
            iters = std::max(iters, st.iters);
            selected += report[(size_t)ci * BSP_C_WORDS + BSP_C_SELECTED];
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, recs[ci].ev[0], recs[ci].ev[1])); t_val += ms;
            CU(cudaEventElapsedTime(&ms, recs[ci].ev[1], recs[ci].ev[2])); t_vec += ms;
            CU(cudaEventElapsedTime(&ms, recs[ci].ev[2], recs[ci].ev[3])); t_fin += ms;
        }
        for (auto x : ctx) timed_collect(x);
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e1, e2)); t_asm += ms;
    }
    CU(cudaStreamWaitEvent(h->st, pd_done, 0));
    if ((rc = mail_info_flags(h))) return rc;
    CU(cudaEventRecord(e1, h->st));   /* every chunk stream has been drained */
    CU(cudaStreamSynchronize(h->st));
    {
        auto t0 = std::chrono::steady_clock::now();
        if (streaming) CU(cudaEventSynchronize(copies_done));
        h->stats[21] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    float total = 0;
    CU(cudaEventElapsedTime(&total, e0, e1));
    h->stats[0] = (double)(h->launches + aux_launches() - launches0);
    h->stats[1] = rounds; h->stats[2] = iters;
    /* stage times are summed over the chunk streams: with several streams they overlap in wall time */
    h->stats[3] = t_asm; h->stats[4] = t_val; h->stats[5] = t_vec; h->stats[6] = t_fin; h->stats[7] = total;
    for (int i = 0; i < 4; ++i) {
        h->stats[8 + i] = h->k_ms[i];
        h->stats[12 + i] = (double)h->k_cnt[i];
        for (auto x : h->aux) { h->stats[8 + i] += x->k_ms[i]; h->stats[12 + i] += (double)x->k_cnt[i]; }
    }
    h->stats[19] = redone; h->stats[20] = (double)selected; h->stats[22] = (double)h->c_bytes_copied;
    h->ran = true;
    return 0;
}
} // namespace

extern "C" {

int bspatom_batch_download(bspatom_handle h, double *E, double *C, int *info)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!h->ran) { h->err = "batch_download before batch_run"; return BSPATOM_ESTATE; }
    size_t mail_off = BSP_MAIL_REPORT_INTS;
    if (info)
        for (auto &o : h->outside) info[o.first] = o.second;
    for (auto &G : h->groups) {
        G.pdinfo.resize(G.ninst);
        G.bad.resize(G.npencil);
        if (h->mail_info) {
            memcpy(G.pdinfo.data(), h->h_counter + mail_off, sizeof(int) * G.ninst);
            mail_off += (size_t)G.ninst;
            memcpy(G.bad.data(), h->h_counter + mail_off, sizeof(int) * G.npencil);
            mail_off += (size_t)G.npencil;
        } else {
            CU(cudaMemcpyAsync(G.pdinfo.data(), G.d_pdinfo, sizeof(int) * G.ninst, cudaMemcpyDeviceToHost, h->st));
            CU(cudaMemcpyAsync(G.bad.data(), G.d_bad, sizeof(int) * G.npencil, cudaMemcpyDeviceToHost, h->st));
        }
        long long bytes = 0;
        if ((rc = copy_chunk_out(h, G, 0, G.npencil, E, C, h->st, G.any_sel ? h->h_sel + G.sel_off : nullptr, bytes))) return rc;
        if (G.any_sel) h->c_bytes_copied += bytes;   /* selected columns only */
    }
    CU(cudaStreamSynchronize(h->st));
    if (info) {
        for (auto &G : h->groups)
            for (int p = 0; p < G.npencil; ++p) {
                const int pd = G.pdinfo[G.inst[p]];
                info[G.prob_index[p]] = pd ? G.n + pd : G.bad[p];
            }
    }
    return 0;
}

int bspatom_batch_sizes(bspatom_handle h, int *nprob, int *n)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!nprob) return -2;
    if (!h->uploaded) { h->err = "batch_sizes before batch_upload / band_upload"; return BSPATOM_ESTATE; }
    *nprob = h->nprob;
    if (n) std::copy(h->p_n.begin(), h->p_n.end(), n);
    return 0;
}

int bspatom_get_selection(bspatom_handle h, int *nsel)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!nsel) return -2;
    if (!h->ran) { h->err = "get_selection before a run"; return BSPATOM_ESTATE; }
    for (auto &o : h->outside) nsel[o.first] = 0;
    for (auto &G : h->groups)
        for (int p = 0; p < G.npencil; ++p)
            nsel[G.prob_index[p]] = G.any_sel ? std::min(h->h_sel[G.sel_off + p], G.nvec[p]) : G.nvec[p];
    return 0;
}

} /* extern "C" */

namespace {

/* run + download of an uploaded batch (upload began at host clock t0) */
int run_and_download(bspatom_handle h, double *E, double *C, int *info, double t0)
{
    const double t1 = host_ms();
    /* pinned (cudaHostAlloc / cudaHostRegister / bspatom_alloc_host) output buffers are filled chunk by
     * chunk while the next chunk computes; pageable ones after the run */
    const bool pe = is_pinned(E), pc = is_pinned(C);
    int rc = run_internal(h, pe ? E : nullptr, pc ? C : nullptr);
    if (rc) return rc;
    const double t2 = host_ms();
    rc = bspatom_batch_download(h, pe ? nullptr : E, pc ? nullptr : C, info);
    const double t3 = host_ms();
    h->stats[16] = t1 - t0; h->stats[17] = t2 - t1; h->stats[18] = t3 - t2;   /* host wall ms: upload, run(+overlapped copies), download */
    return rc;
}

bool is_upper(char uplo) { return uplo == 'U' || uplo == 'u'; }

/* every entry of the stored triangle of a symmetric band in LAPACK storage (leading dimension ld) is finite */
bool band_finite(const double *M, int ld, int k, int n, bool upper)
{
    for (int j = 0; j < n; ++j) {
        const int r0 = upper ? std::max(0, k - j) : 0, r1 = upper ? k : std::min(k, n - 1 - j);
        for (int r = r0; r <= r1; ++r)
            if (!std::isfinite(M[(size_t)j * ld + r])) return false;
    }
    return true;
}

/* the stored triangle of a band -> packed storage with leading dimension k+1 (entries outside the matrix become 0) */
void band_pack(double *dst, const double *M, int ld, int k, int n, bool upper)
{
    for (int j = 0; j < n; ++j) {
        const int r0 = upper ? std::max(0, k - j) : 0, r1 = upper ? k : std::min(k, n - 1 - j);
        for (int r = 0; r <= k; ++r) dst[(size_t)j * (k + 1) + r] = (r >= r0 && r <= r1) ? M[(size_t)j * ld + r] : 0.0;
    }
}

/* 0, -3 (malformed; *why says how) or BSPATOM_EUNSUPPORTED */
int validate_band(const bsp_band_pencil &q, const char *&why)
{
    why = "";
    if (q.n < 0) { why = "n < 0"; return -3; }
    if (q.ka < 0 || q.kb < 0) { why = "negative half bandwidth"; return -3; }
    if (q.ka > BSP_KMAX - 1 || q.kb > BSP_KMAX - 1) { why = "half bandwidth above 9"; return BSPATOM_EUNSUPPORTED; }
    if (!is_upper(q.uplo) && q.uplo != 'L' && q.uplo != 'l') { why = "uplo is neither 'U' nor 'L'"; return -3; }
    if (q.ldab < q.ka + 1) { why = "ldab < ka + 1"; return -3; }
    if (q.ldbb < q.kb + 1) { why = "ldbb < kb + 1"; return -3; }
    if (q.n > 0 && (!q.AB || !q.BB)) { why = "AB or BB is NULL"; return -3; }
    if (q.nvec < 0 || q.nvec > q.n) { why = "nvec outside 0..n"; return -3; }
    if (q.n > 0 && !band_finite(q.AB, q.ldab, q.ka, q.n, is_upper(q.uplo))) { why = "NaN or Inf in the stored band of AB"; return -3; }
    if (q.n > 0 && !band_finite(q.BB, q.ldbb, q.kb, q.n, is_upper(q.uplo))) { why = "NaN or Inf in the stored band of BB"; return -3; }
    return 0;
}

template <class T>
size_t doubles_for(size_t count) { return (count * sizeof(T) + sizeof(double) - 1) / sizeof(double); }

} // namespace

extern "C" {

int bspatom_solve_batch(bspatom_handle h, int nprob, const bsp_problem *probs, double *E, double *C, int *info)
{
    const double t0 = host_ms();
    int rc = bspatom_batch_upload(h, nprob, probs);
    if (rc) return rc;
    return run_and_download(h, E, C, info, t0);
}

/* Caller-supplied bands.  The host checks every pencil, then packs all bands and their descriptors into one pinned
 * staging buffer that one copy takes to the device; per (n, B) group one ingest launch writes the full-band rows of
 * S, H0 and Q and one launch checks S for positive definiteness.  Pencils whose S fails are dropped from their
 * group before the per-pencil tables are built, so the solver never sees them. */
int bspatom_band_upload(bspatom_handle h, int nprob, const bsp_band_pencil *pens)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (nprob < 0) return -2;
    if (nprob > 0 && !pens) return -3;
    for (int i = 0; i < nprob; ++i) {   /* before any device work: a rejected batch leaves the handle as it was */
        const char *why = "";
        if ((rc = validate_band(pens[i], why))) { h->err = "bsp_band_pencil at index " + std::to_string(i) + ": " + why; return rc; }
    }
    free_batch(h);
    h->band = true;
    h->nprob = nprob;
    h->e_off.assign(nprob + 1, 0);
    h->c_off.assign(nprob + 1, 0);
    h->p_n.assign(nprob, 0);
    h->p_nvec.assign(nprob, 0);
    std::map<std::pair<int, int>, int> gid;
    std::vector<std::vector<int>> members;
    size_t ndesc = 0, nband = 0;
    for (int i = 0; i < nprob; ++i) {
        const bsp_band_pencil &q = pens[i];
        h->p_n[i] = q.n;
        h->p_nvec[i] = q.nvec;
        h->e_off[i + 1] = h->e_off[i] + q.n;
        h->c_off[i + 1] = h->c_off[i] + (long long)q.n * q.nvec;
        if (q.n == 0) { h->outside.push_back({i, 0}); continue; }
        /* a band wider than the matrix (ka > n - 1 is legal LAPACK storage) holds nothing beyond n - 1 */
        const int B = std::max(std::min(std::max(q.ka, q.kb), q.n - 1), BSP_KMIN - 1);
        auto it = gid.find({q.n, B});
        if (it == gid.end()) {
            it = gid.insert({{q.n, B}, (int)h->groups.size()}).first;
            h->groups.emplace_back();
            members.emplace_back();
            Group &G = h->groups.back();
            G.band = true;
            G.k = B + 1; G.nkp = q.n + G.k; G.ka = 1;
            set_geometry(G, q.n, B);
        }
        members[it->second].push_back(i);
        ++ndesc;
        nband += (size_t)(q.ka + 1 + q.kb + 1) * q.n;
    }
    /* staging: the descriptors of every pencil, group by group, then the packed bands */
    const size_t ddesc = doubles_for<BspBandSrc>(ndesc), total = ddesc + nband;
    if (total > h->h_stage_cap) {
        if (h->h_stage) cudaFreeHost(h->h_stage);
        h->h_stage = nullptr; h->h_stage_cap = 0;
        CU(cudaHostAlloc((void **)&h->h_stage, sizeof(double) * total, cudaHostAllocDefault));
        h->h_stage_cap = total;
    }
    {
        BspBandSrc *desc = (BspBandSrc *)h->h_stage;
        size_t d = 0, off = ddesc;
        for (auto &mem : members)
            for (int i : mem) {
                const bsp_band_pencil &q = pens[i];
                const bool up = is_upper(q.uplo);
                BspBandSrc &s = desc[d++];
                s.ka = q.ka; s.kb = q.kb; s.upper = up;
                s.a_off = (long long)off;
                band_pack(h->h_stage + off, q.AB, q.ldab, q.ka, q.n, up);
                off += (size_t)(q.ka + 1) * q.n;
                s.b_off = (long long)off;
                band_pack(h->h_stage + off, q.BB, q.ldbb, q.kb, q.n, up);
                off += (size_t)(q.kb + 1) * q.n;
            }
    }
    double *d_stage = nullptr;
    if ((rc = dev_alloc(h, &d_stage, total))) return rc;
    struct StageGuard {   /* gives the staging buffer back to the pool on every exit */
        bspatom_handle h; double *p; size_t count;
        ~StageGuard() { cudaStreamSynchronize(h->st); dev_free(h, p, count); }
    } stage_guard{h, d_stage, total};
    if (total) CU(cudaMemcpyAsync(d_stage, h->h_stage, sizeof(double) * total, cudaMemcpyHostToDevice, h->st));
    std::vector<std::vector<int>> pd(h->groups.size());
    size_t d = 0;
    for (size_t gi = 0; gi < h->groups.size(); ++gi) {
        Group &G = h->groups[gi];
        G.ninst = (int)members[gi].size();
        if ((rc = alloc_group_rows(h, G))) return rc;
        const unsigned grid = (unsigned)((G.nrows + BSP_INGEST_TR - 1) / BSP_INGEST_TR) * (unsigned)G.ninst;
        bsp_band_ingest_kernel<<<grid, BSP_INGEST_THREADS, 0, h->st>>>(d_stage, (const BspBandSrc *)d_stage + d, G.n, G.B,
                                                                     G.nrows, G.d_fbS, G.d_fbH0, G.d_fbQ);
        h->launches++;
        CU(cudaGetLastError());
        d += (size_t)G.ninst;
        if ((rc = launch_pdcheck(h, G, h->st))) return rc;
        pd[gi].resize(G.ninst);
        CU(cudaMemcpyAsync(pd[gi].data(), G.d_pdinfo, sizeof(int) * G.ninst, cudaMemcpyDeviceToHost, h->st));
    }
    CU(cudaStreamSynchronize(h->st));
    std::vector<Group> kept;
    for (size_t gi = 0; gi < h->groups.size(); ++gi) {
        Group &G = h->groups[gi];
        for (int s = 0; s < G.ninst; ++s) {
            const int i = members[gi][s];
            if (pd[gi][s]) { h->outside.push_back({i, G.n + pd[gi][s]}); continue; }
            G.prob_index.push_back(i);
            G.inst.push_back(s);
            G.nvec.push_back(pens[i].nvec);
            G.cl.push_back(0.0);
            G.coff.push_back(G.c_elems);
            G.c_elems += (long long)G.n * pens[i].nvec;
        }
        G.npencil = (int)G.prob_index.size();
        if (G.npencil == 0) { free_group(h, G); continue; }
        kept.push_back(G);
    }
    h->groups = kept;
    for (auto &G : h->groups)
        if ((rc = upload_group_pencils(h, G))) return rc;
    h->uploaded = true;
    return 0;
}

int bspatom_solve_band_batch(bspatom_handle h, int nprob, const bsp_band_pencil *pens, double *E, double *C, int *info)
{
    const double t0 = host_ms();
    int rc = bspatom_band_upload(h, nprob, pens);
    if (rc) return rc;
    return run_and_download(h, E, C, info, t0);
}

/* ------------------------------------------------------------------------- */
int bspatom_assemble_band(bspatom_handle h, const bsp_problem *p, double *S, double *H0, double *Q, double *T,
                          double *V, double *R, double *Rinv, double *D)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!p) return -2;
    bsp_problem q = *p;
    q.l = 0; q.nvec = 0;
    if ((rc = validate_problem(q))) return rc;
    Group G;
    G.k = q.k; G.nkp = q.nkp; G.ka = q.ka;
    set_geometry(G, q.nfun, q.k - 1);
    std::vector<const bsp_problem *> insts = {&q};
    G.ninst = 1;
    if ((rc = upload_group_instances(h, G, insts))) { free_group(h, G); return rc; }
    const size_t per_mat = (size_t)G.nrows * G.FS;
    double *d_all = nullptr;
    if ((rc = dev_alloc(h, &d_all, per_mat * BSP_NMAT))) { free_group(h, G); return rc; }
    BspAsmArgs a;
    memset(&a, 0, sizeof a);
    a.n = G.n; a.nkp = G.nkp; a.ka = G.ka; a.nrows = G.nrows; a.ninst = 1; a.want_pi = 1;
    a.rt = G.d_rt; a.xgwg = G.d_xgwg; a.par = G.d_par; a.vtab = G.d_vtab;
    for (int m = 0; m < BSP_NMAT; ++m) a.fb[m] = d_all + per_mat * m;
    rc = launch_assembly(h, G.k, a);
    std::vector<double> host(per_mat * BSP_NMAT);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(host.data(), d_all, host.size() * sizeof(double), cudaMemcpyDeviceToHost, h->st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->st);
        if (e != cudaSuccess) { h->err = cudaGetErrorString(e); rc = BSPATOM_ECUDA; }
    }
    dev_free(h, d_all, per_mat * BSP_NMAT);
    free_group(h, G);
    if (rc) return rc;
    const int n = q.nfun, kd = q.k - 1, FS = 2 * kd + 2;
    double *sym[7] = {S, H0, Q, T, V, R, Rinv};
    for (int m = 0; m < 7; ++m) {
        if (!sym[m]) continue;
        const double *fb = host.data() + per_mat * m;
        for (int j = 0; j < n; ++j)
            for (int r = 0; r <= kd; ++r) {
                const int i = j - kd + r; /* AB(kd+1+i-j, j) 1-based -> row r = kd+i-j */
                sym[m][(size_t)j * (kd + 1) + r] = (i >= 0) ? fb[(size_t)i * FS + (j - i + kd)] : 0.0;
            }
    }
    if (D) {
        const double *fb = host.data() + per_mat * BSP_MAT_D;
        const int ld = 2 * kd + 1;
        for (int j = 0; j < n; ++j)
            for (int r = 0; r < ld; ++r) {
                const int i = j - kd + r;
                D[(size_t)j * ld + r] = (i >= 0 && i < n) ? fb[(size_t)i * FS + (j - i + kd)] : 0.0;
            }
    }
    return 0;
}

} /* extern "C" */

/* ---- driven equation (H - z S) x = b on the resident batch (bspatom_shifted_solve[_z]) ------------------------ */
namespace {

bool device_accessible(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

/* one chunk of a group's systems, laid out in slots (see BspShiftChunk) */
struct ShiftChunkPlan {
    std::vector<int> pen;              /* pencils of the group whose H_l the chunk forms, in row-block order */
    std::vector<int> blk_pen;          /* per block: index into pen                                        */
    std::vector<int> sys;              /* per slot: caller's system or -1                                  */
};

template <int B, class T>
int enqueue_shifted_b(bspatom_handle h, const BspShiftChunk<T> &c, const long long *d_off, T *d_B, T *d_X, int *d_info_out,
                      double *d_berr_out)
{
    const int nblk = c.nslot / BSP_EIG_THREADS;
    const dim3 lay((c.n + 31) / 32, (c.nslot + 31) / 32, (unsigned)c.nrhs), lay_t(32, 8);
    if (c.nrhs > 0) { bsp_shifted_layout_kernel<T, true><<<lay, lay_t, 0, h->st>>>(c, d_off, d_B, c.Bv ? (T *)c.Bv : nullptr, nullptr); h->launches++; }
    bsp_shifted_factor_kernel<B, T><<<nblk, BSP_EIG_THREADS, 0, h->st>>>(c);
    h->launches++;
    if (c.nrhs > 0) {
        /* every step is enqueued up front: finished columns return at once (BspShiftChunk::done) */
        const dim3 grid(nblk, 1, c.nrhs);
        for (int step = 0; step <= BSP_SHIFT_MAXSTEPS + 1; ++step) {
            bsp_shifted_forward_kernel<B, T><<<grid, BSP_EIG_THREADS, 0, h->st>>>(c, step);
            if (step <= BSP_SHIFT_MAXSTEPS) bsp_shifted_back_kernel<B, T><<<grid, BSP_EIG_THREADS, 0, h->st>>>(c, step);
            h->launches += 2;
        }
    }
    bsp_shifted_report_kernel<T><<<nblk, BSP_EIG_THREADS, 0, h->st>>>(c, d_info_out, d_berr_out);
    h->launches++;
    if (c.nrhs > 0) { bsp_shifted_layout_kernel<T, false><<<lay, lay_t, 0, h->st>>>(c, d_off, d_X, c.X, d_info_out); h->launches++; }
    CU(cudaGetLastError());
    return 0;
}

/* device bytes of a chunk: per slot (factor, x, Y, b, state) and per pencil (its H_l rows) */
template <class T>
size_t shift_slot_bytes(const Group &G, int nrhs)
{
    return sizeof(T) * ((size_t)G.n * (G.B + 1) + 3 * (size_t)G.n * nrhs) + (size_t)nrhs * (4 + 8 + 8) + 2 * 8 + 8 + 4 * 3 + 8;
}

template <class T>
int shifted_solve(bspatom_handle h, int nsys, const int *iprob, const double *z, int nrhs, const T *Bm, T *Xm, int *info,
                  double *berr)
{
    constexpr bool CPLX = std::is_same<T, BspZ>::value;
    int rc = check_device(h);
    if (rc) return rc;
    /* every check before any device work: a rejected call leaves the handle as it was */
    if (nsys < 0) return -2;
    if (nsys > 0 && !iprob) return -3;
    if (nsys > 0 && !z) return -4;
    if (nrhs < 0 || nrhs > 65535) return -5;
    const bool any_rhs = (long long)nsys * nrhs > 0;
    if (any_rhs && !Bm) return -6;
    if (any_rhs && !Xm) return -7;
    if (nsys > 0 && !info) return -8;
    if (!h->uploaded) { h->err = "shifted_solve before batch_upload / band_upload"; return BSPATOM_ESTATE; }
    for (int s = 0; s < nsys; ++s) {
        if (iprob[s] < 0 || iprob[s] >= h->nprob) { h->err = "iprob[" + std::to_string(s) + "] out of range"; return -3; }
        const double zr = z[CPLX ? 2 * s : s], zi = CPLX ? z[2 * s + 1] : 0.0;
        if (!std::isfinite(zr) || !std::isfinite(zi)) { h->err = "z of system " + std::to_string(s) + " is not finite"; return -4; }
    }
    /* where each caller problem lives: (group, pencil), or outside every group with its upload info */
    std::vector<int> pg(h->nprob, -1), pp(h->nprob, -1), pinfo(h->nprob, 0);
    for (auto &o : h->outside) pinfo[o.first] = o.second;
    for (size_t gi = 0; gi < h->groups.size(); ++gi)
        for (int p = 0; p < h->groups[gi].npencil; ++p) { pg[h->groups[gi].prob_index[p]] = (int)gi; pp[h->groups[gi].prob_index[p]] = p; }
    std::vector<long long> off(nsys + 1, 0);
    for (int s = 0; s < nsys; ++s) off[s + 1] = off[s] + (long long)h->p_n[iprob[s]] * nrhs;
    for (int s = 0; s < nsys; ++s)
        if (pg[iprob[s]] < 0) { info[s] = pinfo[iprob[s]]; if (berr) berr[s] = 0.0; }
    const size_t total = (size_t)off[nsys];
    h->stats[24] = 0.0; h->stats[25] = 0.0; h->stats[26] = 0.0;

    struct Bufs {   /* gives every device buffer of the call back to the pool on every exit */
        bspatom_handle h;
        std::vector<std::pair<void *, size_t>> v;
        ~Bufs() { cudaStreamSynchronize(h->st); for (auto &b : v) h->pool.insert({pool_round(b.second), b.first}), h->pool_bytes += pool_round(b.second); }
    } bufs{h};
    auto take = [&](auto **p, size_t count) -> int {
        using E = typename std::remove_reference<decltype(**p)>::type;
        const int r = dev_alloc(h, p, count);
        if (!r) bufs.v.push_back({(void *)*p, (count ? count : 1) * sizeof(E)});
        return r;
    };
    T *d_B = nullptr, *d_X = nullptr;
    const bool b_dev = total > 0 && device_accessible(Bm), x_dev = total > 0 && device_accessible(Xm);
    if (total > 0) {
        if (b_dev) d_B = const_cast<T *>(Bm);
        else {
            if ((rc = take(&d_B, total))) return rc;
            CU(cudaMemcpyAsync(d_B, Bm, total * sizeof(T), cudaMemcpyDefault, h->st));
        }
        if (x_dev) d_X = Xm;
        else if ((rc = take(&d_X, total))) return rc;
    }
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    CU(cudaEventCreate(&ev0));
    struct EvGuard { cudaEvent_t &a, &b; ~EvGuard() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); } } evg{ev0, ev1};
    CU(cudaEventCreate(&ev1));
    float ms_total = 0.0f;
    int steps_max = 0;
    unsigned long long corrections = 0;
    std::vector<char> solved(nsys, 0);   /* X_s was written */

    size_t budget = h->budget_bytes;
    if (budget == 0) {
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        budget = std::max<size_t>(std::min<size_t>((free_b + h->ws.bytes + h->pool_bytes) / 2, (size_t)64 << 30), 1);
    }
    constexpr int NT = BSP_EIG_THREADS;
    for (size_t gi = 0; gi < h->groups.size(); ++gi) {
        Group &G = h->groups[gi];
        std::vector<int> mine;
        for (int s = 0; s < nsys; ++s) if (pg[iprob[s]] == (int)gi) mine.push_back(s);
        if (mine.empty()) continue;
        std::stable_sort(mine.begin(), mine.end(), [&](int a, int b) { return pp[iprob[a]] < pp[iprob[b]]; });
        if (!G.band && !G.rows_built && (rc = assemble_group(h, G))) return rc;
        /* blocks of NT slots, each on one pencil; chunks of whole blocks within the workspace budget */
        const size_t per_mat = (size_t)G.nrows * G.FS;
        const size_t slot_b = shift_slot_bytes<T>(G, nrhs), pen_b = per_mat * sizeof(double) + 64;
        /* the layout kernels' grid.y counts tiles of 32 slots: at most 65535 of them per chunk */
        const long long max_slots = (65535LL * 32 / NT) * NT;
        const long long cap_sys = std::min<long long>(h->opt.shifted_chunk > 0 ? h->opt.shifted_chunk : max_slots, max_slots);
        std::vector<ShiftChunkPlan> plans(1);
        size_t bytes = 0;
        for (size_t i = 0; i < mine.size();) {
            const int p = pp[iprob[mine[i]]];
            size_t j = i;
            while (j < mine.size() && pp[iprob[mine[j]]] == p && (long long)(j - i) < NT) ++j;   /* one block */
            ShiftChunkPlan *pl = &plans.back();
            const bool new_pen = pl->pen.empty() || pl->pen.back() != p;
            const size_t add = NT * slot_b + (new_pen ? pen_b : 0);
            const long long used_sys = (long long)pl->blk_pen.size() * NT;
            if (!pl->blk_pen.empty() && (bytes + add > budget || used_sys + NT > cap_sys)) {
                plans.emplace_back();
                pl = &plans.back();
                bytes = 0;
            }
            if (pl->pen.empty() || pl->pen.back() != p) { pl->pen.push_back(p); bytes += pen_b; }
            pl->blk_pen.push_back((int)pl->pen.size() - 1);
            for (size_t k = i; k < j; ++k) pl->sys.push_back(mine[k]);
            for (size_t k = j - i; k < (size_t)NT; ++k) pl->sys.push_back(-1);
            bytes += NT * slot_b;
            i = j;
        }
        for (auto &pl : plans) {
            const int nslot = (int)pl.sys.size(), npen = (int)pl.pen.size(), nblk = nslot / NT;
            /* per-chunk tables, one host-to-device copy */
            std::vector<double> zr(nslot, 0.0), zi(nslot, 0.0), cl(npen);
            std::vector<long long> soff(nslot, 0);
            std::vector<int> ints;   /* blk_inst[nblk], sys[nslot], pen_inst[npen] */
            for (int b = 0; b < nblk; ++b) ints.push_back(G.inst[pl.pen[pl.blk_pen[b]]]);
            for (int k = 0; k < nslot; ++k) {
                const int s = pl.sys[k];
                ints.push_back(s);
                if (s < 0) continue;
                zr[k] = z[CPLX ? 2 * s : s];
                zi[k] = CPLX ? z[2 * s + 1] : 0.0;
                soff[k] = off[s];
            }
            for (int q = 0; q < npen; ++q) { ints.push_back(G.inst[pl.pen[q]]); cl[q] = G.cl[pl.pen[q]]; }
            ints.insert(ints.end(), pl.blk_pen.begin(), pl.blk_pen.end());
            Carver cv{nullptr};
            auto carve = [&](char *base, BspShiftChunk<T> &c, double *&d_z, double *&d_cl, long long *&d_off, int *&d_ints,
                             int *&d_info_out, double *&d_berr_out, double *&d_fbH) {
                cv = Carver{base};
                d_fbH = cv.take<double>((size_t)npen * per_mat);
                c.L = cv.take<T>((size_t)G.n * (G.B + 1) * nslot);
                c.X = cv.take<T>((size_t)G.n * nrhs * nslot);
                c.Y = cv.take<T>((size_t)G.n * nrhs * nslot);
                c.Bv = cv.take<T>((size_t)G.n * nrhs * nslot);
                d_z = cv.take<double>(2 * (size_t)nslot);
                d_cl = cv.take<double>(npen);
                d_off = cv.take<long long>(nslot);
                d_ints = cv.take<int>(ints.size());
                c.info = cv.take<int>(nslot);
                c.done = cv.take<int>((size_t)nrhs * nslot);
                c.berr = cv.take<double>((size_t)nrhs * nslot);
                c.bprev = cv.take<double>((size_t)nrhs * nslot);
                c.steps = cv.take<int>(1);
                c.corrections = cv.take<unsigned long long>(1);
                d_info_out = cv.take<int>(nslot);
                d_berr_out = cv.take<double>(nslot);
                return cv.used;
            };
            BspShiftChunk<T> c;
            memset(&c, 0, sizeof c);
            double *d_z, *d_cl, *d_berr_out, *d_fbH;
            long long *d_off;
            int *d_ints, *d_info_out;
            const size_t need = carve(nullptr, c, d_z, d_cl, d_off, d_ints, d_info_out, d_berr_out, d_fbH);
            if ((rc = ensure_workspace(h, need))) return rc;
            carve(h->ws.base, c, d_z, d_cl, d_off, d_ints, d_info_out, d_berr_out, d_fbH);
            std::vector<double> zz(zr);
            zz.insert(zz.end(), zi.begin(), zi.end());
            CU(cudaMemcpyAsync(d_z, zz.data(), sizeof(double) * zz.size(), cudaMemcpyHostToDevice, h->st));
            CU(cudaMemcpyAsync(d_cl, cl.data(), sizeof(double) * npen, cudaMemcpyHostToDevice, h->st));
            CU(cudaMemcpyAsync(d_off, soff.data(), sizeof(long long) * nslot, cudaMemcpyHostToDevice, h->st));
            CU(cudaMemcpyAsync(d_ints, ints.data(), sizeof(int) * ints.size(), cudaMemcpyHostToDevice, h->st));
            CU(cudaMemsetAsync(c.steps, 0, sizeof(int), h->st));
            CU(cudaMemsetAsync(c.corrections, 0, sizeof(unsigned long long), h->st));
            const int *d_blk_inst = d_ints, *d_sys = d_ints + nblk, *d_pen_inst = d_sys + nslot, *d_blk_pen = d_pen_inst + npen;
            c.n = G.n; c.npad = G.npad; c.nslot = nslot; c.nrhs = nrhs; c.nrows = G.nrows;
            c.fbH = d_fbH; c.fbS = G.d_fbS; c.blk_pen = d_blk_pen; c.blk_inst = d_blk_inst; c.sys = d_sys;
            c.zr = d_z; c.zi = d_z + nslot;
            CU(cudaEventRecord(ev0, h->st));
            {
                /* H_l of the chunk's pencils, as bsp_combine_kernel forms it for the eigen stages */
                dim3 grid((unsigned)((per_mat + 255) / 256), npen);
                bsp_combine_kernel<<<grid, 256, 0, h->st>>>(d_fbH, G.d_fbH0, G.d_fbQ, d_pen_inst, d_cl, per_mat);
                h->launches++;
            }
            rc = with_half_band(G.B, [&](auto B) { return enqueue_shifted_b<B, T>(h, c, d_off, d_B, d_X, d_info_out, d_berr_out); });
            if (rc) return rc;
            CU(cudaEventRecord(ev1, h->st));
            std::vector<int> iout(nslot);
            std::vector<double> bout(nslot);
            int st = 0;
            unsigned long long corr = 0;
            CU(cudaMemcpyAsync(iout.data(), d_info_out, sizeof(int) * nslot, cudaMemcpyDeviceToHost, h->st));
            CU(cudaMemcpyAsync(bout.data(), d_berr_out, sizeof(double) * nslot, cudaMemcpyDeviceToHost, h->st));
            CU(cudaMemcpyAsync(&st, c.steps, sizeof(int), cudaMemcpyDeviceToHost, h->st));
            CU(cudaMemcpyAsync(&corr, c.corrections, sizeof corr, cudaMemcpyDeviceToHost, h->st));
            CU(cudaStreamSynchronize(h->st));
            float ms = 0.0f;
            CU(cudaEventElapsedTime(&ms, ev0, ev1));
            ms_total += ms;
            steps_max = std::max(steps_max, st);
            corrections += corr;
            for (int k = 0; k < nslot; ++k) {
                const int s = pl.sys[k];
                if (s < 0) continue;
                info[s] = iout[k];
                if (berr) berr[s] = bout[k];
                solved[s] = (iout[k] == 0 || iout[k] == G.n + 1);
            }
        }
    }
    if (total > 0 && !x_dev) {
        /* the solutions that were written, in runs of consecutive systems */
        int s = 0;
        while (s < nsys) {
            if (!solved[s] || off[s + 1] == off[s]) { ++s; continue; }
            int q = s;
            while (q + 1 < nsys && solved[q + 1]) ++q;
            CU(cudaMemcpyAsync(Xm + off[s], d_X + off[s], sizeof(T) * (size_t)(off[q + 1] - off[s]), cudaMemcpyDefault, h->st));
            s = q + 1;
        }
        CU(cudaStreamSynchronize(h->st));
    }
    h->stats[24] = ms_total;
    h->stats[25] = steps_max;
    h->stats[26] = (double)corrections;
    return 0;
}

} // namespace

extern "C" {

int bspatom_shifted_solve(bspatom_handle h, int nsys, const int *iprob, const double *z, int nrhs, const double *B, double *X,
                          int *info, double *berr)
{
    return shifted_solve<double>(h, nsys, iprob, z, nrhs, B, X, info, berr);
}

int bspatom_shifted_solve_z(bspatom_handle h, int nsys, const int *iprob, const double *z, int nrhs, const double *B, double *X,
                            int *info, double *berr)
{
    return shifted_solve<BspZ>(h, nsys, iprob, z, nrhs, (const BspZ *)B, (BspZ *)X, info, berr);
}

} /* extern "C" */

#include "bsp_api_extra.cuh"
