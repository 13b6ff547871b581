/*
 * bsp_kernels.cuh -- __global__ wrappers around the per-thread bodies of
 * bsp_core.h plus the small data-movement kernels (band combine, transpose).
 * Thread mapping everywhere: blockIdx.y = pencil, blockIdx.x*blockDim.x +
 * threadIdx.x = eigen index e, so a warp streams 32 consecutive e of one
 * pencil: every workspace access X/L[row][e] is a fully coalesced 256 B
 * line.  The band rows of the pencil, which every thread of a block walks in the
 * same order, come through shared-memory tiles filled by bulk copies (BspRowsStaged).
 */
#ifndef BSP_KERNELS_CUH
#define BSP_KERNELS_CUH

#include <cuda_runtime.h>
#include "bsp_core.h"
#include "bsp_assembly.cuh"
#include <assert.h>

#ifndef BSP_EIG_THREADS
#define BSP_EIG_THREADS 128
#endif

/* resident blocks per SM the register allocator is asked to allow, by half bandwidth:
 * the pivot window is (B+1)(B+2)/2 doubles, so wide bands get fewer blocks instead of spills */
#ifndef BSP_MINB_ROUND
#define BSP_MINB_ROUND 4
#endif
#ifndef BSP_MINB_FACTOR
#define BSP_MINB_FACTOR 3
#endif
#ifndef BSP_MINB_BACK
#define BSP_MINB_BACK 4
#endif
constexpr int bsp_minb_128(int base, int B) { return B <= 6 ? base : (B == 7 ? (base > 3 ? 3 : base) : 2); }
/* `base` counts blocks of 128 threads; larger blocks keep the same number of resident warps */
constexpr int bsp_minb(int base, int B) { return (bsp_minb_128(base, B) * 128) / BSP_EIG_THREADS > 0 ? (bsp_minb_128(base, B) * 128) / BSP_EIG_THREADS : 1; }

__global__ void bsp_zero_words_kernel(int *w, int n)
{
    if ((int)threadIdx.x < n) w[threadIdx.x] = 0;
}

__global__ void bsp_bounds_pick_kernel(BspEigChunk g, const double *cand_s, const int *cand_c)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < g.npencil) bsp_bounds_pick(g, p, cand_s, cand_c);
}

/* true in exactly one thread of the grid: thread 0 of the block that finishes last */
__device__ __forceinline__ bool bsp_last_block(int *arrive)
{
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y * gridDim.z;
        const unsigned t = atomicAdd((unsigned *)arrive, 1u);
        s_last = (t == total - 1);
        if (s_last) { *arrive = 0; __threadfence(); }
    }
    __syncthreads();
    return s_last && threadIdx.x == 0;
}

/* ------------------------------------------------------------------------- *
 * Band-row staging for the sweeps.  Every thread of a block works on the same
 * pencil and walks its band rows in the same order, so the rows are brought
 * into shared memory once per block by the bulk-copy engine (cp.async.bulk,
 * completion on an mbarrier) in tiles of BSP_TILE_GROUPS*(B+1) rows, two tiles
 * in flight, and the threads read them as shared-memory broadcasts.  A forward
 * tile carries B+1 extra rows: step j brings row j+B+1 into the window, so all
 * reads of the steps of tile t stay inside tile t.  Without the staging the leading warp of an SM pays the
 * L2 latency on every new row and the other warps queue up behind it.
 * ------------------------------------------------------------------------- */
template <int B, int G = BSP_TILE_GROUPS(B)>
struct BspTile {
    static constexpr int K1 = B + 1;
    static constexpr int FS = 2 * B + 2;
    static constexpr int TR = G * (B + 1);        /* steps per tile                         */
    static constexpr int ROWS = TR + K1;          /* band rows staged per (forward) tile    */
    static constexpr int DOUBLES = ROWS * FS;     /* per matrix                             */
    static constexpr unsigned ROW_BYTES = FS * 8u; /* 16(B+1): bulk copies stay 16-byte aligned */
    static constexpr int STAGES = 2;
    static constexpr int SMEM_DOUBLES = STAGES * 2 * DOUBLES;
};
static_assert(BSP_SEG_BLOCKS % 4 == 0, "npad must be a whole number of tiles");

__device__ __forceinline__ unsigned bsp_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void bsp_mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bsp_smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void bsp_mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "BSP_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra BSP_DONE_%=;\n\t"
        "bra BSP_WAIT_%=;\n\t"
        "BSP_DONE_%=:\n\t}" ::"r"(bsp_smem_u32(bar)), "r"(parity) : "memory");
}

/* one thread: expect `bytes` on the barrier and start the bulk copy global -> shared */
__device__ __forceinline__ void bsp_bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(bsp_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(bsp_smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void bsp_mbar_expect(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bsp_smem_u32(bar)), "r"(bytes) : "memory");
}

/* row source of the sweeps (see BspRowsGlobal): tiles staged in shared memory.  One object per sweep; every
 * thread of the block calls the same sequence (the release is a block barrier), thread 0 drives the copies. */
template <int B, int RING = 0, int G = BSP_TILE_GROUPS(B)>
struct BspRowsStaged {
    using T = BspTile<B, G>;
    static constexpr bool GL = false;
    static constexpr int TR = T::TR;
    static constexpr int RHS_RING = RING;   /* groups of right-hand-side look-ahead in flight (factor kernel) */
    double *sm;
    uint64_t *bars;   /* two mbarriers, count 1, not used by an earlier sweep of this launch */
    const double *gH, *gS;
    double *rq = nullptr;   /* this thread's column of the look-ahead ring: rq[slot_row * blockDim.x] */
#if defined(BSP_DEBUG)
    int dbg_issued = 0, dbg_acquired = 0;   /* thread 0: tiles issued / acquired so far (each stage: issue -> acquire -> release) */
#endif

    __device__ __forceinline__ void rhs_issue(int slot_row, const double *src)
    {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(bsp_smem_u32(rq + (size_t)slot_row * blockDim.x)), "l"(src) : "memory");
    }
    __device__ __forceinline__ void rhs_zero(int slot_row) { rq[(size_t)slot_row * blockDim.x] = 0.0; }
    __device__ __forceinline__ void rhs_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
    template <int N>
    __device__ __forceinline__ void rhs_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
    __device__ __forceinline__ double rhs_read(int slot_row) { return rq[(size_t)slot_row * blockDim.x]; }

    __device__ __forceinline__ void issue(int seq, const double *srcH, const double *srcS, int rows, int dst_row)
    {
        const int stage = seq & 1;
        double *dH = sm + (size_t)stage * 2 * T::DOUBLES + (size_t)dst_row * T::FS, *dS = dH + T::DOUBLES;
        const unsigned bytes = (unsigned)rows * T::ROW_BYTES;
#if defined(BSP_DEBUG)
        /* tiles go out in sequence, at most two ahead of the one being consumed, and fit their stage */
        BSP_ASSERT(seq == dbg_issued && dbg_issued - dbg_acquired <= 2 && (dst_row + rows) * T::FS <= T::DOUBLES && rows > 0);
        ++dbg_issued;
#endif
        bsp_mbar_expect(bars + stage, 2u * bytes);
        bsp_bulk_g2s(dH, srcH, bytes, bars + stage);
        bsp_bulk_g2s(dS, srcS, bytes, bars + stage);
    }
    __device__ __forceinline__ void acquire(int seq, const double *&tH, const double *&tS)
    {
        const int stage = seq & 1;
#if defined(BSP_DEBUG)
        if (threadIdx.x == 0) { BSP_ASSERT(seq == dbg_acquired && seq < dbg_issued); ++dbg_acquired; }
#endif
        bsp_mbar_wait(bars + stage, (unsigned)(seq >> 1) & 1u);
        tH = sm + (size_t)stage * 2 * T::DOUBLES;
        tS = tH + T::DOUBLES;
    }
    __device__ __forceinline__ void fence_before_first_copy()
    {
        /* the stages may alias shared memory the block wrote with ordinary stores before the last barrier */
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    /* forward: tile t = rows t*TR .. t*TR + ROWS - 1 */
    __device__ __forceinline__ void issue_forward(int t)
    {
        issue(t, gH + (size_t)t * T::TR * T::FS, gS + (size_t)t * T::TR * T::FS, T::ROWS, 0);
    }
    __device__ __forceinline__ void begin_forward(int ntiles)
    {
        if (threadIdx.x == 0) {
            fence_before_first_copy();
            issue_forward(0);
            if (ntiles > 1) issue_forward(1);
        }
    }
    __device__ __forceinline__ void acquire_forward(int t, const double *&tH, const double *&tS) { acquire(t, tH, tS); }
    __device__ __forceinline__ void release_forward(int t, int ntiles)
    {
        __syncthreads(); /* every thread is through with this stage: it may be refilled */
        if (threadIdx.x == 0 && t + 2 < ntiles) issue_forward(t + 2);
    }
    /* backward: tile t = rows t*TR .. (t+1)*TR - 1, taken in descending t */
    __device__ __forceinline__ void issue_backward(int t, int ntiles)
    {
        issue(ntiles - 1 - t, gH + (size_t)t * T::TR * T::FS, gS + (size_t)t * T::TR * T::FS, T::TR, 0);
    }
    __device__ __forceinline__ void begin_backward(int ntiles)
    {
        if (threadIdx.x == 0) {
            fence_before_first_copy();
            issue_backward(ntiles - 1, ntiles);
            if (ntiles > 1) issue_backward(ntiles - 2, ntiles);
        }
    }
    __device__ __forceinline__ void acquire_backward(int t, int ntiles, const double *&tH, const double *&tS)
    {
        acquire(ntiles - 1 - t, tH, tS);
    }
    __device__ __forceinline__ void release_backward(int t, int ntiles)
    {
        __syncthreads();
        if (threadIdx.x == 0 && t - 2 >= 0) issue_backward(t - 2, ntiles);
    }
    /* backward order with forward-sized tiles (rows t*TR .. t*TR + ROWS - 1): the check-pointed back sweep
     * re-eliminates a tile (needs the B+1 rows beyond it) before it back-substitutes it */
    __device__ __forceinline__ void issue_backward_wide(int t, int ntiles)
    {
        issue(ntiles - 1 - t, gH + (size_t)t * T::TR * T::FS, gS + (size_t)t * T::TR * T::FS, T::ROWS, 0);
    }
    __device__ __forceinline__ void begin_backward_wide(int ntiles)
    {
        if (threadIdx.x == 0) {
            fence_before_first_copy();
            issue_backward_wide(ntiles - 1, ntiles);
            if (ntiles > 1) issue_backward_wide(ntiles - 2, ntiles);
        }
    }
    __device__ __forceinline__ void acquire_backward_wide(int t, int ntiles, const double *&tH, const double *&tS)
    {
        acquire(ntiles - 1 - t, tH, tS);
    }
    __device__ __forceinline__ void release_backward_wide(int t, int ntiles)
    {
        __syncthreads();
        if (threadIdx.x == 0 && t - 2 >= 0) issue_backward_wide(t - 2, ntiles);
    }
};

__device__ __forceinline__ void bsp_stage_bars_init(uint64_t *bars)
{
    if (threadIdx.x == 0) {
        bsp_mbar_init(bars, 1);
        bsp_mbar_init(bars + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
}

/* spectrum bounds: the BSP_NCAND shifts of the ladder, one thread each, band rows staged like in the sweeps */
template <int B>
__global__ void __launch_bounds__(BSP_NCAND) bsp_bounds_kernel(BspEigChunk g, double *cand_s, int *cand_c)
{
    __shared__ __align__(128) double sm[BspTile<B>::SMEM_DOUBLES];
    __shared__ __align__(8) uint64_t bars[2];
    const int p = blockIdx.x, lane = threadIdx.x;
    constexpr int FS = 2 * B + 2;
    bsp_stage_bars_init(bars);
    double sig, pivmin;
    bsp_bounds_shift<B>(g, p, lane, sig, pivmin);
    __syncthreads();    /* publishes the mbarrier initialisation */
    BspRowsStaged<B> src{sm, bars, g.fbH + (size_t)p * g.nrows * FS, g.fbS + (size_t)g.inst[p] * g.nrows * FS};
    cand_s[p * BSP_NCAND + lane] = sig;
    cand_c[p * BSP_NCAND + lane] = bsp_sturm_sweep<B>(src, g.npad, true, sig, pivmin, nullptr, nullptr, nullptr);
}

__device__ __forceinline__ float bsp_frcp_fast(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

/* block-cooperative form of bsp_deflation_sum: the bracket midpoints of the pencil go through shared memory in
 * tiles of BSP_DEFL_TILE; same four summation chains as the plain form */
#define BSP_DEFL_TILE 1024
__device__ __forceinline__ double bsp_deflation_sum_block(const BspEigChunk &g, int p, int e, int round, const BspRoundState &st,
                                                          bool want, double *sm)
{
    const int n = g.n;
    const size_t rd = (size_t)(round & 1) * (size_t)g.npencil * g.ldw;
    const double *Lo = g.lo + rd + (size_t)p * g.ldw, *Hi = g.hi + rd + (size_t)p * g.ldw;
    const double mid = 0.5 * (st.lo + st.hi);
    float b0 = 0.0f, b1 = 0.0f, b2 = 0.0f, b3 = 0.0f;
    for (int k0 = 0; k0 < n; k0 += BSP_DEFL_TILE) {
        const int cnt = min(BSP_DEFL_TILE, n - k0), cnt4 = (cnt + 3) & ~3;
        __syncthreads();
        for (int i = threadIdx.x; i < cnt4; i += blockDim.x)
            sm[i] = (i < cnt) ? 0.5 * (Lo[k0 + i] + Hi[k0 + i]) : INFINITY; /* 1/(mid - inf) = 0 */
        __syncthreads();
        if (want) {
            const int el = e - k0;
#pragma unroll 2
            for (int i = 0; i < cnt4; i += 4) {
                const double2 m01 = *reinterpret_cast<const double2 *>(sm + i);
                const double2 m23 = *reinterpret_cast<const double2 *>(sm + i + 2);
                const float d0 = (float)(mid - m01.x), d1 = (float)(mid - m01.y);
                const float d2 = (float)(mid - m23.x), d3 = (float)(mid - m23.y);
                const float r0 = bsp_frcp_fast(d0), r1 = bsp_frcp_fast(d1), r2 = bsp_frcp_fast(d2), r3 = bsp_frcp_fast(d3);
                b0 += (i != el && d0 != 0.0f) ? r0 : 0.0f;
                b1 += (i + 1 != el && d1 != 0.0f) ? r1 : 0.0f;
                b2 += (i + 2 != el && d2 != 0.0f) ? r2 : 0.0f;
                b3 += (i + 3 != el && d3 != 0.0f) ? r3 : 0.0f;
            }
        }
    }
    __syncthreads();
    return (double)b0 + (double)b1 + (double)b2 + (double)b3;
}

/* One bracketing round.  Threads are mapped to the eigen indices that still have work through the compaction
 * list of the pencil (g.olist / g.ocount, built by the previous round): a bracket that is done re-publishes its
 * state once more (so that both bracket buffers hold it) and then drops out, blocks beyond the list return at
 * once, and the cost of the late rounds follows the number of open brackets instead of n.  The order of the list
 * (atomic appends) varies from run to run; the result of an eigen index does not depend on its slot. */
template <int B>
__global__ void __launch_bounds__(BSP_EIG_THREADS, bsp_minb(BSP_MINB_ROUND, B)) bsp_round_kernel(BspEigChunk g, int round, int max_rounds, int open_ok)
{
    using T = BspTile<B>;
    constexpr int SMD = T::SMEM_DOUBLES > BSP_DEFL_TILE ? T::SMEM_DOUBLES : BSP_DEFL_TILE;
    __shared__ __align__(128) double sm[SMD];
    __shared__ __align__(8) uint64_t bars[2];
    if (g.counters[BSP_C_BRACKETED]) return;       /* written by the previous kernel: grid-uniform */
    const int p = blockIdx.y, slot = blockIdx.x * blockDim.x + threadIdx.x;
    const bool compact = g.olist != nullptr;
    const int rdb = round & 1, wrb = (round + 1) & 1;
    /* two lists per pencil in one array: open brackets from the front (they sweep: kept dense), brackets that
     * became done in the previous round from the back (they only re-publish) */
    const bool listed = compact && round > 0;
    const int cnt_open = listed ? g.ocount[(rdb * g.npencil + p) * 2] : g.n;
    const int cnt = listed ? cnt_open + g.ocount[(rdb * g.npencil + p) * 2 + 1] : g.n;
    if ((int)(blockIdx.x * blockDim.x) < cnt) {     /* block-uniform */
        const bool valid = slot < cnt;
        const int *list = g.olist + ((size_t)rdb * g.npencil + p) * g.ldw;
        BSP_ASSERT(cnt >= 0 && cnt <= g.n && cnt_open >= 0 && cnt_open <= cnt);
        const int e = !valid ? g.n : (!listed ? slot : (slot < cnt_open ? list[slot] : list[g.ldw - 1 - (slot - cnt_open)]));
        BSP_ASSERT(e >= 0 && e <= g.n);
        bsp_stage_bars_init(bars);
        BspRoundState st;
        st.want_defl = 0; st.want_count = 0; st.done = 1; st.was_done = 1; st.lo = st.hi = 0.0;
        if (valid) bsp_round_begin(g, p, e, round, st);
        /* the barriers below also publish the mbarrier initialisation */
        double bsum = 0.0;
        if (__syncthreads_or(st.want_defl)) bsum = bsp_deflation_sum_block(g, p, e, round, st, st.want_defl != 0, sm);
        if (valid) bsp_round_pick(st, bsum);
        if (__syncthreads_or(st.want_count)) {
            constexpr int FS = 2 * B + 2;
            BspRowsStaged<B> src{sm, bars, g.fbH + (size_t)p * g.nrows * FS, g.fbS + (size_t)g.inst[p] * g.nrows * FS};
            double fm;
            int fe;
            const double pivmin = st.want_count ? bsp_round_pivmin(g, p, st.s) : 1.0;
            const int c = bsp_sturm_sweep<B>(src, g.npad, st.want_count != 0, st.s, pivmin, nullptr, &fm, &fe);
            if (st.want_count) { st.c = c; st.sfm = fm; st.sfe = fe; }
        }
        if (valid) {
            bsp_round_end(g, p, e, round, st);
            if (compact && !st.was_done) {
                int *wl = g.olist + ((size_t)wrb * g.npencil + p) * g.ldw;
                const int at = !st.done ? atomicAdd(g.ocount + (wrb * g.npencil + p) * 2, 1)
                                        : g.ldw - 1 - atomicAdd(g.ocount + (wrb * g.npencil + p) * 2 + 1, 1);
                BSP_ASSERT(at >= 0 && at < g.ldw);
                wl[at] = e;
            }
        }
    }
    if (bsp_last_block(g.counters + BSP_C_ARRIVE)) {
        bsp_round_ctl(g, round, max_rounds, open_ok);
        /* the counts this round consumed are the ones the next round appends to */
        if (compact) for (int q = 0; q < 2 * g.npencil; ++q) g.ocount[rdb * 2 * g.npencil + q] = 0;
    }
}

/* device-side state selection of the chunk (one thread: the running maximum over l is sequential); the counts also
 * go to the mapped mailbox, from which the host sizes the result copies while the refinement runs */
__global__ void bsp_select_kernel(BspEigChunk g, const BspSelect *sel, int *nvec_eff, int *report)
{
    bsp_select_states(g, sel, nvec_eff, report);
    __threadfence_system();
}

__global__ void bsp_prepare_kernel(BspEigChunk g)
{
    bsp_refine_prepare(g, blockIdx.y, blockIdx.x * blockDim.x + threadIdx.x);
}

#ifndef BSP_RHS_RING
#define BSP_RHS_RING 3   /* groups of B+1 rows of x in flight per thread in the factor kernel */
#endif
/* wide bands: fewer groups, so that tiles + ring stay within the 48 KB of static shared memory */
__host__ __device__ constexpr int bsp_rhs_ring(int B) { return B <= 6 ? BSP_RHS_RING : (B == 7 ? (BSP_RHS_RING < 2 ? BSP_RHS_RING : 2) : 1); }
/* thread -> (eigen index, factor column): identity at full width; in an optional (compacted) pass the slot-th
 * entry of the list the previous convergence check wrote.  Returns false for the whole block when it has nothing
 * to do (block-uniform). */
__device__ __forceinline__ bool bsp_refine_map(const BspEigChunk &g, int p, int iter, int listed, int &e, bool &active)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (listed) {
        const int cnt = g.rcount[((iter - 1) & 1) * g.npencil + p];
        if ((int)(blockIdx.x * blockDim.x) >= cnt) return false;
        active = slot < cnt;
        e = active ? g.rlist[((size_t)((iter - 1) & 1) * g.npencil + p) * g.ldw + slot] : 0;
        BSP_ASSERT(cnt <= g.n && e >= 0 && e < g.n);
    } else {
        e = slot;
        active = bsp_refine_active(g, p, e);
    }
    return true;
}

/* RHS: BSP_RHS_* (bsp_factor_forward_rhs) */
template <int B, int RHS>
__global__ void __launch_bounds__(BSP_EIG_THREADS, bsp_minb(BSP_MINB_FACTOR, B)) bsp_factor_kernel(BspEigChunk g, int iter, int optional)
{
    __shared__ __align__(128) double sm[BspTile<B>::SMEM_DOUBLES];
    constexpr int RING = bsp_rhs_ring(B);
    __shared__ __align__(16) double ring[(RING + 1) * (B + 1) * BSP_EIG_THREADS];
    __shared__ __align__(8) uint64_t bars[2];
    if (optional && g.counters[BSP_C_REFINED]) return;
    const int p = blockIdx.y, ls = blockIdx.x * blockDim.x + threadIdx.x;
    int e;
    bool active;
    if (!bsp_refine_map(g, p, iter, optional && g.rlist != nullptr, e, active)) return;
    bsp_stage_bars_init(bars);
    if (!__syncthreads_or(active)) return;
    constexpr int FS = 2 * B + 2;
    BspRowsStaged<B, RING> src{sm, bars, g.fbH + (size_t)p * g.nrows * FS, g.fbS + (size_t)g.inst[p] * g.nrows * FS};
    src.rq = ring + threadIdx.x;
    bsp_factor_forward_rhs<B, RHS>(g, p, e, ls, active, src);
}

template <int B>
__global__ void __launch_bounds__(BSP_EIG_THREADS, bsp_minb(BSP_MINB_BACK, B)) bsp_back_kernel(BspEigChunk g, int iter, int corr_now, int corr_next, int optional)
{
    __shared__ __align__(128) double sm[BspTile<B>::SMEM_DOUBLES];
    __shared__ __align__(8) uint64_t bars[2];
    if (optional && g.counters[BSP_C_REFINED]) return;
    const int p = blockIdx.y, ls = blockIdx.x * blockDim.x + threadIdx.x;
    int e;
    bool active;
    if (!bsp_refine_map(g, p, iter, optional && g.rlist != nullptr, e, active)) return;
    bsp_stage_bars_init(bars);
    if (!__syncthreads_or(active)) return;
    constexpr int FS = 2 * B + 2;
    BspRowsStaged<B> src{sm, bars, g.fbH + (size_t)p * g.nrows * FS, g.fbS + (size_t)g.inst[p] * g.nrows * FS};
    bsp_back_substitute_rows<B>(g, p, e, ls, corr_now, corr_next, active, src);
}

/* ---- check-pointed solves (full-width iterations 0 and 1) ---------------------------------------------------- */
template <int B, int RHS>
__global__ void __launch_bounds__(BSP_EIG_THREADS, bsp_minb(BSP_MINB_FACTOR, B)) bsp_factor_ckpt_kernel(BspEigChunk g)
{
    __shared__ __align__(128) double sm[BspTile<B>::SMEM_DOUBLES];
    constexpr int RING = bsp_rhs_ring(B);
    __shared__ __align__(16) double ring[(RING + 1) * (B + 1) * BSP_EIG_THREADS];
    __shared__ __align__(8) uint64_t bars[2];
    const int p = blockIdx.y, e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = bsp_refine_active(g, p, e);
    bsp_stage_bars_init(bars);
    if (!__syncthreads_or(active)) return;
    constexpr int FS = 2 * B + 2;
    BspRowsStaged<B, RING> src{sm, bars, g.fbH + (size_t)p * g.nrows * FS, g.fbS + (size_t)g.inst[p] * g.nrows * FS};
    src.rq = ring + threadIdx.x;
    bsp_factor_forward_rhs<B, RHS, true>(g, p, e, e, active, src);
}

/* scratch of the check-pointed back sweep: one column of shared memory per thread (slot i at base[i * blockDim.x]:
 * conflict-free), also the landing zone of the asynchronous copy of the next check-point */
struct BspScratchShared {
    double *base;
    int nt;
    __device__ __forceinline__ double &slot(int i) { BSP_ASSERT(i >= 0); return base[(size_t)i * nt]; }
    __device__ __forceinline__ void prefetch(int i, const double *gp)
    {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(bsp_smem_u32(base + (size_t)i * nt)), "l"(gp) : "memory");
    }
    __device__ __forceinline__ void prefetch_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
    __device__ __forceinline__ void prefetch_wait() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
    __device__ __forceinline__ double fetched(int i, const double *) { return base[(size_t)i * nt]; }
};

#ifndef BSP_CKB_THREADS
#define BSP_CKB_THREADS 128
#endif
#ifndef BSP_CKB_MINB
#define BSP_CKB_MINB 2
#endif
template <int B>
constexpr size_t bsp_back_ckpt_smem(int threads)
{
    return (size_t)(BspTile<B, BSP_CK_GROUPS(B)>::SMEM_DOUBLES + BSP_CK_STEPS(B) * (B + 1) * threads) * sizeof(double);
}
template <int B>
__global__ void __launch_bounds__(BSP_CKB_THREADS, BSP_CKB_MINB) bsp_back_ckpt_kernel(BspEigChunk g, int iter, int corr_next)
{
    extern __shared__ __align__(128) double dsm[];
    __shared__ __align__(8) uint64_t bars[2];
    using T = BspTile<B, BSP_CK_GROUPS(B)>;
    const int p = blockIdx.y, e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = bsp_refine_active(g, p, e);
    bsp_stage_bars_init(bars);
    if (!__syncthreads_or(active)) return;
    constexpr int FS = 2 * B + 2;
    BspRowsStaged<B, 0, BSP_CK_GROUPS(B)> src{dsm, bars, g.fbH + (size_t)p * g.nrows * FS, g.fbS + (size_t)g.inst[p] * g.nrows * FS};
    BspScratchShared scr{dsm + T::SMEM_DOUBLES + threadIdx.x, (int)blockDim.x};
    bsp_back_ckpt_rows<B>(g, p, e, e, iter, corr_next, active, src, scr);
}

__global__ void bsp_check_kernel(BspEigChunk g, int iter, int select)
{
    if (g.counters[BSP_C_REFINED]) return;
    const int p = blockIdx.y, e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool keep = bsp_check_keep(g, p, e, select);
    /* a warp appends its eigen indices as one ascending run (one atomic per warp): the compacted passes that
     * follow then read X columns of neighbouring lanes from the same 32-byte sectors -- the selected pairs are
     * the ones with close neighbours and come in runs of consecutive indices */
    const unsigned mask = __ballot_sync(0xffffffffu, keep);
    if (mask) {
        const int lane = threadIdx.x & 31, cnt = __popc(mask);
        int base = 0;
        if (lane == 0) {
            atomicAdd(g.counters + BSP_C_UNCONV, cnt);
            if (g.rlist) base = atomicAdd(g.rcount + (iter & 1) * g.npencil + p, cnt);
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        if (keep && g.rlist) {
            const int slot = base + __popc(mask & ((1u << lane) - 1u));
            BSP_ASSERT(slot >= 0 && slot < g.n);
            g.rlist[((size_t)(iter & 1) * g.npencil + p) * g.ldw + slot] = e;
        }
    }
    if (bsp_last_block(g.counters + BSP_C_ARRIVE)) bsp_check_ctl(g, iter);
}

/* copy the chunk's control block into the run report and clear it for the next chunk of this stream */
__global__ void bsp_report_kernel(BspEigChunk g, int *report)
{
    if (threadIdx.x < BSP_C_WORDS) {
        report[threadIdx.x] = g.counters[threadIdx.x];
        g.counters[threadIdx.x] = 0;
    }
}

__global__ void bsp_copy_ints_kernel(int *dst, const int *src, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}

__global__ void bsp_finalize_kernel(BspEigChunk g, double *E, double *fac, int *bad, double res_tol)
{
    bsp_finalize_eigen(g, blockIdx.y, blockIdx.x * blockDim.x + threadIdx.x, E, fac, bad, res_tol);
}

/* Literal CHKPHS (matrices.f90:398-449; option "sign_rule" = 1): after the default sign convention, evaluate
 *   fr(i) = sum_j c(j) bsp(j - (left - nbc1)),  j = left-nbc1+1 .. MIN(left-nbc1+k, nfun),  r = ra + i (0.1 - ra)/3, i = 1..3
 * with the reference's own index mapping (jfun = j - (left - nbc1): one function higher than WRITE_WF's
 * j = left - k + jfun when nbc1 = k-1, SURVEY.md 8(f) row f-1 -- reproduced, not fixed) and flip the vector when all
 * three values are negative.  nbc1 = multiplicity of the first knot (rt(1:nbc1) = ra, grid.f90:16-18). */
template <int K>
__global__ void bsp_chkphs_kernel(BspEigChunk g, const double *__restrict__ rt_all, int nkp, double *fac)
{
    const int p = blockIdx.y, e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= g.nvec[p] || e >= g.n) return;
    const double *rt = rt_all + (size_t)g.inst[p] * nkp;
    const size_t id = (size_t)p * g.ldw + e;
    const double *Xp = g.X + (size_t)p * g.xrows * g.ldw + e;
    const double ra = rt[0];
    int nbc1 = 1;
    while (nbc1 < nkp && rt[nbc1] == ra) ++nbc1;
    const double dr = (0.1 - ra) / 3.0;
    int neg = 0;
    for (int i = 1; i <= 3; ++i) {
        const double r = ra + (double)i * dr;
        int left = 1;                                   /* interv: largest left with rt(left) <= r < rt(left+1) */
        while (left < nkp && rt[left] <= r) ++left;     /* rt[left] is rt(left+1) */
        if (left >= nkp || !(rt[left] > rt[left - 1])) { left = 1; }
        double bsp[K], dbsp[K];
        bsp_deboor<K>(rt, nkp, g.n, left, r, bsp, dbsp);
        const int jmin = left - nbc1 + 1, jmax = min(jmin + K - 1, g.n);
        double sumf = 0.0;
        for (int j = jmin; j <= jmax; ++j) {
            const int jfun = j - (left - nbc1);
            if (j >= 1) sumf += fac[id] * Xp[(size_t)(j - 1) * g.ldw] * bsp[jfun - 1];
        }
        neg += (sumf < 0.0);
    }
    if (neg == 3) fac[id] = -fac[id];
}

/* C[p] (n x nvec_p, column-major, column e = eigenvector e) = fac[e] * X[p][row][e]
 * shared-memory transpose of BSP_TR_TILES tiles of 32x32 per block (all loads of a block in flight before its
 * barrier); coff[p] = offset of pencil p's block in C. */
#define BSP_TR_TILES 4
__global__ void bsp_transpose_kernel(BspEigChunk g, const double *fac, double *C, const long long *coff)
{
    __shared__ double tile[BSP_TR_TILES][32][33];
    const int p = blockIdx.z;
    const int nv = g.nvec[p];
    const int e0 = blockIdx.x * 32, r00 = blockIdx.y * 32 * BSP_TR_TILES;
    if (e0 >= nv) return;
    const double *X = g.X + (size_t)p * g.xrows * g.ldw;
    const int e_in = e0 + threadIdx.x;
    const double f = e_in < nv ? fac[(size_t)p * g.ldw + e_in] : 0.0;
#pragma unroll
    for (int t = 0; t < BSP_TR_TILES; ++t) {
#pragma unroll
        for (int rr = threadIdx.y; rr < 32; rr += 8) {
            const int r = r00 + t * 32 + rr;
            double v = 0.0;
            if (r < g.n && e_in < nv) v = X[(size_t)r * g.ldw + e_in] * f;
            tile[t][rr][threadIdx.x] = v;
        }
    }
    __syncthreads();
    double *Cp = C + coff[p];
#pragma unroll
    for (int t = 0; t < BSP_TR_TILES; ++t) {
#pragma unroll
        for (int ee = threadIdx.y; ee < 32; ee += 8) {
            const int e = e0 + ee, r = r00 + t * 32 + threadIdx.x;
            if (e < nv && r < g.n) Cp[(size_t)e * g.n + r] = tile[t][threadIdx.x][ee];
        }
    }
}

/* fbH[p] = fbH0[inst] + cl[p] * fbQ[inst]   (Hij = Tij + Uij(:,:,l) + Vij, matrices.f90:244) */
__global__ void bsp_combine_kernel(double *fbH, const double *fbH0, const double *fbQ, const int *inst,
                                   const double *cl, size_t per_mat)
{
    const int p = blockIdx.y;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= per_mat) return;
    const size_t src = (size_t)inst[p] * per_mat + i;
    fbH[(size_t)p * per_mat + i] = bsp_combine_entry(cl[p], fbQ[src], fbH0[src]);
}

/* ---- driven equation (H - z S) x = b (bsp_shifted_*_rows): one thread per system slot, blockIdx.z = right-hand
 * side; a block's slots all belong to pencil blk_pen[blockIdx.x], whose band rows the block stages once ---------- */
template <int B, class T>
__global__ void __launch_bounds__(BSP_EIG_THREADS) bsp_shifted_factor_kernel(BspShiftChunk<T> c)
{
    __shared__ __align__(128) double sm[BspTile<B>::SMEM_DOUBLES];
    __shared__ __align__(8) uint64_t bars[2];
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = slot < c.nslot && c.sys[slot] >= 0;
    bsp_stage_bars_init(bars);
    if (!__syncthreads_or(active)) return;
    constexpr int FS = 2 * B + 2;
    BspRowsStaged<B> src{sm, bars, c.fbH + (size_t)c.blk_pen[blockIdx.x] * c.nrows * FS,
                         c.fbS + (size_t)c.blk_inst[blockIdx.x] * c.nrows * FS};
    bsp_shifted_factor_rows<B, T>(c, slot, active, src);
}

template <int B, class T>
__global__ void __launch_bounds__(BSP_EIG_THREADS) bsp_shifted_forward_kernel(BspShiftChunk<T> c, int step)
{
    __shared__ __align__(128) double sm[BspTile<B>::SMEM_DOUBLES];
    __shared__ __align__(8) uint64_t bars[2];
    const int slot = blockIdx.x * blockDim.x + threadIdx.x, col = blockIdx.z;
    const bool active = bsp_shift_active(c, slot, col);   /* finished systems return */
    bsp_stage_bars_init(bars);
    if (!__syncthreads_or(active)) return;
    constexpr int FS = 2 * B + 2;
    BspRowsStaged<B> src{sm, bars, c.fbH + (size_t)c.blk_pen[blockIdx.x] * c.nrows * FS,
                         c.fbS + (size_t)c.blk_inst[blockIdx.x] * c.nrows * FS};
    bsp_shifted_forward_rows<B, T>(c, slot, col, step, active, src);
}

template <int B, class T>
__global__ void __launch_bounds__(BSP_EIG_THREADS) bsp_shifted_back_kernel(BspShiftChunk<T> c, int step)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x, col = blockIdx.z;
    if (bsp_shift_active(c, slot, col)) bsp_shifted_back_rows<B, T>(c, slot, col, step);
}

template <class T>
__global__ void bsp_shifted_report_kernel(BspShiftChunk<T> c, int *info_out, double *berr_out)
{
    bsp_shifted_report(c, blockIdx.x * blockDim.x + threadIdx.x, info_out, berr_out);
}

/* caller layout (system s: n x nrhs column-major at off[slot]) <-> slot-fastest workspace [col][row][slot], through
 * 32 x 32 shared-memory tiles tile[slot][row]: the caller side is read or written along rows, the workspace side
 * along slots, so both sides move whole lines.  The scatter writes only the systems whose solution is defined
 * (info 0 or n + 1). */
template <class T, bool GATHER>
__global__ void bsp_shifted_layout_kernel(BspShiftChunk<T> c, const long long *off, T *caller, T *ws, const int *info)
{
    __shared__ T tile[32][33];
    const int r0 = blockIdx.x * 32, s0 = blockIdx.y * 32, col = blockIdx.z, n = c.n;
    const size_t ld = c.nslot;
    /* caller side: lane = row, one system per step */
    auto caller_ok = [&](int slot) {
        if (slot >= c.nslot || c.sys[slot] < 0) return false;
        if (GATHER) return true;
        const int i = info[slot];
        return i == 0 || i == n + 1;
    };
    if (GATHER) {
        for (int ss = threadIdx.y; ss < 32; ss += blockDim.y) {
            const int slot = s0 + ss, row = r0 + threadIdx.x;
            if (row < n && caller_ok(slot)) tile[ss][threadIdx.x] = caller[off[slot] + (long long)col * n + row];
        }
    } else {   /* workspace side: lane = slot, one row per step */
        for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
            const int row = r0 + rr, slot = s0 + threadIdx.x;
            if (row < n && slot < c.nslot) tile[threadIdx.x][rr] = ws[((size_t)col * n + row) * ld + slot];
        }
    }
    __syncthreads();
    if (GATHER) {
        for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
            const int row = r0 + rr, slot = s0 + threadIdx.x;
            if (row < n && slot < c.nslot && c.sys[slot] >= 0) ws[((size_t)col * n + row) * ld + slot] = tile[threadIdx.x][rr];
        }
    } else {
        for (int ss = threadIdx.y; ss < 32; ss += blockDim.y) {
            const int slot = s0 + ss, row = r0 + threadIdx.x;
            if (row < n && caller_ok(slot)) caller[off[slot] + (long long)col * n + row] = tile[ss][threadIdx.x];
        }
    }
}

/* Where pencil p's bands sit in the staging buffer of bspatom_band_upload: A and B packed column-major with leading
 * dimensions ka+1 and kb+1, in the caller's LAPACK layout (upper: AB(k+1+i-j, j), lower: AB(1+i-j, j), 1-based). */
struct BspBandSrc {
    long long a_off, b_off;   /* offsets in doubles */
    int ka, kb, upper;
};

#define BSP_INGEST_TR 32        /* full-band rows per block */
#define BSP_INGEST_THREADS 128

/* A(i, j) of a symmetric band read from its stored triangle (0-based, |i - j| <= k) */
__device__ __forceinline__ double bsp_band_at(const double *__restrict__ M, int k, int upper, int i, int j)
{
    const int lo = min(i, j), hi = max(i, j);
    return upper ? M[(size_t)hi * (k + 1) + k + lo - hi] : M[(size_t)lo * (k + 1) + hi - lo];
}

/* caller-supplied bands -> full-band rows fb[i*FS + c] = M(i, i-B+c) of S (from B) and H0 (from A), Q = 0, padded
 * exactly as bsp_assemble_kernel pads: rows n..nrows-1 hold diag(H0) = 1 and 0 elsewhere, column 2B+1 is 0.
 * grid = ceil(nrows / BSP_INGEST_TR) * npencil blocks along x (row tiles of pencil 0, then of pencil 1, ...: a batch
 * of many small pencils is not limited by the 65535 blocks of grid.y); pencil p becomes instance p of the group. */
__global__ void __launch_bounds__(BSP_INGEST_THREADS) bsp_band_ingest_kernel(const double *__restrict__ stage,
                                                                             const BspBandSrc *__restrict__ src, int n, int B,
                                                                             int nrows, double *fbS, double *fbH0, double *fbQ)
{
    const int ntiles = (nrows + BSP_INGEST_TR - 1) / BSP_INGEST_TR;
    const int p = blockIdx.x / ntiles, FS = 2 * B + 2;
    const BspBandSrc s = src[p];
    const int i0 = (blockIdx.x % ntiles) * BSP_INGEST_TR;
    const int nout = min(BSP_INGEST_TR, nrows - i0) * FS;
    const size_t base = ((size_t)p * nrows + i0) * FS;
    for (int o = threadIdx.x; o < nout; o += BSP_INGEST_THREADS) {
        const int i = i0 + o / FS, c = o % FS, j = i - B + c;
        double a = 0.0, b = 0.0;
        if (i < n && c <= 2 * B && j >= 0 && j < n) {
            const int d = abs(i - j);
            if (d <= s.ka) a = bsp_band_at(stage + s.a_off, s.ka, s.upper, i, j);
            if (d <= s.kb) b = bsp_band_at(stage + s.b_off, s.kb, s.upper, i, j);
        } else if (i >= n && c == B) {
            a = 1.0;   /* padding row: decoupled, positive pivot */
        }
        fbS[base + o] = b;
        fbH0[base + o] = a;
        fbQ[base + o] = 0.0;
    }
}

/* S positive definite?  one thread per instance walks the LDL^T pivots of S with the register-window
 * recurrence of the Sturm count (H := S, sigma = 0).  pd_info as below. */
template <int B>
__global__ void bsp_pdcheck_fast_kernel(const double *fbS, int n, int npad, int nrows, int ninst, int *pd_info)
{
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= ninst) return;
    const double *S = fbS + (size_t)inst * nrows * (2 * B + 2);
    int first = -1;
    bsp_sturm_count<B>(S, S, npad, 0.0, 1e-300, &first);
    pd_info[inst] = (first >= 0 && first < n) ? first + 1 : 0;
}

/* S positive definite?  one thread per instance: banded Cholesky pivots.
 * pd_info[inst] = 0 or the 1-based index of the first non-positive pivot
 * (LAPACK dpotrf numbering; DSYGV reports N + that, matrices.f90:250). */
__global__ void bsp_pdcheck_kernel(const double *fbS, int n, int nrows, int B, int ninst, int *pd_info,
                                   double *Lout /* NULL or [ninst][n][B+1]: L(j+i,j) */)
{
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= ninst) return;
    const int FS = 2 * B + 2;
    const double *S = fbS + (size_t)inst * nrows * FS;
    /* window of the last B columns of L (scaled), generic B <= 15 */
    double w[16][16];
    for (int a = 0; a < 16; ++a) for (int b = 0; b < 16; ++b) w[a][b] = 0.0;
    int info = 0;
    for (int j = 0; j < n && !info; ++j) {
        /* column j of the Schur complement: a(j+i,j) - sum_{c<j} l(j+i,c) l(j,c) d(c) */
        double col[16];
        for (int i = 0; i <= B; ++i) {
            double v = (j + i < n) ? S[(size_t)(j + i) * FS + (B - i)] : 0.0;
            /* previous columns c = j-1 .. j-B are kept in w[(c)%16][*] as l(c+t,c)*sqrt(d) */
            for (int t = 1; t <= B - i; ++t) {
                const int c = j - t;
                if (c < 0) break;
                v -= w[c & 15][t + i] * w[c & 15][t];
            }
            col[i] = v;
        }
        if (!(col[0] > 0.0)) { info = j + 1; break; }
        const double d = sqrt(col[0]);
        w[j & 15][0] = d;
        for (int i = 1; i <= B; ++i) w[j & 15][i] = col[i] / d;
        for (int i = B + 1; i < 16; ++i) w[j & 15][i] = 0.0;
        if (Lout)
            for (int i = 0; i <= B; ++i) Lout[((size_t)inst * n + j) * (B + 1) + i] = w[j & 15][i];
    }
    pd_info[inst] = info;
}

#endif
