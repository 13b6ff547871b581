/*
 * bsp_driver.h -- stage schedule of the banded eigensolver for one chunk of pencils, written against
 * an executor so that the CUDA enqueuer (bsp_api.cu) and the CPU replay used by tests/emul share it.
 *
 * The schedule is STATIC: everything is enqueued up front and nothing is read back by the host while
 * a chunk runs.  Data-dependent control lives in the chunk's device-side control block (BSP_C_* in
 * bsp_core.h): once the bracketing is finished the remaining round kernels see BSP_C_BRACKETED and
 * return at once, and the optional extra refinement iterations see BSP_C_REFINED.  The host inspects the
 * per-chunk report after the whole batch and re-runs a chunk with larger limits only if it had to.
 *
 * Exec must provide:
 *   void bounds();                            // bracket [lo0,hi0] per pencil
 *   void round(int r, int max_rounds);        // one bracketing round + its bookkeeping
 *   void select();                            // device-side state selection (no-op unless the batch asks for it)
 *   void prepare();                           // hand brackets to the refinement
 *   void factor(int iter, int optional);      // F pass (optional: compacted to the eigenpairs the last check listed,
 *                                             //         skipped once everything converged)
 *   void back(int iter, int corr_now, int corr_next, int optional);
 *   void check(int iter, int select);         // convergence marks, compaction list of what is left, bookkeeping
 */
#ifndef BSP_DRIVER_H
#define BSP_DRIVER_H

struct BspSchedule {
    int rounds;     /* bracketing rounds enqueued (the flag makes surplus ones free)       */
    int min_iters;  /* solves every eigenpair gets (2: default, a third only where the residual / gap test asks
                       for it; 3: the round-1 schedule, everybody gets the correction pass) */
    int max_iters;  /* iterations enqueued; those beyond min_iters only touch stragglers   */
};

struct BspRunStats {
    int rounds;
    int iters;
    int brackets_open;    /* brackets handed over open (each isolating its eigenvalue)      */
    int brackets_crowded; /* ... of which not isolating: the chunk must be re-run           */
    int unconverged;      /* eigenpairs above conv_tol after the last iteration             */
};

template <class Exec>
inline void bsp_enqueue_chunk(Exec &ex, const BspSchedule &sch)
{
    ex.bounds();
    for (int r = 0; r < sch.rounds; ++r) ex.round(r, sch.rounds);
    ex.select();
    ex.prepare();
    /* iteration t: plain for t < 2 (inverse iteration at the bracket midpoint, then at the Rayleigh quotient),
     * residual-correction form afterwards.  Default (min_iters = 2): the back sweep of the second solve carries the
     * sums from which the residual norm against its NEW Rayleigh quotient follows (bsp_back_finish), and the check
     * keeps in the iteration what misses conv_tol or has ||r||_2 / gap > vec_tol (bsp_check_converged): 10-17 % of
     * the eigenpairs of the N = 1000 pencils.  The passes from there on are COMPACTED to that list
     * (bsp_listed_index), so the correction pass that brings the S-orthogonality of neighbouring vectors from ~1e-8
     * to ~1e-12 costs what its eigenpairs cost.  No pass writes a right-hand side: every factor pass forms its own
     * from the vector in X (S x, or r = (H - rho S) x) while it walks the band rows.  A back sweep followed by the
     * check leaves the quotient and shift a correction after it needs: r against its new quotient, the shift delta
     * away from that (bsp_back_finish). */
    const bool select = sch.min_iters <= 2;
    for (int t = 0; t < sch.max_iters; ++t) {
        const int optional = (t >= sch.min_iters);
        const bool check_follows = (t + 1 == sch.min_iters && select);
        const bool lean = select && optional;
        ex.factor(t, optional);
        ex.back(t, t >= 2, (check_follows || lean) ? -1 : (t + 1 >= 2), optional);
        /* check: 1 = residual / gap test that selects the correction pass; 2 = the looser one after a correction (not
         * after the last enqueued pass: what is still listed there counts as unconverged and the chunk is redone) */
        if (t + 1 >= sch.min_iters) ex.check(t, check_follows ? 1 : ((select && t + 1 < sch.max_iters) ? 2 : 0));
    }
}

#endif
