/* C entry over bsp_plan_chunks (bspatom_b200/csrc/bsp_plan.h) for tests/test_chunk_plan.py.
 * sel_mode / sel_group: per pencil, or NULL for a group without device-side selection.
 * Returns the number of chunks (bounds_out receives nchunks + 1 entries), or -1 when a selection group does not fit
 * one chunk. */
#include "../../bspatom_b200/csrc/bsp_plan.h"

extern "C" int emul_plan(int npencil, int n, int budget_pencils, int workers, int stream_workers, int stream_chunks,
                         int chunk, int streaming, const int *sel_mode, const int *sel_group, int *bounds_out,
                         int *streams_out, int *largest_out)
{
    BspPlanInput in;
    in.npencil = npencil; in.n = n; in.budget_pencils = budget_pencils;
    in.workers = workers; in.stream_workers = stream_workers; in.stream_chunks = stream_chunks; in.chunk = chunk;
    in.streaming = streaming != 0;
    bool any = false;
    for (int p = 0; sel_mode && p < npencil; ++p) any = any || sel_mode[p] != 0;
    for (int p = 0; any && p < npencil; ++p) in.sel.push_back({sel_mode[p], sel_group[p]});
    const BspChunkPlan plan = bsp_plan_chunks(in);
    if (plan.group_too_large) return -1;
    for (int i = 0; i <= plan.nchunks(); ++i) bounds_out[i] = plan.bounds[i];
    *streams_out = plan.streams;
    *largest_out = plan.largest;
    return plan.nchunks();
}
