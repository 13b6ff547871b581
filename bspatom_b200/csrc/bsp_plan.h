/*
 * bsp_plan.h -- how the batch runner cuts a group of pencils into chunks.  Host code without CUDA, so that the
 * tests compile it with g++ (tests/emul/emul_plan.cpp).
 *
 * Chunk streams: `workers` streams (each with its own workspace) run chunks concurrently and back-fill each other's
 * partial waves and latency-bound kernels (late bracketing rounds); blocks run a whole sweep (~1 ms), so stream
 * priorities cannot order the chunks -- the chunk sizes do.  Resident batches use `workers` equal chunks.  When
 * results stream to the host the D2H (PCIe, ~53 GB/s, 57 ms per 408 solves of N = 1000) is the longer leg: the
 * batch is cut into `stream_chunks` chunks whose sizes SHRINK (weights n+2, n+1, ..., 3): the first copies start as
 * early as with equal chunks and keep the link busy, and the last chunks -- whose copies nothing can hide -- are
 * small.  (Measured, single handle, 408 solves: shrinking 79.6 ms, equal 84 ms, growing 95 ms per batch: a chunk
 * below ~40 pencils takes ~17 ms whatever its size, its kernel chain being latency-bound, so small chunks must not
 * come first.)
 */
#ifndef BSP_PLAN_H
#define BSP_PLAN_H

#include <algorithm>
#include <utility>
#include <vector>

constexpr int BSP_PLAN_THREADS = 128;   /* threads of an eigen-stage block (BSP_EIG_THREADS) */

struct BspPlanInput {
    int npencil = 0;
    int n = 0;                 /* order of the group's pencils */
    int budget_pencils = 1;    /* pencils whose workspaces fit the memory budget */
    int workers = 2, stream_workers = 2, stream_chunks = 6, chunk = 0;   /* the options of these names */
    bool streaming = false;    /* results stream to the host chunk by chunk */
    std::vector<std::pair<int, int>> sel;   /* per pencil (sel.mode, sel.group); empty without device-side selection */
};

struct BspChunkPlan {
    std::vector<int> bounds;   /* chunk i holds pencils [bounds[i], bounds[i+1]) */
    int streams = 0;           /* chunk streams */
    int largest = 0;           /* pencils of the largest chunk: the workspace of each stream is sized for it */
    bool group_too_large = false;   /* a chunk that keeps its selection groups whole exceeds the workspace */
    int nchunks() const { return (int)bounds.size() - 1; }
};

inline BspChunkPlan bsp_plan_chunks(const BspPlanInput &in)
{
    BspChunkPlan out;
    const int npencil = in.npencil;
    const bool any_sel = !in.sel.empty();
    const int blocks_per_pencil = (in.n + BSP_PLAN_THREADS - 1) / BSP_PLAN_THREADS;
    const int fill_pencils = std::max(1, (148 * 4 + blocks_per_pencil - 1) / blocks_per_pencil); /* one full wave */
    int workers = std::max(1, std::min(in.streaming ? in.stream_workers : in.workers, npencil / fill_pencils));
    const int cap = std::max(1, std::min(in.budget_pencils / workers, 1024));   /* workspace per stream */
    std::vector<int> &bounds = out.bounds;
    bounds.assign(1, 0);
    if (in.chunk > 0) {
        const int chunk = std::min(in.chunk, npencil), nchunks = (npencil + chunk - 1) / chunk;
        for (int i = 1; i <= nchunks; ++i) bounds.push_back(std::min(i * chunk, npencil));
    } else {
        int want = workers;
        /* with a device-side selection the copies are small and every chunk carries the latency-bound tail of the
         * rounds that close the values-only brackets: no extra chunks for streaming */
        if (in.streaming && !any_sel) want = std::max(want, std::min(in.stream_chunks, std::max(1, (2 * npencil) / fill_pencils)));
        int nchunks = std::min(std::max(want, (npencil + cap - 1) / cap), npencil);
        const bool shrink = in.streaming && nchunks >= 4 && (long long)cap * (nchunks + 5) >= 2LL * npencil;
        if (shrink) {
            /* weights n+2, n+1, ..., 3: the largest chunk is < 2x the mean and must fit the workspace */
            double tot = 0.0, accw = 0.0;
            for (int i = 0; i < nchunks; ++i) tot += (double)(nchunks + 2 - i);
            for (int i = 0; i < nchunks; ++i) {
                accw += (double)(nchunks + 2 - i);
                int bnd = (i + 1 == nchunks) ? npencil : (int)(npencil * accw / tot + 0.5);
                bnd = std::max(bnd, bounds.back() + 1);
                bnd = std::min(bnd, npencil - (nchunks - 1 - i));
                bounds.push_back(bnd);
            }
        } else {
            const int eq = (npencil + nchunks - 1) / nchunks;
            nchunks = (npencil + eq - 1) / eq;
            for (int i = 1; i <= nchunks; ++i) bounds.push_back(std::min(i * eq, npencil));
        }
    }
    if (any_sel) {
        /* the running maximum of a selection group is sequential over its pencils: a group stays in one chunk */
        const auto &sel = in.sel;
        for (size_t b = 1; b + 1 < bounds.size(); ++b) {
            int x = std::max(bounds[b], bounds[b - 1]);
            while (x < npencil && x > 0 && sel[x].first && sel[x].second >= 0 && sel[x - 1].first &&
                   sel[x - 1].second == sel[x].second) ++x;
            bounds[b] = x;
        }
        std::vector<int> nb(1, 0);
        for (size_t b = 1; b < bounds.size(); ++b) if (bounds[b] > nb.back()) nb.push_back(bounds[b]);
        bounds = nb;
    }
    for (int i = 0; i < out.nchunks(); ++i) out.largest = std::max(out.largest, bounds[i + 1] - bounds[i]);
    out.group_too_large = any_sel && out.largest > cap && in.chunk <= 0;
    out.streams = std::min(workers, out.nchunks());
    return out;
}

#endif
