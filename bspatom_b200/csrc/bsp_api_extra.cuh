/*
 * bsp_api_extra.cuh -- included at the end of bsp_api.cu: the LAPACK-shaped
 * entry (Level 0), the dense dipole contraction and wavefunction synthesis.
 */
#ifndef BSP_API_EXTRA_CUH
#define BSP_API_EXTRA_CUH

#include "bsp_assembly_z.cuh"

namespace {

/* psi(ip, iv) = sum_j C(j,iv) B_j(r_ip)      WRITE_WF, Bsp_Atom.f90:118-146 */
template <int K>
__global__ void bsp_wavefunction_kernel(int nfun, int nkp, const double *__restrict__ rt, double ra, double rb,
                                        int npts, int nvec, const double *__restrict__ C,
                                        double *__restrict__ r_out, double *__restrict__ psi)
{
    const int ip = blockIdx.x * blockDim.x + threadIdx.x;
    if (ip > npts) return;
    const double dr = (rb - ra) / (double)npts;            /* :120 */
    const double r = ra + (double)ip * dr;                 /* :127 */
    if (blockIdx.y == 0) r_out[ip] = r;
    /* interv (interv.f90:86-116) for non-decreasing knots: largest left with
     * rt(left) <= r < rt(left+1); r == rt(nkp) walks down to the last interval
     * of positive width; outside the knots the reference returns left = 1 */
    int left;
    const double tlast = rt[nkp - 1];
    if (r > tlast || r < rt[0]) {
        left = 1;
    } else if (r == tlast) {
        left = nkp;
        while (left > 1 && !(rt[left - 1] < tlast)) --left;
    } else {
        int a = 1, b = nkp; /* rt(a) <= r < rt(b) */
        while (b - a > 1) {
            const int m = (a + b) >> 1;
            if (rt[m - 1] <= r) a = m; else b = m;
        }
        left = a;
    }
    double bsp[K], dbsp[K];
    bool ok = rt[min(left, nkp - 1)] > rt[left - 1];       /* bsplvb.f90:30 */
    if (ok) bsp_deboor<K>(rt, nkp, nfun, left, r, bsp, dbsp);
    for (int iv = blockIdx.y; iv < nvec; iv += gridDim.y) {
        double s = 0.0;
        if (ok) {
#pragma unroll
            for (int a = 0; a < K; ++a) {
                const int j = left - K + 1 + a;            /* :133-141 */
                if (j >= 1 && j <= nfun) s += C[(size_t)iv * nfun + j - 1] * bsp[a];
            }
        }
        psi[(size_t)iv * (npts + 1) + ip] = s;
    }
}

template <int K>
void launch_wavefunction(bspatom_handle h, int nfun, int nkp, const double *rt, double ra, double rb, int npts,
                         int nvec, const double *C, double *r_out, double *psi)
{
    dim3 grid((npts + 1 + 127) / 128, std::min(nvec, 64));
    bsp_wavefunction_kernel<K><<<grid, 128, 0, h->st>>>(nfun, nkp, rt, ra, rb, npts, nvec, C, r_out, psi);
    h->launches++;
}

/* ---- device-side verification of a resident batch (bspatom_batch_verify) --------------------------------- *
 * Y(:, v) = S c_v and the scaled residual max_i |(H_l c_v)_i - E_v (S c_v)_i| / max(1, |E_v|) of every eigenpair
 * of the pencils [p0, p0 + np) of a group, from the assembled full-band rows (H_l = H0 + c_l Q, matrices.f90:244).
 * The maximum is taken with an integer atomicMax on the bits of the (non-negative) double. */
__device__ __forceinline__ void bsp_atomic_max_pos(double *addr, double v)
{
    if (v == v) atomicMax((unsigned long long *)addr, (unsigned long long)__double_as_longlong(v));
    else atomicMax((unsigned long long *)addr, (unsigned long long)__double_as_longlong(INFINITY));
}

__global__ void bsp_verify_matvec_kernel(int n, int B, int nrows, const double *__restrict__ fbS, const double *__restrict__ fbH0,
                                         const double *__restrict__ fbQ, const int *__restrict__ inst,
                                         const double *__restrict__ cl, const int *__restrict__ nvec,
                                         const long long *__restrict__ coff, const double *__restrict__ Cg,
                                         const double *__restrict__ E, double *__restrict__ Y, long long ystride,
                                         int p0, double *out)
{
    const int p = p0 + blockIdx.z, v = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvec[p]) return;
    const int FS = 2 * B + 2;
    const size_t mo = (size_t)inst[p] * nrows * FS;
    const double c_l = cl[p], ev = E[(size_t)p * n + v];
    const double *c = Cg + coff[p] + (size_t)v * n;
    double r = 0.0;
    if (i < n) {
        double s = 0.0, h = 0.0;
        const double *rs = fbS + mo + (size_t)i * FS, *rh = fbH0 + mo + (size_t)i * FS, *rq = fbQ + mo + (size_t)i * FS;
        for (int d = 0; d <= 2 * B; ++d) {
            const int j = i - B + d;
            if (j < 0 || j >= n) continue;
            const double x = c[j];
            s = fma(rs[d], x, s);
            h = fma(fma(c_l, rq[d], rh[d]), x, h);
        }
        Y[(size_t)blockIdx.z * ystride + (size_t)v * n + i] = s;
        r = fabs(h - ev * s) / fmax(1.0, fabs(ev));
    }
    __shared__ double red[128];
    red[threadIdx.x] = r;
    __syncthreads();
    for (int w = 64; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) red[threadIdx.x] = (red[threadIdx.x] >= red[threadIdx.x + w] || red[threadIdx.x] != red[threadIdx.x]) ? red[threadIdx.x] : red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) bsp_atomic_max_pos(out + 0, red[0]);
}

/* max |G - I| over the nv x nv Gram matrices G = C^T S C of the chunk; and the smallest E(v+1) - E(v) */
__global__ void bsp_verify_gram_kernel(int n, const int *__restrict__ nvec, const double *__restrict__ G, long long gstride,
                                       int ldg, const double *__restrict__ E, int p0, double *out)
{
    const int p = p0 + blockIdx.z, nv = nvec[p];
    const int j = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nv) return;
    double d = 0.0;
    if (i < nv) d = fabs(G[(size_t)blockIdx.z * gstride + (size_t)j * ldg + i] - (i == j ? 1.0 : 0.0));
    __shared__ double red[128];
    red[threadIdx.x] = d;
    __syncthreads();
    for (int w = 64; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) red[threadIdx.x] = (red[threadIdx.x] >= red[threadIdx.x + w] || red[threadIdx.x] != red[threadIdx.x]) ? red[threadIdx.x] : red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) bsp_atomic_max_pos(out + 1, red[0]);
    if (j == 0 && i + 1 < n) {
        /* ascending spectrum: record the most negative step as a positive number (0 = strictly ascending) */
        const double step = E[(size_t)p * n + i + 1] - E[(size_t)p * n + i];
        if (!(step > 0.0)) bsp_atomic_max_pos(out + 2, fabs(step) + 1e-300);
    }
}

bspatom_handle g_level0 = nullptr;
std::mutex g_level0_mu;   /* the LAPACK-shaped entries share one lazily created handle: calls are serialised */

/* that handle, created on the current device on first use (call with g_level0_mu held); nullptr and *info set on failure */
bspatom_handle level0_handle(int *info)
{
    if (!g_level0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) { *info = -100 - BSPATOM_ENODEVICE; return nullptr; }
        int rc = bspatom_create(&g_level0, dev);
        if (rc) { *info = -100 - rc; return nullptr; }
    }
    return g_level0;
}

} // namespace

extern "C" {

int bspatom_wavefunction(bspatom_handle h, int k, int nfun, int nkp, const double *rt, double ra, double rb,
                         int npts, int nvec, const double *C, double *r_out, double *psi_out)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (k < BSP_KMIN || k > BSP_KMAX) return BSPATOM_EUNSUPPORTED;
    if (nfun < 1 || nkp != nfun + k || !rt || npts < 1 || nvec < 1 || !C || !r_out || !psi_out) return -2;
    double *d_rt = nullptr, *d_C = nullptr, *d_r = nullptr, *d_psi = nullptr;
    if ((rc = dev_alloc(h, &d_rt, (size_t)nkp))) return rc;
    if ((rc = dev_alloc(h, &d_C, (size_t)nfun * nvec))) return rc;
    if ((rc = dev_alloc(h, &d_r, (size_t)npts + 1))) return rc;
    if ((rc = dev_alloc(h, &d_psi, (size_t)(npts + 1) * nvec))) return rc;
    CU(cudaMemcpyAsync(d_rt, rt, sizeof(double) * nkp, cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(d_C, C, sizeof(double) * (size_t)nfun * nvec, cudaMemcpyHostToDevice, h->st));
    switch (k) {
    case 3: launch_wavefunction<3>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 4: launch_wavefunction<4>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 5: launch_wavefunction<5>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 6: launch_wavefunction<6>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 7: launch_wavefunction<7>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 8: launch_wavefunction<8>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 9: launch_wavefunction<9>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    default: launch_wavefunction<10>(h, nfun, nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(r_out, d_r, sizeof(double) * ((size_t)npts + 1), cudaMemcpyDeviceToHost, h->st));
    CU(cudaMemcpyAsync(psi_out, d_psi, sizeof(double) * (size_t)(npts + 1) * nvec, cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    dev_free(h, d_rt, (size_t)nkp); dev_free(h, d_C, (size_t)nfun * nvec);
    dev_free(h, d_r, (size_t)npts + 1); dev_free(h, d_psi, (size_t)(npts + 1) * nvec);
    return 0;
}

int bspatom_dipole(bspatom_handle h, int n, int kd, const double *A_band, int nf, const double *Cf, int ni,
                   const double *Ci, double *D)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (n < 1) return -2;
    if (kd < 0 || kd >= n) return -3;
    if (!A_band) return -4;
    if (nf < 1) return -5;
    if (!Cf) return -6;
    if (ni < 1) return -7;
    if (!Ci) return -8;
    if (!D) return -9;
    const int ld = 2 * kd + 1;
    double *d_A = nullptr, *d_Cf = nullptr, *d_Ci = nullptr, *d_Y = nullptr, *d_D = nullptr;
    if ((rc = dev_alloc(h, &d_A, (size_t)ld * n))) return rc;
    if ((rc = dev_alloc(h, &d_Ci, (size_t)n * ni))) return rc;
    if ((rc = dev_alloc(h, &d_Y, (size_t)n * ni))) return rc;
    if ((rc = dev_alloc(h, &d_D, (size_t)nf * ni))) return rc;
    const bool same = (Cf == Ci && nf == ni);
    if (same) d_Cf = d_Ci;
    else if ((rc = dev_alloc(h, &d_Cf, (size_t)n * nf))) return rc;
    CU(cudaMemcpyAsync(d_A, A_band, sizeof(double) * (size_t)ld * n, cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(d_Ci, Ci, sizeof(double) * (size_t)n * ni, cudaMemcpyHostToDevice, h->st));
    if (!same) CU(cudaMemcpyAsync(d_Cf, Cf, sizeof(double) * (size_t)n * nf, cudaMemcpyHostToDevice, h->st));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, h->st));
    CU(bsp_launch_band_times_dense(h->st, n, kd, d_A, ni, d_Ci, d_Y, 1));
    h->launches++;
    CU(cudaGetLastError());
    CU(bsp_launch_dgemm_tn(h->st, nf, ni, n, d_Cf, n, d_Y, n, d_D, nf, 1, 0, 0, 0));
    h->launches++;
    CU(cudaEventRecord(e1, h->st));
    CU(cudaMemcpyAsync(D, d_D, sizeof(double) * (size_t)nf * ni, cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    h->stats[0] = 2; h->stats[7] = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dev_free(h, d_A, (size_t)ld * n); dev_free(h, d_Ci, (size_t)n * ni); dev_free(h, d_Y, (size_t)n * ni);
    dev_free(h, d_D, (size_t)nf * ni);
    if (!same) dev_free(h, d_Cf, (size_t)n * nf);
    return 0;
}

/* D_l = C_{l+1}^T A C_l for l = 0..nl-2 in two launches (cfg5: all bound/continuum pairs of
 * neighbouring angular momenta).  C_all: nl blocks n x nvec, D_all: nl-1 blocks nvec x nvec. */
int bspatom_dipole_chain(bspatom_handle h, int n, int kd, const double *A_band, int nl, int nvec,
                         const double *C_all, double *D_all)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (n < 1) return -2;
    if (kd < 0 || kd >= n) return -3;
    if (!A_band) return -4;
    if (nl < 2) return -5;
    if (nvec < 1) return -6;
    if (!C_all) return -7;
    if (!D_all) return -8;
    const int ld = 2 * kd + 1;
    const size_t blk = (size_t)n * nvec, dblk = (size_t)nvec * nvec;
    double *d_A = nullptr, *d_C = nullptr, *d_Y = nullptr, *d_D = nullptr;
    if ((rc = dev_alloc(h, &d_A, (size_t)ld * n))) return rc;
    if ((rc = dev_alloc(h, &d_C, blk * nl))) return rc;
    if ((rc = dev_alloc(h, &d_Y, blk * (nl - 1)))) return rc;
    if ((rc = dev_alloc(h, &d_D, dblk * (nl - 1)))) return rc;
    CU(cudaMemcpyAsync(d_A, A_band, sizeof(double) * (size_t)ld * n, cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(d_C, C_all, sizeof(double) * blk * nl, cudaMemcpyHostToDevice, h->st));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, h->st));
    CU(bsp_launch_band_times_dense(h->st, n, kd, d_A, nvec, d_C, d_Y, nl - 1));
    h->launches++;
    CU(cudaGetLastError());
    CU(bsp_launch_dgemm_tn(h->st, nvec, nvec, n, d_C + blk, n, d_Y, n, d_D, nvec, nl - 1, (long long)blk, (long long)blk,
                           (long long)dblk));
    h->launches++;
    CU(cudaEventRecord(e1, h->st));
    CU(cudaMemcpyAsync(D_all, d_D, sizeof(double) * dblk * (nl - 1), cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    h->stats[0] = 2; h->stats[7] = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dev_free(h, d_A, (size_t)ld * n); dev_free(h, d_C, blk * nl); dev_free(h, d_Y, blk * (nl - 1));
    dev_free(h, d_D, dblk * (nl - 1));
    return 0;
}

/* locate caller problem i of the resident batch: group, pencil */
static bool find_resident(bspatom_handle h, int i, Group *&Gout, int &pout)
{
    for (auto &G : h->groups)
        for (int p = 0; p < G.npencil; ++p)
            if (G.prob_index[p] == i) { Gout = &G; pout = p; return true; }
    return false;
}

/* eigenvectors computed for pencil p by the last run */
static int resident_nvec(bspatom_handle h, const Group &G, int p)
{
    return G.any_sel ? std::min(h->h_sel[G.sel_off + p], G.nvec[p]) : G.nvec[p];
}

/* cfg5 on the eigenvectors the last run LEFT IN HBM (no host round trip of the 8 MB blocks: the reference's TRANS_AMP
 * reads Hij / cinl in place, PhotoIon.f90:90-105): D_l = C_{i0+l+1}(:, 1:nvec)^T A C_{i0+l}(:, 1:nvec), l = 0..nl-2,
 * over the nl consecutive problems i0 .. i0+nl-1 of the resident batch. */
int bspatom_dipole_chain_resident(bspatom_handle h, int i0, int nl, int nvec, int kd, const double *A_band, double *D_all)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!h->ran) { h->err = "dipole_chain_resident before a run"; return BSPATOM_ESTATE; }
    if (i0 < 0 || i0 + nl > h->nprob) return -2;
    if (nl < 2) return -3;
    if (nvec < 1) return -4;
    if (!A_band) return -6;
    if (!D_all) return -7;
    Group *G = nullptr;
    int p0 = 0;
    if (!find_resident(h, i0, G, p0)) return -2;
    const int n = G->n;
    if (kd < 0 || kd >= n) return -5;
    std::vector<const double *> blocks(nl);
    bool uniform = true;
    for (int l = 0; l < nl; ++l) {
        Group *Gl = nullptr;
        int pl = 0;
        if (!find_resident(h, i0 + l, Gl, pl) || Gl != G) { h->err = "dipole_chain_resident: problems of different shapes"; return -2; }
        if (resident_nvec(h, *G, pl) < nvec) { h->err = "dipole_chain_resident: fewer eigenvectors resident than asked for"; return -4; }
        blocks[l] = G->d_C + G->coff[pl];
        if (l > 0 && blocks[l] - blocks[l - 1] != blocks[1] - blocks[0]) uniform = false;
    }
    const int ld = 2 * kd + 1;
    const size_t yblk = (size_t)n * nvec, dblk = (size_t)nvec * nvec;
    double *d_A = nullptr, *d_Y = nullptr, *d_D = nullptr;
    if ((rc = dev_alloc(h, &d_A, (size_t)ld * n))) return rc;
    if ((rc = dev_alloc(h, &d_Y, yblk * (nl - 1)))) return rc;
    if ((rc = dev_alloc(h, &d_D, dblk * (nl - 1)))) return rc;
    CU(cudaMemcpyAsync(d_A, A_band, sizeof(double) * (size_t)ld * n, cudaMemcpyHostToDevice, h->st));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, h->st));
    if (uniform) {
        const long long cs = (long long)(blocks[1] - blocks[0]);
        CU(bsp_launch_band_times_dense(h->st, n, kd, d_A, nvec, blocks[0], d_Y, nl - 1, cs, (long long)yblk));
        CU(cudaGetLastError());
        CU(bsp_launch_dgemm_tn(h->st, nvec, nvec, n, blocks[1], n, d_Y, n, d_D, nvec, nl - 1, cs, (long long)yblk, (long long)dblk));
        h->launches += 2;
    } else {
        for (int l = 0; l + 1 < nl; ++l) {
            CU(bsp_launch_band_times_dense(h->st, n, kd, d_A, nvec, blocks[l], d_Y + yblk * l, 1));
            CU(cudaGetLastError());
            CU(bsp_launch_dgemm_tn(h->st, nvec, nvec, n, blocks[l + 1], n, d_Y + yblk * l, n, d_D + dblk * l, nvec, 1, 0, 0, 0));
            h->launches += 2;
        }
    }
    CU(cudaEventRecord(e1, h->st));
    CU(cudaMemcpyAsync(D_all, d_D, sizeof(double) * dblk * (nl - 1), cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    h->stats[23] = ms;    /* device time of the contraction alone (the solver's own stats stay in place) */
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dev_free(h, d_A, (size_t)ld * n); dev_free(h, d_Y, yblk * (nl - 1)); dev_free(h, d_D, dblk * (nl - 1));
    return 0;
}

/* WRITE_WF on eigenvectors still resident: psi(ip, iv) for the vectors ivec0 .. ivec0+nvec-1 of problem iprob of
 * the last batch, on the problem's own knots (Bsp_Atom.f90:101-152 reads Hij(:, n0_ini) in place). */
int bspatom_wavefunction_resident(bspatom_handle h, int iprob, int ivec0, int nvec, double ra, double rb, int npts,
                                  double *r_out, double *psi_out)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!h->ran) { h->err = "wavefunction_resident before a run"; return BSPATOM_ESTATE; }
    if (h->band) { h->err = "wavefunction_resident: a band batch has no knots"; return BSPATOM_ESTATE; }
    Group *G = nullptr;
    int p = 0;
    if (iprob < 0 || iprob >= h->nprob || !find_resident(h, iprob, G, p)) return -2;
    if (ivec0 < 0 || nvec < 1 || ivec0 + nvec > resident_nvec(h, *G, p)) return -3;
    if (npts < 1 || !r_out || !psi_out) return -6;
    double *d_r = nullptr, *d_psi = nullptr;
    if ((rc = dev_alloc(h, &d_r, (size_t)npts + 1))) return rc;
    if ((rc = dev_alloc(h, &d_psi, (size_t)(npts + 1) * nvec))) return rc;
    const double *d_rt = G->d_rt + (size_t)G->inst[p] * G->nkp;
    const double *d_C = G->d_C + G->coff[p] + (size_t)ivec0 * G->n;
    switch (G->k) {
    case 3: launch_wavefunction<3>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 4: launch_wavefunction<4>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 5: launch_wavefunction<5>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 6: launch_wavefunction<6>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 7: launch_wavefunction<7>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 8: launch_wavefunction<8>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    case 9: launch_wavefunction<9>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    default: launch_wavefunction<10>(h, G->n, G->nkp, d_rt, ra, rb, npts, nvec, d_C, d_r, d_psi); break;
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(r_out, d_r, sizeof(double) * ((size_t)npts + 1), cudaMemcpyDeviceToHost, h->st));
    CU(cudaMemcpyAsync(psi_out, d_psi, sizeof(double) * (size_t)(npts + 1) * nvec, cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    dev_free(h, d_r, (size_t)npts + 1); dev_free(h, d_psi, (size_t)(npts + 1) * nvec);
    return 0;
}

/* General (structured-light) branch of TRANS_AMP, PhotoIon.f90:218-232: for one angular block (il, jl, component)
 * the reference loops over every (bra, ket) pair and calls ZHVMV = ZHEMV('U') + ZDOTU (Modules.f90:398-425) on the
 * N x N complex block zAij(:,:,il,jl,i) with the REAL eigenvectors as zx, zy.  ZHEMV('U') reads the upper triangle
 * only, takes the lower one as its conjugate and ignores the imaginary part of the diagonal, so
 *   T = Cf^T Re(A_h) Ci + i Cf^T Im(A_h) Ci,  Re(A_h) symmetric, Im(A_h) antisymmetric (zero diagonal),
 * two real banded-operator contractions that share Cf and Ci: two band x dense launches and one batched DMMA GEMM
 * give all (bra, ket) pairs of the block at once. */
int bspatom_trans_amp_hermitian(bspatom_handle h, int n, int kd, const double *zA_upper, int nf, const double *Cf,
                                int ni, const double *Ci, double *T)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (n < 1) return -2;
    if (kd < 0 || kd >= n) return -3;
    if (!zA_upper) return -4;
    if (nf < 1) return -5;
    if (!Cf) return -6;
    if (ni < 1) return -7;
    if (!Ci) return -8;
    if (!T) return -9;
    const int ld = 2 * kd + 1, ldu = kd + 1;
    const size_t abytes = (size_t)ld * n;
    std::vector<double> ab(2 * abytes, 0.0);   /* [0]: Re(A_h), [1]: Im(A_h), general band AB(kd+i-j, j) = A(i,j) */
    double *ar = ab.data(), *ai = ab.data() + abytes;
    for (int j = 0; j < n; ++j)
        for (int i = std::max(0, j - kd); i <= j; ++i) {
            const double re = zA_upper[2 * ((size_t)j * ldu + (kd + i - j))], im = zA_upper[2 * ((size_t)j * ldu + (kd + i - j)) + 1];
            ar[(size_t)j * ld + (kd + i - j)] = re;                 /* A(i,j) */
            ar[(size_t)i * ld + (kd + j - i)] = re;                 /* A(j,i) */
            if (i != j) {
                ai[(size_t)j * ld + (kd + i - j)] = im;
                ai[(size_t)i * ld + (kd + j - i)] = -im;
            }
        }
    const size_t yblk = (size_t)n * ni, dblk = (size_t)nf * ni;
    double *d_A = nullptr, *d_Cf = nullptr, *d_Ci = nullptr, *d_Y = nullptr, *d_D = nullptr;
    if ((rc = dev_alloc(h, &d_A, 2 * abytes))) return rc;
    if ((rc = dev_alloc(h, &d_Ci, yblk))) return rc;
    if ((rc = dev_alloc(h, &d_Y, 2 * yblk))) return rc;
    if ((rc = dev_alloc(h, &d_D, 2 * dblk))) return rc;
    const bool same = (Cf == Ci && nf == ni);
    if (same) d_Cf = d_Ci;
    else if ((rc = dev_alloc(h, &d_Cf, (size_t)n * nf))) return rc;
    CU(cudaMemcpyAsync(d_A, ab.data(), sizeof(double) * 2 * abytes, cudaMemcpyHostToDevice, h->st));
    CU(cudaMemcpyAsync(d_Ci, Ci, sizeof(double) * yblk, cudaMemcpyHostToDevice, h->st));
    if (!same) CU(cudaMemcpyAsync(d_Cf, Cf, sizeof(double) * (size_t)n * nf, cudaMemcpyHostToDevice, h->st));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, h->st));
    for (int part = 0; part < 2; ++part) {
        CU(bsp_launch_band_times_dense(h->st, n, kd, d_A + part * abytes, ni, d_Ci, d_Y + part * yblk, 1));
        h->launches++;
    }
    CU(cudaGetLastError());
    CU(bsp_launch_dgemm_tn(h->st, nf, ni, n, d_Cf, n, d_Y, n, d_D, nf, 2, 0, (long long)yblk, (long long)dblk));
    h->launches++;
    CU(cudaEventRecord(e1, h->st));
    std::vector<double> d(2 * dblk);
    CU(cudaMemcpyAsync(d.data(), d_D, sizeof(double) * 2 * dblk, cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    for (size_t q = 0; q < dblk; ++q) { T[2 * q] = d[q]; T[2 * q + 1] = d[dblk + q]; }
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    h->stats[0] = 3; h->stats[7] = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dev_free(h, d_A, 2 * abytes); dev_free(h, d_Ci, yblk); dev_free(h, d_Y, 2 * yblk); dev_free(h, d_D, 2 * dblk);
    if (!same) dev_free(h, d_Cf, (size_t)n * nf);
    return 0;
}


/* ---- several GPUs from ONE host process (the Fortran driver is one process): SURVEY.md 8(b) ---------------------- *
 * The problem list is cut into ndev contiguous ranges of equal weight (nfun^2 k per problem; a selection group is never
 * split), one handle and one host thread per device; every device writes its range of the caller's E / C / info directly
 * (contiguous slices: E is nfun_p doubles per problem, C nfun_p * nvec_p), so there is no exchange and no collective --
 * the work list shards by (instance, l) exactly like the one-process-per-GPU path of bench.py. */
struct bspatom_multi_s {
    std::vector<bspatom_handle> h;
    std::string err;
};

int bspatom_create_multi(bspatom_multi *m, int ndev, const int *dev_ids)
{
    if (!m) return -1;
    *m = nullptr;
    if (ndev < 1) return -2;
    if (!dev_ids) return -3;
    bspatom_multi x = new bspatom_multi_s();
    for (int d = 0; d < ndev; ++d) {
        bspatom_handle hd = nullptr;
        const int rc = bspatom_create(&hd, dev_ids[d]);
        if (rc) {
            for (auto y : x->h) bspatom_destroy(y);
            delete x;
            return rc;
        }
        x->h.push_back(hd);
    }
    *m = x;
    return 0;
}

int bspatom_destroy_multi(bspatom_multi m)
{
    if (!m) return -1;
    for (auto y : m->h) bspatom_destroy(y);
    delete m;
    return 0;
}

const char *bspatom_last_error_multi(bspatom_multi m) { return m ? m->err.c_str() : "null handle"; }

int bspatom_set_option_multi(bspatom_multi m, const char *name, double value)
{
    if (!m) return -1;
    int rc = 0;
    for (auto y : m->h) if (int r = bspatom_set_option(y, name, value)) rc = r;
    return rc;
}

int bspatom_solve_batch_multi(bspatom_multi m, int nprob, const bsp_problem *probs, double *E, double *C, int *info)
{
    if (!m) return -1;
    if (nprob < 1) return -2;
    if (!probs) return -3;
    if (!E) return -4;
    const int ndev = (int)m->h.size();
    std::vector<double> w(nprob);
    double tot = 0.0;
    for (int p = 0; p < nprob; ++p) { w[p] = (double)probs[p].nfun * probs[p].nfun * probs[p].k; tot += w[p]; }
    std::vector<int> cut(ndev + 1, nprob);
    cut[0] = 0;
    {
        double acc = 0.0;
        int d = 1;
        for (int p = 0; p < nprob && d < ndev; ++p) {
            acc += w[p];
            const bool in_group = p + 1 < nprob && probs[p].sel_mode && probs[p + 1].sel_mode && probs[p].sel_group >= 0 &&
                                  probs[p].sel_group == probs[p + 1].sel_group;
            if (acc >= tot * d / ndev && !in_group) cut[d++] = p + 1;
        }
    }
    std::vector<long long> eoff(nprob + 1, 0), coff(nprob + 1, 0);
    for (int p = 0; p < nprob; ++p) {
        eoff[p + 1] = eoff[p] + probs[p].nfun;
        coff[p + 1] = coff[p] + (long long)probs[p].nfun * std::max(0, probs[p].nvec);
    }
    std::vector<int> rcs(ndev, 0);
    std::vector<std::thread> th;
    for (int d = 0; d < ndev; ++d) {
        const int p0 = cut[d], p1 = cut[d + 1];
        if (p1 <= p0) continue;
        th.emplace_back([&, d, p0, p1] {
            rcs[d] = bspatom_solve_batch(m->h[d], p1 - p0, probs + p0, E + eoff[p0], C ? C + coff[p0] : nullptr,
                                         info ? info + p0 : nullptr);
        });
    }
    for (auto &t : th) t.join();
    for (int d = 0; d < ndev; ++d)
        if (rcs[d]) {
            m->err = "device " + std::to_string(d) + ": " + bspatom_last_error(m->h[d]);
            return rcs[d];
        }
    return 0;
}

/* ---- KIND_PI >= 3 branch of MATRIX_SVT: complex band matrices zAij from the tabulated angular integrals ------- */
int bspatom_assemble_zaij(bspatom_handle h, const bsp_problem *p, int kind_pi, int nblk, int ncomp_in, const double *zIth,
                          int ncomp_out, double *zA)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!p) return -2;
    if (kind_pi < 3) return -3;
    if (nblk < 1) return -4;
    if (!zIth) return -6;
    if (ncomp_out < 1 || ncomp_out > BSP_ZTERMS) return -7;
    if (!zA) return -8;
    bsp_problem q = *p;
    q.l = 0; q.nvec = 0;
    if ((rc = validate_problem(q))) return rc;
    BspZArgs a;
    memset(&a, 0, sizeof a);
    a.nterm = ncomp_out;
    int need_in = 1;
    for (int c = 0; c < ncomp_out; ++c) {
        BspZTerm &t = a.term[c];
        if (kind_pi == 3 || kind_pi == 4) {       /* matrices.f90:117-121 */
            t.src = c < 2 ? 0 : -1; t.div_r = (c == 0); t.deriv = (c == 1);
        } else {                                  /* :127-136 */
            t.src = (c < 2 || kind_pi >= 8) ? c : -1; t.div_r = 0; t.deriv = 0;
        }
        if (t.src >= 0) need_in = std::max(need_in, t.src + 1);
    }
    if (ncomp_in < need_in) return -5;
    Group G;
    G.k = q.k; G.B = q.k - 1; G.n = q.nfun; G.nkp = q.nkp; G.ka = q.ka; G.FS = 2 * G.B + 2;
    G.npad = BSP_NPAD(G.n, G.B);
    G.nrows = BSP_NROWS(G.npad, G.B);
    std::vector<const bsp_problem *> insts = {&q};
    G.ninst = 1;
    if ((rc = upload_group_instances(h, G, insts))) { free_group(h, G); return rc; }
    const int n = q.nfun, ld = 2 * q.k - 1;
    const size_t n_in = (size_t)q.nkp * q.ka * nblk * ncomp_in, n_out = (size_t)ld * n * nblk * ncomp_out;
    double *d_in = nullptr, *d_out = nullptr;
    if ((rc = dev_alloc(h, &d_in, 2 * n_in)) || (rc = dev_alloc(h, &d_out, 2 * n_out))) {
        if (d_in) dev_free(h, d_in, 2 * n_in);
        free_group(h, G);
        return rc;
    }
    cudaError_t e = cudaMemcpyAsync(d_in, zIth, sizeof(double) * 2 * n_in, cudaMemcpyHostToDevice, h->st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_out, 0, sizeof(double) * 2 * n_out, h->st);
    a.n = n; a.nkp = q.nkp; a.ka = q.ka; a.nblk = nblk;
    a.rt = G.d_rt; a.xgwg = G.d_xgwg;
    a.zIth = (const double2 *)d_in; a.zA = (double2 *)d_out;
    const dim3 grid((n + BSP_ZTR - 1) / BSP_ZTR, nblk);
    const size_t smem = sizeof(double) * (size_t)(BSP_ZTR + q.k - 1) * q.ka * (2 * q.k + 2);
    if (e == cudaSuccess) {
        switch (q.k) {
#define BSP_Z_CASE(K_) case K_: \
            e = cudaFuncSetAttribute(bsp_assemble_zaij_kernel<K_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            if (e == cudaSuccess) bsp_assemble_zaij_kernel<K_><<<grid, 128, smem, h->st>>>(a); break;
            BSP_Z_CASE(3) BSP_Z_CASE(4) BSP_Z_CASE(5) BSP_Z_CASE(6) BSP_Z_CASE(7) BSP_Z_CASE(8) BSP_Z_CASE(9) BSP_Z_CASE(10)
#undef BSP_Z_CASE
        default: rc = BSPATOM_EUNSUPPORTED; break;
        }
        h->launches++;
    }
    if (e == cudaSuccess && !rc) e = cudaGetLastError();
    if (e == cudaSuccess && !rc) e = cudaMemcpyAsync(zA, d_out, sizeof(double) * 2 * n_out, cudaMemcpyDeviceToHost, h->st);
    if (e == cudaSuccess && !rc) e = cudaStreamSynchronize(h->st);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); rc = BSPATOM_ECUDA; }
    dev_free(h, d_in, 2 * n_in); dev_free(h, d_out, 2 * n_out);
    free_group(h, G);
    return rc;
}

/* Device-side check of the batch that bspatom_batch_run left resident (nothing crosses PCIe but 4 doubles):
 *   out[0] = max over every eigenpair of every pencil of |H_l c - E S c|_inf / max(1, |E|)   (north star: < 1e-9)
 *   out[1] = max over every pencil of |C^T S C - I|                                          (DSYGV ITYPE=1 normalisation)
 *   out[2] = 0 if every spectrum is strictly ascending, else the largest non-positive step
 *   out[3] = number of eigenpairs checked
 * against the library's own assembled bands (whose parity with MATRIX_SVT is a separate 1e-13 test).  The Gram
 * matrices go through the batched DMMA GEMM, 2 N^3 flops per pencil. */
int bspatom_batch_verify(bspatom_handle h, double *out)
{
    int rc = check_device(h);
    if (rc) return rc;
    if (!out) return -2;
    if (!h->ran) { h->err = "batch_verify before batch_run"; return BSPATOM_ESTATE; }
    double *d_out = nullptr;
    if ((rc = dev_alloc(h, &d_out, 4))) return rc;
    CU(cudaMemsetAsync(d_out, 0, 4 * sizeof(double), h->st));
    double checked = 0.0;
    for (auto &G : h->groups) {
        /* with a device-side selection only the first nsel columns of a pencil were computed: check those */
        std::vector<int> nvec(G.npencil);
        const int *d_nvec = G.any_sel ? G.d_nvec_eff : G.d_nvec;
        int maxnv = 0;
        for (int p = 0; p < G.npencil; ++p) maxnv = std::max(maxnv, nvec[p] = resident_nvec(h, G, p));
        if (maxnv == 0) continue;
        /* scratch per pencil: Y (n x maxnv) + Gram (maxnv x maxnv); chunks of <= 2 GB */
        const size_t per = ((size_t)G.n + maxnv) * maxnv;
        const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)G.npencil, ((size_t)2 << 30) / (per * sizeof(double))));
        double *d_Y = nullptr, *d_G = nullptr;
        if ((rc = dev_alloc(h, &d_Y, (size_t)chunk * G.n * maxnv))) return rc;
        if ((rc = dev_alloc(h, &d_G, (size_t)chunk * maxnv * maxnv))) return rc;
        for (int p0 = 0; p0 < G.npencil; p0 += chunk) {
            const int np = std::min(chunk, G.npencil - p0);
            bsp_verify_matvec_kernel<<<dim3((G.n + 127) / 128, maxnv, np), 128, 0, h->st>>>(
                G.n, G.B, G.nrows, G.d_fbS, G.d_fbH0, G.d_fbQ, G.d_inst, G.d_cl, d_nvec, G.d_coff, G.d_C, G.d_E, d_Y,
                (long long)G.n * maxnv, p0, d_out);
            CU(cudaGetLastError());
            /* Gram matrices: pencils of a group may have different nvec, so one GEMM launch per run of equal nvec */
            int q = 0;
            while (q < np) {
                int q1 = q;
                const int nv = nvec[p0 + q];
                while (q1 + 1 < np && nvec[p0 + q1 + 1] == nv &&
                       G.coff[p0 + q1 + 1] - G.coff[p0 + q1] == (long long)G.n * nv) ++q1;
                if (nv > 0) {
                    CU(bsp_launch_dgemm_tn(h->st, nv, nv, G.n, G.d_C + G.coff[p0 + q], G.n, d_Y + (size_t)q * G.n * maxnv, G.n,
                                           d_G + (size_t)q * maxnv * maxnv, maxnv, q1 - q + 1, (long long)G.n * nv,
                                           (long long)G.n * maxnv, (long long)maxnv * maxnv));
                }
                q = q1 + 1;
            }
            bsp_verify_gram_kernel<<<dim3((std::max(maxnv, G.n) + 127) / 128, maxnv, np), 128, 0, h->st>>>(
                G.n, d_nvec, d_G, (long long)maxnv * maxnv, maxnv, G.d_E, p0, d_out);
            CU(cudaGetLastError());
            h->launches += 3;
        }
        for (int p = 0; p < G.npencil; ++p) checked += nvec[p];
        CU(cudaStreamSynchronize(h->st));
        dev_free(h, d_Y, (size_t)chunk * G.n * maxnv);
        dev_free(h, d_G, (size_t)chunk * maxnv * maxnv);
    }
    CU(cudaMemcpyAsync(out, d_out, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->st));
    CU(cudaStreamSynchronize(h->st));
    out[3] = checked;
    dev_free(h, d_out, 4);
    return 0;
}

/*
 * DSYGV-shaped entry.  Accepts the dense pencil exactly as matrices.f90:244-248
 * hands it to LAPACK, finds the half bandwidth from the zero pattern and runs
 * the banded device pipeline on it.  info: 0 ok; -i argument i illegal (also -5
 * when the pencil is not banded within the compiled range, half bandwidth <= 9);
 * 1..n eigenpairs missed the tolerance; n+i S not positive definite at minor i;
 * -100 - code for device errors.
 */
void bspatom_dsygv_(const int *itype, const char *jobz, const char *uplo, const int *n_, double *A, const int *lda_,
                    double *Bmat, const int *ldb_, double *w, double *work, const int *lwork, int *info, ...)
{
    (void)work; (void)lwork;
    if (!info) return;
    *info = 0;
    const int n = n_ ? *n_ : -1, lda = lda_ ? *lda_ : 0, ldb = ldb_ ? *ldb_ : 0;
    const bool wantz = jobz && (*jobz == 'V' || *jobz == 'v');
    const bool upper = uplo && (*uplo == 'U' || *uplo == 'u');
    if (!itype || *itype != 1) { *info = -1; return; }
    if (!jobz || !(wantz || *jobz == 'N' || *jobz == 'n')) { *info = -2; return; }
    if (!uplo || !(upper || *uplo == 'L' || *uplo == 'l')) { *info = -3; return; }
    if (n < 0) { *info = -4; return; }
    if (!A || lda < std::max(1, n)) { *info = -6; return; }
    if (!Bmat || ldb < std::max(1, n)) { *info = -8; return; }
    if (!w) { *info = -9; return; }
    if (n == 0) return;
    std::lock_guard<std::mutex> level0_lock(g_level0_mu);
    bspatom_handle h = level0_handle(info);
    if (!h) return;
    auto a = [&](const double *M, int ld, int i, int j) -> double {   /* symmetric read of the stored triangle */
        if (upper) return (i <= j) ? M[(size_t)j * ld + i] : M[(size_t)i * ld + j];
        return (i >= j) ? M[(size_t)j * ld + i] : M[(size_t)i * ld + j];
    };
    int kd = 0;
    for (int j = 0; j < n; ++j)
        for (int i = 0; i <= j; ++i) {
            const double va = upper ? A[(size_t)j * lda + i] : A[(size_t)i * lda + j];
            const double vb = upper ? Bmat[(size_t)j * ldb + i] : Bmat[(size_t)i * ldb + j];
            if ((va != 0.0 || vb != 0.0) && j - i > kd) kd = j - i;
        }
    if (kd > BSP_KMAX - 1) { *info = -5; h->err = "bspatom_dsygv_: pencil half bandwidth exceeds 9"; return; }
    const int B = std::max(kd, BSP_KMIN - 1);
    Group G;
    G.k = B + 1; G.B = B; G.n = n; G.nkp = n + G.k; G.ka = 1; G.FS = 2 * B + 2;
    G.npad = BSP_NPAD(n, B);
    G.nrows = BSP_NROWS(G.npad, B); G.xrows = G.npad + B + 1; G.ldw = ((n + 31) / 32) * 32;
    G.ninst = 1; G.npencil = 1;
    G.prob_index = {0}; G.inst = {0}; G.nvec = {wantz ? n : 0}; G.cl = {0.0}; G.coff = {0};
    G.c_elems = wantz ? (long long)n * n : 0;
    const size_t per_mat = (size_t)G.nrows * G.FS;
    std::vector<double> fbH(per_mat, 0.0), fbS(per_mat, 0.0);
    for (int i = 0; i < n; ++i)
        for (int c = 0; c <= 2 * B; ++c) {
            const int j = i - B + c;
            if (j < 0 || j >= n || abs(i - j) > kd) continue;
            fbH[(size_t)i * G.FS + c] = a(A, lda, i, j);
            fbS[(size_t)i * G.FS + c] = a(Bmat, ldb, i, j);
        }
    for (int i = n; i < G.nrows; ++i) fbH[(size_t)i * G.FS + B] = 1.0;
    auto fail = [&](int rc) { free_batch(h); *info = -100 - rc; };
    if (cudaSetDevice(h->dev) != cudaSuccess) { *info = -100 - BSPATOM_ECUDA; return; }
    free_batch(h);
    int rc = 0;
    double *d_L = nullptr;
    do {
        if ((rc = dev_alloc(h, &G.d_fbS, per_mat))) break;
        if ((rc = dev_alloc(h, &G.d_fbH0, per_mat))) break;
        if ((rc = dev_alloc(h, &G.d_fbQ, per_mat))) break;
        if ((rc = dev_alloc(h, &G.d_inst, 1))) break;
        if ((rc = dev_alloc(h, &G.d_nvec, 1))) break;
        if ((rc = dev_alloc(h, &G.d_cl, 1))) break;
        if ((rc = dev_alloc(h, &G.d_coff, 1))) break;
        if ((rc = dev_alloc(h, &G.d_pdinfo, 1))) break;
        if ((rc = dev_alloc(h, &G.d_bad, 1))) break;
        if ((rc = dev_alloc(h, &G.d_E, (size_t)n))) break;
        if ((rc = dev_alloc(h, &G.d_C, (size_t)G.c_elems))) break;
        if ((rc = dev_alloc(h, &d_L, (size_t)n * (B + 1)))) break;
    } while (0);
    if (rc) { free_group(h, G); dev_free(h, d_L, (size_t)n * (B + 1)); *info = -100 - rc; return; }
    cudaError_t ce = cudaSuccess;      /* first failing copy / launch of the set-up (checked once, below) */
    auto ck = [&](cudaError_t e) { if (ce == cudaSuccess) ce = e; };
    ck(cudaMemcpyAsync(G.d_fbS, fbS.data(), per_mat * sizeof(double), cudaMemcpyHostToDevice, h->st));
    ck(cudaMemcpyAsync(G.d_fbH0, fbH.data(), per_mat * sizeof(double), cudaMemcpyHostToDevice, h->st));
    ck(cudaMemsetAsync(G.d_fbQ, 0, per_mat * sizeof(double), h->st));
    ck(cudaMemcpyAsync(G.d_inst, G.inst.data(), sizeof(int), cudaMemcpyHostToDevice, h->st));
    ck(cudaMemcpyAsync(G.d_nvec, G.nvec.data(), sizeof(int), cudaMemcpyHostToDevice, h->st));
    ck(cudaMemcpyAsync(G.d_cl, G.cl.data(), sizeof(double), cudaMemcpyHostToDevice, h->st));
    ck(cudaMemcpyAsync(G.d_coff, G.coff.data(), sizeof(long long), cudaMemcpyHostToDevice, h->st));
    ck(cudaMemsetAsync(G.d_bad, 0, sizeof(int), h->st));
    bsp_pdcheck_kernel<<<1, 32, 0, h->st>>>(G.d_fbS, n, G.nrows, B, 1, G.d_pdinfo, d_L);
    ck(cudaGetLastError());
    h->launches++;
    int pd = 0;
    ck(cudaMemcpyAsync(&pd, G.d_pdinfo, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    ck(cudaStreamSynchronize(h->st));
    if (ce != cudaSuccess) {
        h->err = std::string("bspatom_dsygv_: ") + cudaGetErrorString(ce);
        free_group(h, G); dev_free(h, d_L, (size_t)n * (B + 1)); *info = -100 - BSPATOM_ECUDA; return;
    }
    if (pd) { free_group(h, G); dev_free(h, d_L, (size_t)n * (B + 1)); *info = n + pd; return; }
    /* run the eigen stages on this explicit pencil */
    h->groups.clear();
    h->groups.push_back(G);
    Group &GG = h->groups.back();
    ChunkPtrs c;
    const size_t need = carve_chunk(GG, 1, nullptr, c, use_ckpt(h, GG));
    ChunkTimes tm;
    bool ev_ok = true;
    for (int i = 0; i < 4; ++i) ev_ok = ev_ok && (cudaEventCreate(&tm.ev[i]) == cudaSuccess);
    rc = ev_ok ? ensure_workspace(h, need) : BSPATOM_ECUDA;
    int *d_report = nullptr;
    if (!rc) rc = dev_alloc(h, &d_report, (size_t)BSP_C_WORDS);
    if (!rc) {
        carve_chunk(GG, 1, h->ws.base, c, use_ckpt(h, GG));
        h->ev_used = 0;
        const BspSchedule sch = {h->opt.max_rounds, h->opt.min_iters, h->opt.max_iters};   /* one pencil: full limits at once */
        rc = enqueue_chunk(h, GG, 0, 1, c, sch, tm, d_report);
    }
    std::vector<double> Lb((size_t)n * (B + 1)), Cout(wantz ? (size_t)n * n : 0);
    int bad = 0;
    if (!rc) {
        cudaMemcpyAsync(w, GG.d_E, sizeof(double) * n, cudaMemcpyDeviceToHost, h->st);
        cudaMemcpyAsync(Lb.data(), d_L, sizeof(double) * Lb.size(), cudaMemcpyDeviceToHost, h->st);
        cudaMemcpyAsync(&bad, GG.d_bad, sizeof(int), cudaMemcpyDeviceToHost, h->st);
        if (wantz) cudaMemcpyAsync(Cout.data(), GG.d_C, sizeof(double) * Cout.size(), cudaMemcpyDeviceToHost, h->st);
        if (cudaStreamSynchronize(h->st) != cudaSuccess) rc = BSPATOM_ECUDA;
    }
    if (ev_ok) for (int i = 0; i < 4; ++i) cudaEventDestroy(tm.ev[i]);
    cudaStreamSynchronize(h->st);
    h->ev_used = 0;
    if (d_report) dev_free(h, d_report, (size_t)BSP_C_WORDS);
    dev_free(h, d_L, (size_t)n * (B + 1));
    if (rc) { fail(rc); return; }
    free_batch(h);
    /* eigenvectors overwrite A; the Cholesky factor overwrites the stored triangle of B */
    if (wantz)
        for (int j = 0; j < n; ++j) memcpy(A + (size_t)j * lda, Cout.data() + (size_t)j * n, sizeof(double) * n);
    for (int j = 0; j < n; ++j)
        for (int i = 0; i <= B && j + i < n; ++i) {
            const double v = Lb[(size_t)j * (B + 1) + i]; /* L(j+i, j) */
            if (upper) Bmat[(size_t)(j + i) * ldb + j] = v;   /* U(j, j+i) */
            else Bmat[(size_t)j * ldb + (j + i)] = v;
        }
    *info = bad;
}

/*
 * DSBGV-shaped entry: one pencil through bspatom_solve_band_batch on the shared handle.  Arguments are checked in
 * DSBGV's order (info = -i); AB and BB are only read.
 */
void bspatom_dsbgv_(const char *jobz, const char *uplo, const int *n_, const int *ka_, const int *kb_, double *AB,
                    const int *ldab_, double *BB, const int *ldbb_, double *w, double *Z, const int *ldz_, double *work,
                    int *info, ...)
{
    (void)work;
    if (!info) return;
    *info = 0;
    const bool wantz = jobz && (*jobz == 'V' || *jobz == 'v');
    const bool upper = uplo && is_upper(*uplo);
    const int n = n_ ? *n_ : -1, ka = ka_ ? *ka_ : -1, kb = kb_ ? *kb_ : -1;
    const int ldab = ldab_ ? *ldab_ : 0, ldbb = ldbb_ ? *ldbb_ : 0, ldz = ldz_ ? *ldz_ : 0;
    if (!jobz || !(wantz || *jobz == 'N' || *jobz == 'n')) { *info = -1; return; }
    if (!uplo || !(upper || *uplo == 'L' || *uplo == 'l')) { *info = -2; return; }
    if (n < 0) { *info = -3; return; }
    if (ka < 0 || ka > BSP_KMAX - 1) { *info = -4; return; }
    if (kb < 0 || kb > ka) { *info = -5; return; }
    if (!AB) { *info = -6; return; }
    if (ldab < ka + 1) { *info = -7; return; }
    if (!BB) { *info = -8; return; }
    if (ldbb < kb + 1) { *info = -9; return; }
    if (!w) { *info = -10; return; }
    if (wantz && !Z) { *info = -11; return; }
    if (ldz < 1 || (wantz && ldz < n)) { *info = -12; return; }
    if (n == 0) return;
    if (!band_finite(AB, ldab, ka, n, upper)) { *info = -6; return; }
    if (!band_finite(BB, ldbb, kb, n, upper)) { *info = -8; return; }
    std::lock_guard<std::mutex> level0_lock(g_level0_mu);
    bspatom_handle h = level0_handle(info);
    if (!h) return;
    const bsp_band_pencil p = {n, ka, kb, upper ? 'U' : 'L', AB, ldab, BB, ldbb, wantz ? n : 0};
    std::vector<double> E((size_t)n), Cv(wantz ? (size_t)n * n : 0);
    int pinfo = 0;
    const int rc = bspatom_solve_band_batch(h, 1, &p, E.data(), wantz ? Cv.data() : nullptr, &pinfo);
    free_batch(h);
    if (rc) { *info = -100 - rc; return; }
    *info = pinfo;
    if (pinfo > n) return;   /* B not positive definite: nothing was solved */
    memcpy(w, E.data(), sizeof(double) * n);
    if (wantz)
        for (int j = 0; j < n; ++j) memcpy(Z + (size_t)j * ldz, Cv.data() + (size_t)j * n, sizeof(double) * n);
}

} /* extern "C" */

#endif
