// The check-pointed factor kernel (bsp_factor_ckpt_kernel, bsp_kernels.cuh) on the device, with its staged band
// tiles and its cp.async look-ahead ring, forming the right-hand side from x; compared by tests/test_gpu_rhs.py with
// the column-sweep order of emul_rhs.cpp.  TEST INFRASTRUCTURE ONLY.
#include <cstdio>
#include <vector>
#include "../../bspatom_b200/csrc/bsp_kernels.cuh"
#include "emul_rhs.cpp"

#define CK_(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s\n", cudaGetErrorString(e_)); return -1; } } while (0)

template <class T>
static T *upload(const std::vector<T> &v)
{
    T *d = nullptr;
    if (cudaMalloc(&d, v.size() * sizeof(T)) != cudaSuccess) return nullptr;
    cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    return d;
}

// x: n x n, column e (x[e * n + j]) is the vector of eigen index e.  fused[e * n + i] = the formed raw right-hand side
// of row i (NaN where the check-points do not hold it), ref[e * n + i] = the column-sweep order.
extern "C" int gpu_rhs(int n, const double *hb, const double *sb, const double *x, double rho, int resid,
                       double *fused, double *ref)
{
    constexpr int B = 6, FS = 2 * B + 2, K1 = B + 1, ST = BSP_CK_STEPS(B), CKD = BSP_CK_DOUBLES(B);
    BspEigChunk g;
    memset(&g, 0, sizeof(g));
    g.n = n;
    g.npad = BSP_NPAD(n, B);
    g.nrows = BSP_NROWS(g.npad, B);
    g.xrows = g.npad + B + 1;
    g.ldw = ((n + 31) / 32) * 32;
    g.npencil = 1;
    std::vector<double> H((size_t)g.nrows * FS, 0.0), S((size_t)g.nrows * FS, 0.0);
    for (int i = 0; i < n; ++i)
        for (int d = 0; d <= B; ++d) {
            if (i + d < n) { H[(size_t)i * FS + B + d] = hb[(size_t)d * n + i]; S[(size_t)i * FS + B + d] = sb[(size_t)d * n + i]; }
            if (i - d >= 0) { H[(size_t)i * FS + B - d] = hb[(size_t)d * n + i - d]; S[(size_t)i * FS + B - d] = sb[(size_t)d * n + i - d]; }
        }
    for (int i = n; i < g.nrows; ++i) H[(size_t)i * FS + B] = 1.0;
    std::vector<double> X((size_t)g.xrows * g.ldw, 0.0);
    for (int e = 0; e < n; ++e)
        for (int j = 0; j < n; ++j) X[(size_t)j * g.ldw + e] = x[(size_t)e * n + j];
    const size_t nck = (size_t)(g.npad / ST) * CKD * g.ldw;
    std::vector<double> lo(g.ldw, -INFINITY), hi(g.ldw, INFINITY), rr(g.ldw, rho), one(g.ldw, 1.0), ck(nck, NAN);
    std::vector<double> pbound = {0.0, 0.0, 1.0, 1.0};
    std::vector<int> status(g.ldw, 0), inst(1, 0);
    double *dH = upload(H), *dS = upload(S), *dX = upload(X), *dlo = upload(lo), *dhi = upload(hi), *drho = upload(rr),
           *dsig = upload(rr), *dsc = upload(one), *dck = upload(ck), *dpb = upload(pbound);
    int *dst = upload(status), *dinst = upload(inst);
    if (!dH || !dS || !dX || !dlo || !dhi || !drho || !dsig || !dsc || !dck || !dpb || !dst || !dinst) return -1;
    g.fbH = dH; g.fbS = dS; g.X = dX; g.lo = dlo; g.hi = dhi; g.rho = drho; g.rho_prev = drho; g.sigma = dsig;
    g.scale = dsc; g.CK = dck; g.pbound = dpb; g.status = dst; g.inst = dinst;
    const dim3 grid((n + BSP_EIG_THREADS - 1) / BSP_EIG_THREADS, 1);
    if (resid) bsp_factor_ckpt_kernel<B, BSP_RHS_RESID><<<grid, BSP_EIG_THREADS>>>(g);
    else bsp_factor_ckpt_kernel<B, BSP_RHS_SX><<<grid, BSP_EIG_THREADS>>>(g);
    CK_(cudaGetLastError());
    CK_(cudaDeviceSynchronize());
    CK_(cudaMemcpy(ck.data(), dck, nck * sizeof(double), cudaMemcpyDeviceToHost));
    for (void *p : {(void *)dH, (void *)dS, (void *)dX, (void *)dlo, (void *)dhi, (void *)drho, (void *)dsig, (void *)dsc,
                    (void *)dck, (void *)dpb, (void *)dst, (void *)dinst})
        cudaFree(p);
    for (int e = 0; e < n; ++e) {
        double *f = fused + (size_t)e * n;
        for (int i = 0; i < n; ++i) f[i] = NAN;
        for (int s = 0; s < g.npad / ST; ++s)
            for (int t = 0; t < K1; ++t) {
                const int row = s * ST + K1 + t;
                if (row < n) f[row] = ck[((size_t)s * CKD + CKD - K1 + t) * g.ldw + e];
            }
        column_sweep<B>(n, g.npad, H.data(), S.data(), x + (size_t)e * n, rho, resid, 0, ref + (size_t)e * n);
    }
    return 0;
}
