// CPU replay of the right-hand side the factor sweep forms from x (bsp_factor_forward_rows, bsp_core.h), against
// the order in which the back sweep's column sweep summed the same values.  TEST INFRASTRUCTURE ONLY, like
// emul_eig.cpp: tests/test_emul_rhs.py builds it.
//
// The formed values are read where the sweep itself stores them: the check-pointed form keeps, at every segment
// start, the raw right-hand side of rows js+B+1 .. js+2B+1 (BSP_CK_DOUBLES), so rows in those positions of every
// segment are observed directly, in whichever form (S x or (H - rho S) x) the sweep is instantiated for.
#include <cmath>
#include <cstring>
#include <vector>
#include "../../bspatom_b200/csrc/bsp_core.h"

// (S x)_i or fma(-rho, (S x)_i, (H x)_i) in the order of the column sweep of the back substitution: walk the rows
// from the last to the first; when x_j appears, rows j+1 .. j+B take A(j, j+d) x_j and row j starts from its upper
// part sum_{d=0..B} A(j, j+d) x_{j+d}.  swap = 1 sums the lower part first instead (a wrong order, for the test's
// sensitivity check).
template <int B>
static void column_sweep(int n, int npad, const double *H, const double *S, const double *x, double rho, int resid,
                         int swap, double *out)
{
    constexpr int FS = 2 * B + 2;
    auto xv = [&](int j) { return (j >= 0 && j < n) ? x[j] : 0.0; };
    for (int i = 0; i < n; ++i) {
        double h = 0.0, s = 0.0;
        auto upper = [&] {
            for (int d = 0; d <= B; ++d) {
                h = fma(H[(size_t)i * FS + B + d], xv(i + d), h);
                s = fma(S[(size_t)i * FS + B + d], xv(i + d), s);
            }
        };
        auto lower = [&] {
            for (int d = 1; d <= B && i - d >= 0; ++d) {
                h = fma(H[(size_t)(i - d) * FS + B + d], xv(i - d), h);
                s = fma(S[(size_t)(i - d) * FS + B + d], xv(i - d), s);
            }
        };
        if (swap) { lower(); upper(); } else { upper(); lower(); }
        out[i] = resid ? fma(-rho, s, h) : s;
    }
    (void)npad;
}

template <int B, int RHS>
static void formed(const BspEigChunk &g0, double *out)
{
    BspEigChunk g = g0;
    constexpr int K1 = B + 1, ST = BSP_CK_STEPS(B), CKD = BSP_CK_DOUBLES(B);
    BspRowsGlobal<B> src{g.fbH, g.fbS};
    bsp_factor_forward_rhs<B, RHS, true>(g, 0, 0, 0, true, src);
    for (int s = 0; s < g.npad / ST; ++s)
        for (int t = 0; t < K1; ++t) {
            const int row = s * ST + K1 + t;
            if (row < g.n) out[row] = g.CK[((size_t)s * CKD + CKD - K1 + t) * g.ldw];
        }
}

template <int B>
static int run(int n, const double *hb, const double *sb, const double *x, double rho, int resid, int swap,
               double *fused, double *ref)
{
    constexpr int FS = 2 * B + 2;
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
    for (int j = 0; j < n; ++j) X[(size_t)j * g.ldw] = x[j];
    const int inst = 0;
    double pbound[4] = {0.0, 0.0, 1.0, 1.0};
    std::vector<double> lo(g.ldw, -INFINITY), hi(g.ldw, INFINITY), sigma(g.ldw, rho), rr(g.ldw, rho), scale(g.ldw, 1.0);
    std::vector<double> CK((size_t)(g.npad / BSP_CK_STEPS(B)) * BSP_CK_DOUBLES(B) * g.ldw, NAN);
    g.fbH = H.data(); g.fbS = S.data(); g.inst = &inst; g.pbound = pbound;
    g.lo = lo.data(); g.hi = hi.data(); g.sigma = sigma.data(); g.rho = rr.data(); g.rho_prev = rr.data();
    g.scale = scale.data(); g.X = X.data(); g.CK = CK.data();
    for (int i = 0; i < n; ++i) fused[i] = NAN;
    if (resid) formed<B, BSP_RHS_RESID>(g, fused);
    else formed<B, BSP_RHS_SX>(g, fused);
    column_sweep<B>(n, g.npad, H.data(), S.data(), x, rho, resid, swap, ref);
    return 0;
}

// hb, sb: upper bands, hb[d * n + i] = A(i, i + d).  fused[i] = the formed raw right-hand side where the sweep
// stores it (NaN elsewhere), ref = the column-sweep order.
extern "C" int emul_rhs(int n, int B, const double *hb, const double *sb, const double *x, double rho, int resid,
                        int swap, double *fused, double *ref)
{
#define CASE(b) case b: return run<b>(n, hb, sb, x, rho, resid, swap, fused, ref);
    switch (B) { CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) default: return -2; }
}
