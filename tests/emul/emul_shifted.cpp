// CPU replay of the shifted solves (bspatom_shifted_solve[_z]): the same per-thread bodies of bsp_core.h
// (bsp_shifted_factor_rows, bsp_shifted_forward_rows, bsp_shifted_back_rows, bsp_shifted_report) and the same step
// schedule as the device (bsp_api.cu: enqueue_shifted_b), one system after the other, band rows read straight from
// memory.  TEST INFRASTRUCTURE ONLY, like emul_eig.cpp: tests/test_emul_shifted.py builds it with -ffp-contract=off,
// so that every sum and product rounds as the explicit fma / mul / add of the device code.
#include <cmath>
#include <cstring>
#include <vector>
#include "../../bspatom_b200/csrc/bsp_core.h"

// full-band rows fb[i*FS + c] = A(i, i-B+c) from upper bands ub[d*n + i] = A(i, i+d), padded as the assembly pads
template <int B>
static std::vector<double> full_rows(int n, int nrows, const double *ub, double pad_diag)
{
    constexpr int FS = 2 * B + 2;
    std::vector<double> fb((size_t)nrows * FS, 0.0);
    for (int i = 0; i < n; ++i)
        for (int d = 0; d <= B; ++d) {
            if (i + d < n) fb[(size_t)i * FS + B + d] = ub[(size_t)d * n + i];
            if (i - d >= 0) fb[(size_t)i * FS + B - d] = ub[(size_t)d * n + i - d];
        }
    for (int i = n; i < nrows; ++i) fb[(size_t)i * FS + B] = pad_diag;
    return fb;
}

template <int B, class T>
static int run(int n, const double *h0b, const double *qb, const double *sb, double cl, int nsys, const double *z, int nrhs,
               const T *Bm, T *Xm, int *info, double *berr, int *steps)
{
    const int npad = BSP_NPAD(n, B), nrows = BSP_NROWS(npad, B);
    std::vector<double> H0 = full_rows<B>(n, nrows, h0b, 1.0), Q = full_rows<B>(n, nrows, qb, 0.0),
                        S = full_rows<B>(n, nrows, sb, 0.0), H(H0.size());
    for (size_t i = 0; i < H.size(); ++i) H[i] = bsp_combine_entry(cl, Q[i], H0[i]);
    constexpr bool CPLX = sizeof(T) == 16;
    const int ns = nsys;
    std::vector<int> sys(ns), inf(ns), done((size_t)nrhs * ns), iout(ns);
    std::vector<double> zr(ns), zi(ns), be((size_t)nrhs * ns), bp((size_t)nrhs * ns), bout(ns);
    std::vector<T> L((size_t)n * (B + 1) * ns), X((size_t)n * nrhs * ns), Y((size_t)n * nrhs * ns), Bv((size_t)n * nrhs * ns);
    for (int k = 0; k < ns; ++k) {
        sys[k] = k;
        zr[k] = z[CPLX ? 2 * k : k];
        zi[k] = CPLX ? z[2 * k + 1] : 0.0;
        for (int col = 0; col < nrhs; ++col)
            for (int r = 0; r < n; ++r) Bv[((size_t)col * n + r) * ns + k] = Bm[((size_t)k * nrhs + col) * n + r];
    }
    BspShiftChunk<T> c;
    memset(&c, 0, sizeof c);
    c.n = n; c.npad = npad; c.nslot = ns; c.nrhs = nrhs; c.nrows = nrows;
    c.fbH = H.data(); c.fbS = S.data(); c.sys = sys.data(); c.zr = zr.data(); c.zi = zi.data();
    c.L = L.data(); c.X = X.data(); c.Y = Y.data(); c.Bv = Bv.data();
    c.info = inf.data(); c.done = done.data(); c.berr = be.data(); c.bprev = bp.data();
    *steps = 0;
    unsigned long long corrections = 0;
    c.steps = steps;
    c.corrections = &corrections;
    BspRowsGlobal<B> src{H.data(), S.data()};
    for (int k = 0; k < ns; ++k) bsp_shifted_factor_rows<B, T>(c, k, true, src);
    for (int col = 0; col < nrhs; ++col)
        for (int step = 0; step <= BSP_SHIFT_MAXSTEPS + 1; ++step) {
            for (int k = 0; k < ns; ++k)
                if (bsp_shift_active(c, k, col)) bsp_shifted_forward_rows<B, T>(c, k, col, step, true, src);
            if (step <= BSP_SHIFT_MAXSTEPS)
                for (int k = 0; k < ns; ++k)
                    if (bsp_shift_active(c, k, col)) bsp_shifted_back_rows<B, T>(c, k, col, step);
        }
    for (int k = 0; k < ns; ++k) {
        bsp_shifted_report(c, k, iout.data(), bout.data());
        info[k] = iout[k];
        berr[k] = bout[k];
        if (iout[k] != 0 && iout[k] != n + 1) continue;   // X_s is not written
        for (int col = 0; col < nrhs; ++col)
            for (int r = 0; r < n; ++r) Xm[((size_t)k * nrhs + col) * n + r] = X[((size_t)col * n + r) * ns + k];
    }
    return 0;
}

// One pencil A = H0 + cl Q, B = S given as upper bands (ub[d*n + i] = M(i, i+d), d = 0..B), nsys shifts z (complex:
// interleaved), right-hand sides Bm / solutions Xm as n x nrhs column-major blocks per system (complex: interleaved).
extern "C" int emul_shifted(int n, int B, const double *h0b, const double *qb, const double *sb, double cl, int nsys,
                            const double *z, int nrhs, int cplx, const double *Bm, double *Xm, int *info, double *berr,
                            int *steps)
{
#define CASE(b)                                                                                                         \
    case b:                                                                                                             \
        return cplx ? run<b, BspZ>(n, h0b, qb, sb, cl, nsys, z, nrhs, (const BspZ *)Bm, (BspZ *)Xm, info, berr, steps) \
                    : run<b, double>(n, h0b, qb, sb, cl, nsys, z, nrhs, Bm, Xm, info, berr, steps);
    switch (B) { CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) default: return -2; }
#undef CASE
}
