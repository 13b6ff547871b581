/*
 * c_band_driver.c -- a plain C program against include/bspatom.h and libbspatom.so only: a pencil the library did not
 * assemble.  Radial hydrogen (l = 0) with linear finite elements on [0, R], psi(0) = psi(R) = 0: A = stiffness / 2 - 1/r,
 * B = consistent mass, both tridiagonal (ka = kb = 1).  The pencil goes through bspatom_solve_band_batch in upper and in
 * lower storage (the same bits), and through bspatom_dsbgv_ (the same bits again); the three lowest levels are checked
 * against E = -1/(2 n^2).
 * exit 0: ok;  77: no CUDA device (bspatom_create -> BSPATOM_ENODEVICE: the path has no CPU fallback);  1: failure.
 */
#include <math.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "bspatom.h"

enum { NN = 1500, NV = NN };   /* every eigenvector: the schedule bspatom_dsbgv_ runs with jobz = 'V' */

int main(void)
{
    printf("c_band_driver: sizeof(bsp_band_pencil) = %zu, offsets ka %zu kb %zu uplo %zu AB %zu ldab %zu BB %zu ldbb %zu nvec %zu\n",
           sizeof(bsp_band_pencil), offsetof(bsp_band_pencil, ka), offsetof(bsp_band_pencil, kb), offsetof(bsp_band_pencil, uplo),
           offsetof(bsp_band_pencil, AB), offsetof(bsp_band_pencil, ldab), offsetof(bsp_band_pencil, BB),
           offsetof(bsp_band_pencil, ldbb), offsetof(bsp_band_pencil, nvec));
    bspatom_handle h = NULL;
    int rc = bspatom_create(&h, 0);
    if (rc == BSPATOM_ENODEVICE) { printf("c_band_driver: no CUDA device (rc=%d), nothing computed\n", rc); return 77; }
    if (rc) { printf("c_band_driver: bspatom_create rc=%d\n", rc); return 1; }
    const double R = 60.0, hh = R / (NN + 1);
    /* 4-point Gauss-Legendre on [0, 1] */
    const double gx[4] = {0.0694318442029737, 0.3300094782075719, 0.6699905217924281, 0.9305681557970263};
    const double gw[4] = {0.1739274225687269, 0.3260725774312731, 0.3260725774312731, 0.1739274225687269};
    static double diagA[NN], offA[NN], diagB[NN], offB[NN];   /* off[j] = M(j-1, j) */
    int i, e, g;
    for (e = 0; e <= NN; ++e) {   /* element [e h, (e+1) h] couples nodes e and e+1 (1-based; nodes 0 and NN+1 are fixed) */
        double v00 = 0, v01 = 0, v11 = 0;
        for (g = 0; g < 4; ++g) {
            const double t = gx[g], r = (e + t) * hh, w = gw[g] * hh / r;
            v00 += w * (1 - t) * (1 - t); v01 += w * (1 - t) * t; v11 += w * t * t;
        }
        const double k = 0.5 / hh, m0 = hh / 3.0, m1 = hh / 6.0;
        if (e >= 1) { diagA[e - 1] += k - v00; diagB[e - 1] += m0; }
        if (e < NN) { diagA[e] += k - v11; diagB[e] += m0; }
        if (e >= 1 && e < NN) { offA[e] = -k - v01; offB[e] = m1; }
    }
    static double ABu[2 * NN], BBu[2 * NN], ABl[2 * NN], BBl[2 * NN];
    for (i = 0; i < NN; ++i) {
        ABu[2 * i + 1] = diagA[i]; ABu[2 * i] = i ? offA[i] : 0.0;      /* AB(2, j) = A(j, j), AB(1, j) = A(j-1, j) */
        BBu[2 * i + 1] = diagB[i]; BBu[2 * i] = i ? offB[i] : 0.0;
        ABl[2 * i] = diagA[i]; ABl[2 * i + 1] = i + 1 < NN ? offA[i + 1] : 0.0;   /* AB(1, j) = A(j, j), AB(2, j) = A(j+1, j) */
        BBl[2 * i] = diagB[i]; BBl[2 * i + 1] = i + 1 < NN ? offB[i + 1] : 0.0;
    }
    bsp_band_pencil p[2];
    memset(p, 0, sizeof p);
    p[0].n = NN; p[0].ka = 1; p[0].kb = 1; p[0].uplo = 'U'; p[0].AB = ABu; p[0].ldab = 2; p[0].BB = BBu; p[0].ldbb = 2; p[0].nvec = NV;
    p[1] = p[0];
    p[1].uplo = 'L'; p[1].AB = ABl; p[1].BB = BBl;
    double *E = (double *)bspatom_alloc_host(sizeof(double) * 2 * NN);
    double *Cv = (double *)bspatom_alloc_host(sizeof(double) * 2 * (size_t)NN * NV);
    int info[2] = {-1, -1};
    rc = bspatom_solve_band_batch(h, 2, p, E, Cv, info);
    if (rc) { printf("c_band_driver: bspatom_solve_band_batch rc=%d: %s\n", rc, bspatom_last_error(h)); return 1; }
    int bad = info[0] != 0 || info[1] != 0;
    if (memcmp(E, E + NN, sizeof(double) * NN) || memcmp(Cv, Cv + (size_t)NN * NV, sizeof(double) * NN * NV)) {
        printf("c_band_driver: upper and lower storage differ\n");
        bad = 1;
    }
    for (i = 0; i < 3; ++i) {
        const double want = -0.5 / ((i + 1.0) * (i + 1.0));
        printf("c_band_driver: E = %.12f (exact %.12f)\n", E[i], want);
        if (fabs(E[i] - want) > 2e-3) bad = 1;
    }
    /* the LAPACK-shaped entry on the same pencil */
    static double w[NN], Z[NN * NN], work[3 * NN];
    const int n = NN, ka = 1, kb = 1, ld = 2, ldz = NN;
    int dinfo = -1;
    bspatom_dsbgv_("V", "U", &n, &ka, &kb, ABu, &ld, BBu, &ld, w, Z, &ldz, work, &dinfo);
    if (dinfo != 0 || memcmp(w, E, sizeof(double) * NN) || memcmp(Z, Cv, sizeof(double) * NN * NV)) {
        printf("c_band_driver: bspatom_dsbgv_ info = %d, or its eigenpairs differ from the batch's\n", dinfo);
        bad = 1;
    }
    printf("c_band_driver: info = %d %d, dsbgv info = %d\n", info[0], info[1], dinfo);
    bspatom_free_host(E); bspatom_free_host(Cv);
    bspatom_destroy(h);
    printf(bad ? "c_band_driver: FAILED\n" : "c_band_driver: ok\n");
    return bad;
}
