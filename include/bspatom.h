/*
 * bspatom.h -- C-ABI of the B200-native replacement for BspAtom's hot path:
 * B-spline matrix assembly (MATRIX_SVT) + generalized symmetric eigensolve
 * H c = E S c per angular momentum l (SOLVE_SYSTEM / LAPACK DSYGV), batched,
 * plus the dense dipole contraction of TRANS_AMP.
 *
 * The reference (carlosmwh1985/BspAtom) has no FFI of its own; the seam this
 * header replaces is
 *     CALL MATRIX_SVT                      Bsp_Atom.f90:72   (matrices.f90:1-200)
 *     CALL SOLVE_SYSTEM                    Bsp_Atom.f90:75   (matrices.f90:204-394)
 *     CALL DSYGV(1,'V','U',nfun,Hij,...)   matrices.f90:248
 *     CALL DGEMV / DDOT                    PhotoIon.f90:95,103
 * INTEGRATION.md shows the ISO_C_BINDING interface module a maintainer adds.
 *
 * Conventions: everything FP64; matrices column-major (Fortran order); plain
 * pointers and sizes only; the caller owns every host buffer and the library
 * keeps no host pointer after a call returns.  Functions return 0 on success,
 * a negative value -i when argument i is invalid (LAPACK style), or a positive
 * BSPATOM_E* code; they never exit()/abort() -- the Fortran caller decides to
 * STOP (matrices.f90:250-254).  One handle drives ONE GPU; multi-GPU runs use
 * one process (handle) per GPU and shard the (problem, l) list (no collective
 * on the compute path).  There is NO CPU fallback: without a CUDA device every
 * entry point fails with BSPATOM_ENODEVICE.
 */
#ifndef BSPATOM_H
#define BSPATOM_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSPATOM_VERSION 100

/* positive error codes */
#define BSPATOM_ENODEVICE 1001 /* no CUDA device / driver                      */
#define BSPATOM_ECUDA 1002     /* CUDA runtime error (see bspatom_last_error)  */
#define BSPATOM_EUNSUPPORTED 1003 /* k (bandwidth) outside the compiled range  */
#define BSPATOM_ESTATE 1004    /* run/download called before upload            */
#define BSPATOM_ENOMEM 1005

/* potential kinds: 0..2 are the reference's KIND_POT (Modules.f90:263-295) */
#define BSPATOM_POT_COULOMB 0     /* -Z/r                    par = {Z}                    */
#define BSPATOM_POT_ROGERS 1      /* par = {Z, Ntot, N1,N2,N3, a1,a2,a3}                  */
#define BSPATOM_POT_SIMONS_FUES 2 /* -Z/r, Bl(l)/r^2 via ul_extra                         */
#define BSPATOM_POT_YUKAWA 10     /* -Z exp(-lambda r)/r     par = {Z, lambda}            */
#define BSPATOM_POT_TIETZ 11      /* -[1+(Z-1)/(1+t r)^2]/r  par = {Z, t}                 */
#define BSPATOM_POT_TABLE (-1)    /* V given at the quadrature points through v_tab       */

typedef struct bspatom_handle_s *bspatom_handle;

/*
 * One radial problem = one (instance, l) pencil.  Mirrors the module globals
 * MATRIX_SVT / SOLVE_SYSTEM read: nfun,k,ka,nkp,rt (Modules.f90:55-58), xg,wg
 * (Modules.f90:29), KIND_POT,Zatom,Numn,Ntot,alphan,Bl (Modules.f90:213-236).
 */
typedef struct bsp_problem {
    int k;            /* B-spline order                                           */
    int nfun;         /* basis size N (after READ_INPUTS' remap)                  */
    int nkp;          /* number of knots = nfun + k                               */
    int ka;           /* Gauss-Legendre points per knot interval (<= 32)          */
    const double *rt; /* knots rt(1:nkp) exactly as GRID computed them (host)     */
    const double *xg; /* GL nodes on [-1,1] (ka) or NULL: library runs gauleg     */
    const double *wg; /* GL weights (ka) or NULL                                  */
    int pot_kind;     /* BSPATOM_POT_*                                            */
    double pot_par[8];
    const double *v_tab; /* BSPATOM_POT_TABLE: V(r) at point g of interval m
                            (1-based m = 1..nkp-1) at v_tab[(m-1)*ka + g]        */
    int l;            /* angular momentum: U_l = [l(l+1) + 2 ul_extra] / (2 r^2)  */
    double ul_extra;  /* Bl(l) for KIND_POT=2 (matrices.f90:151), else 0          */
    int nvec;         /* leading eigenvectors wanted, 0..nfun (upper limit when sel_mode = 1) */
    /* Optional device-side state selection: what SOLVE_SYSTEM keeps of Hij for KIND_PI >= 3
     * (matrices.f90:296-334): ctemp(:, 1:ntemp, l), ntemp = MIN(MAX(n1_fin + 40, nlim), nfun) with
     * n1_fin = #{En <= Emax_fin} + 1 and nlim = the largest #{En <= Elim} of the l solved so far.
     * sel_mode = 1: every eigenvalue is still returned to rounding, but only the eigenvectors
     *   1 .. MIN(nvec, MAX(#{E <= sel_ecut_a} + sel_extra, running max over the group of #{E <= sel_ecut_b}))
     * are computed and copied out; problems of one group (same sel_group >= 0, contiguous in the array, in the
     * order of the reference's l loop) share the running maximum.  The reference's numbers: sel_ecut_a = Emax_fin,
     * sel_extra = 41, sel_ecut_b = Elim (= Emax_fin + 0.25, or Emax_fin for KIND_PI >= 8).  C keeps its layout
     * (nfun x nvec per problem); columns beyond the selected count are not written.  sel_mode = 0: off. */
    int sel_mode;
    int sel_extra;
    int sel_group;
    double sel_ecut_a;
    double sel_ecut_b;
} bsp_problem;

/* ---- handle ------------------------------------------------------------- */
int bspatom_create(bspatom_handle *h, int device_id);
int bspatom_destroy(bspatom_handle h);
const char *bspatom_last_error(bspatom_handle h);
int bspatom_version(void);

/* page-locked host memory for E / C: bspatom_solve_batch copies finished chunks into pinned
 * buffers while the next chunk is still computing (pageable buffers are filled after the run).
 * A Fortran host maps the pointer with C_F_POINTER.  NULL on failure.                      */
void *bspatom_alloc_host(size_t bytes);
void bspatom_free_host(void *p);

/* tunables: "tau", "delta_rel", "conv_tol", "res_tol", "rounds_enqueued", "max_rounds", "min_iters"
 * (2: every eigenpair gets two solves and a residual check, a third -- correction -- solve only where
 * ||r||_2 / gap > "vec_tol" (1e-12); 3: everybody gets the third solve; vec_tol = 1e300 is the fast
 * schedule: S-orthogonality of neighbouring vectors ~1e-8 instead of ~1e-11), "max_iters", "chunk",
 * "workers" (chunk streams of a resident batch, 1..8), "stream_chunks" / "stream_workers" (chunks and
 * chunk streams when results go to pinned host buffers), "trace" (1: chunk / copy timeline on stderr) */
int bspatom_set_option(bspatom_handle h, const char *name, double value);

/* ---- several GPUs from one host process (SURVEY.md 8(b): the Fortran driver is ONE process) ------------------- *
 * bspatom_create_multi opens one handle per listed device; bspatom_solve_batch_multi cuts the problem list into
 * ndev contiguous ranges of equal weight (a selection group is never split) and runs them concurrently, one host
 * thread per device, each writing its slice of the caller's E / C / info: the (instance, l) work list shards with no
 * exchange between devices (the l-loop bodies of SOLVE_SYSTEM share only read-only Sij, Tij, Vij, matrices.f90:242-248).
 * Same arguments, layout and error behaviour as bspatom_solve_batch.                                                */
typedef struct bspatom_multi_s *bspatom_multi;
int bspatom_create_multi(bspatom_multi *m, int ndev, const int *dev_ids);
int bspatom_destroy_multi(bspatom_multi m);
const char *bspatom_last_error_multi(bspatom_multi m);
int bspatom_set_option_multi(bspatom_multi m, const char *name, double value);
int bspatom_solve_batch_multi(bspatom_multi m, int nprob, const bsp_problem *probs, double *E, double *C, int *info);

/* ---- assembly: replaces MATRIX_SVT (matrices.f90:1-200) ------------------ *
 * Outputs in LAPACK band storage (any may be NULL):
 *   S, H0 = T+V, Q = int B_i B_j/(2 r^2), T, V, R = int B_i r B_j,
 *   Rinv = int B_i B_j / r              : upper band, AB(k,nfun), AB(kd+1+i-j,j)=A(i,j), kd=k-1
 *   D = int B_i B_j'  (non-symmetric)   : general band, AB(2k-1,nfun), AB(kd+1+i-j,j)=A(i,j)
 * so that  Uij(:,:,l) = [l(l+1)+2 Bl(l)] Q  and  Hij = T + U_l + V = H0 + c_l Q.
 * Only p->l independent fields of *p are read.                               */
int bspatom_assemble_band(bspatom_handle h, const bsp_problem *p, double *S, double *H0, double *Q,
                          double *T, double *V, double *R, double *Rinv, double *D);

/* ---- fused batched path: replaces MATRIX_SVT + the l-loop of SOLVE_SYSTEM -- *
 * E : sum_p nfun_p doubles, ascending per problem           (En, matrices.f90:248)
 * C : sum_p nfun_p*nvec_p doubles; problem p's block is column-major
 *     nfun_p x nvec_p, column j = eigenvector j, C^T S C = I  (Hij on exit of DSYGV).
 *     Sign: the first coefficient with |c_i| >= 1e-6 max|c| is positive.
 * info[p]: 0 ok; nfun+i: S not positive definite at pivot i; 1..nfun: that
 *     many eigenpairs missed the residual tolerance, left their bracket, or form a
 *     numerically degenerate pair (|E_i - E_{i+1}| <= 256 eps |E|): every vector comes
 *     from its own inverse iteration and nothing re-orthogonalises within such a pair
 *     (LAPACK's dstein would) -- radial Sturm-Liouville spectra are simple, so the
 *     reference's pencils never get there; an arbitrary pencil through bspatom_dsygv_
 *     can, and is told so through info instead of silently non-orthogonal vectors.  */
int bspatom_solve_batch(bspatom_handle h, int nprob, const bsp_problem *probs, double *E, double *C,
                        int *info);

/* same thing in three stages, so that a caller (and bench.py) can keep the
 * batch resident in HBM: upload copies knots/parameters H2D; run launches the
 * kernels only (no host<->device traffic, returns after the stream drained);
 * download copies E, C, info D2H.  C may be NULL to skip the eigenvectors.    */
int bspatom_batch_upload(bspatom_handle h, int nprob, const bsp_problem *probs);
int bspatom_batch_run(bspatom_handle h);
int bspatom_batch_download(bspatom_handle h, double *E, double *C, int *info);   /* E, C: host OR device pointers
                                   (unified addressing: a device destination keeps the eigenpairs on the GPU, e.g. as the
                                   send buffer of the NCCL gather to the rank that runs the writers) */

/* eigenvectors computed per problem by the last run (= nvec unless sel_mode = 1): nsel[nprob] */
int bspatom_get_selection(bspatom_handle h, int *nsel);

/* device-side check of the resident batch (after bspatom_batch_run): out[0] = max scaled residual
 * |H_l c - E S c|_inf / max(1,|E|) over EVERY eigenpair, out[1] = max |C^T S C - I| over every pencil,
 * out[2] = 0 when every spectrum is strictly ascending, out[3] = eigenpairs checked (with sel_mode = 1: the
 * selected ones, bspatom_get_selection, since only those eigenvectors were computed).  What the host would
 * otherwise verify after gathering Hij (matrices.f90:248) -- without moving the eigenvectors.           */
int bspatom_batch_verify(bspatom_handle h, double *out4);

/* ---- caller-supplied banded pencils (DSBGV semantics), batched ---------------- *
 * A x = lambda B x for pencils the caller assembled (a model or core-polarisation term added to Hij, another banded
 * discretisation such as FEM or Numerov), stored in LAPACK band storage.  The library keeps no pointer after a call. */
typedef struct bsp_band_pencil {
    int n;                 /* order, >= 0                                                  */
    int ka, kb;            /* half bandwidths of A and B, 0..9 (BSP_KMAX - 1)               */
    char uplo;             /* 'U': AB(ka+1+i-j, j) = A(i,j), max(1,j-ka) <= i <= j  (LAPACK)
                              'L': AB(1+i-j, j)    = A(i,j), j <= i <= min(n,j+ka)          */
    const double *AB; int ldab;   /* ldab >= ka+1, column-major (ldab, n)                    */
    const double *BB; int ldbb;   /* ldbb >= kb+1                                            */
    int nvec;              /* leading eigenvectors wanted, 0..n                             */
} bsp_band_pencil;

/* bspatom_band_upload takes the place of bspatom_batch_upload for a batch of band pencils; bspatom_batch_run,
 * bspatom_batch_download, bspatom_batch_verify, bspatom_get_selection and bspatom_dipole_chain_resident then work
 * unchanged.  bspatom_solve_band_batch is upload + run + download, with the E / C / info layout of
 * bspatom_solve_batch (offsets by n and nvec in the caller's order; pinned E / C are filled chunk by chunk).
 *  - Pencils are grouped by (n, B), B = max(min(max(ka, kb), n - 1), 2); narrower bands are zero-padded.  Each pencil is its own
 *    instance with c_l = 0 and Q = 0, so the solver sees H = A exactly.  Only the stored triangle is read.
 *  - Returns -3 for a malformed pencil (n < 0, ldab / ldbb too small, NULL AB / BB when n > 0, uplo not U / L,
 *    nvec outside 0..n, or a NaN / Inf in a stored band) before any device work, BSPATOM_EUNSUPPORTED for ka or
 *    kb > 9; bspatom_last_error names the pencil.
 *  - info[p] as for bspatom_solve_batch: n + i when B is not positive definite at pivot i (dpotrf / dpbtrf
 *    numbering), 1..n when that many eigenpairs missed the tolerance or form numerically degenerate pairs.
 *    B is checked during the upload: a pencil that fails never reaches the solver and its E / C slots are not
 *    written.  A pencil with n = 0 has info 0 and empty slots.
 *  - No knots: bspatom_wavefunction_resident returns BSPATOM_ESTATE after a band upload, and sign_rule = 1 (the
 *    literal CHKPHS) is skipped; every eigenvector gets the first-significant-coefficient-positive sign.
 *  - No device-side state selection (sel_mode): nvec only.                                                       */
int bspatom_band_upload(bspatom_handle h, int nprob, const bsp_band_pencil *pens);
int bspatom_solve_band_batch(bspatom_handle h, int nprob, const bsp_band_pencil *pens, double *E, double *C,
                             int *info);

/* LAPACK DSBGV on the batched band path (one pencil).  Arguments are checked in DSBGV's order and an invalid one
 * gives info = -i (also -4 for ka > 9, -6 / -8 for a NaN / Inf in the stored band of AB / BB).  On exit w is
 * ascending and, with jobz = 'V', Z(:, j) is eigenvector j, Z^T B Z = I, signs as for bspatom_solve_batch.  Unlike
 * LAPACK, AB and BB are left unchanged (no split-Cholesky factor is formed) and work is not used.  info > 0 as for
 * bspatom_solve_band_batch; -100 - code for a device error.  Calls share one handle and are serialised with
 * bspatom_dsygv_.  Trailing hidden CHARACTER lengths passed by Fortran compilers are ignored.                    */
void bspatom_dsbgv_(const char *jobz, const char *uplo, const int *n, const int *ka, const int *kb,
                    double *AB, const int *ldab, double *BB, const int *ldbb, double *w,
                    double *Z, const int *ldz, double *work, int *info, ...);

/* ---- LAPACK-compatible entry: one-token rename at matrices.f90:248 --------- *
 * DSYGV semantics for itype=1, jobz='V'|'N', uplo='U'|'L'.  The pencil must be
 * banded (bandwidth found from the zero pattern; the reference's matrices have
 * half-bandwidth k-1, matrices.f90:71-72).  On exit A(:,j) = eigenvector j,
 * w ascending, B = Cholesky factor (U^T U or L L^T).  Trailing hidden
 * CHARACTER lengths passed by Fortran compilers are ignored.                 */
void bspatom_dsygv_(const int *itype, const char *jobz, const char *uplo, const int *n, double *A,
                    const int *lda, double *B, const int *ldb, double *w, double *work,
                    const int *lwork, int *info, ...);

/* ---- dense contraction: replaces DGEMV+DDOT of TRANS_AMP (PhotoIon.f90:90-105)
 * D(nf,ni) = Cf^T * A * Ci, A given as general band AB(2*kd+1, n) (ld 2kd+1),
 * Cf: n x nf, Ci: n x ni, D: nf x ni, all column-major.                      */
int bspatom_dipole(bspatom_handle h, int n, int kd, const double *A_band, int nf, const double *Cf,
                   int ni, const double *Ci, double *D);

/* all neighbouring-l blocks at once (BASELINE cfg5): D_l = C_{l+1}^T A C_l, l = 0..nl-2.
 * C_all: nl column-major blocks n x nvec back to back (cinl(:,:,l), matrices.f90:369-373);
 * D_all: nl-1 column-major blocks nvec x nvec.                                  */
int bspatom_dipole_chain(bspatom_handle h, int n, int kd, const double *A_band, int nl, int nvec,
                         const double *C_all, double *D_all);

/* the same on the eigenvectors the last run left in HBM (no host round trip of the 8 MB blocks; the reference's
 * TRANS_AMP reads Hij / cinl in place): problems i0 .. i0+nl-1 of the resident batch (equal nfun, at least nvec
 * eigenvectors each), D_all as above; out of bspatom_get_stats: out[23] = device ms of the contraction.      */
int bspatom_dipole_chain_resident(bspatom_handle h, int i0, int nl, int nvec, int kd, const double *A_band,
                                  double *D_all);

/* ---- general branch of TRANS_AMP (structured light), PhotoIon.f90:218-232 ------ *
 * One angular block zAij(:,:,il,jl,i) against all (bra, ket) pairs at once:
 *   T(nf,ni) = Cf^T * ZHEMV_U(zA) * Ci   (what ZHVMV = ZHEMV('U') + ZDOTU, Modules.f90:398-425, gives pair by pair:
 *   upper triangle read, lower = its conjugate, imaginary part of the diagonal ignored; Cf, Ci real).
 * zA_upper: COMPLEX*16 upper band AB(kd+1, n), AB(kd+1+i-j, j) = zA(i,j) (re,im interleaved);
 * T: COMPLEX*16 nf x ni column-major.  The scalar ciall(i) and the B_0 term (ciall(5)*mi*Sij) are the caller's. */
int bspatom_trans_amp_hermitian(bspatom_handle h, int n, int kd, const double *zA_upper, int nf, const double *Cf,
                                int ni, const double *Ci, double *T);

/* ---- KIND_PI >= 3 branch of MATRIX_SVT (matrices.f90:110-139, 164-175) --------- *
 * zAij(ibra,jket,il,jl,c) = sum_ibet sum_igl fbra * W_c * (fket | dfket) * dr from the angular integrals the host
 * tabulates on the radial quadrature grid (ZINT_TH, Ang_Ints.f90:544-600):
 *   zIth : COMPLEX*16 zIth(nkp, ka, nblk, ncomp_in), nblk = nlm*nm blocks (il fastest), Fortran order
 *   zA   : COMPLEX*16 general band AB(2k-1, nfun, nblk, ncomp_out), AB(k+i-j, j) = zAij(i,j), Fortran order
 *   kind_pi = 3, 4 : c=1: W = zIth(..,1)/r with fket; c=2: W = zIth(..,1) with dfket; c=3,4 zero (as in the reference)
 *   kind_pi >= 5   : c=1,2: W = zIth(..,c) with fket; kind_pi >= 8 also c=3,4
 * Xij = int B_i r B_j (matrices.f90:174) is bspatom_assemble_band's R.  Only the knots / ka of *p are read.  */
int bspatom_assemble_zaij(bspatom_handle h, const bsp_problem *p, int kind_pi, int nblk, int ncomp_in,
                          const double *zIth, int ncomp_out, double *zA);

/* ---- wavefunction synthesis: WRITE_WF (Bsp_Atom.f90:101-152) --------------- *
 * psi(ip, iv) = sum_j C(j,iv) B_j(r_ip), r_ip = ra + ip (rb-ra)/npts, ip=0..npts */
int bspatom_wavefunction(bspatom_handle h, int k, int nfun, int nkp, const double *rt, double ra,
                         double rb, int npts, int nvec, const double *C, double *r_out,
                         double *psi_out);

/* the same for eigenvectors ivec0 .. ivec0+nvec-1 of problem iprob of the resident batch, on its own knots
 * (WRITE_WF reads Hij(:, n0_ini) in place, matrices.f90:266)                      */
int bspatom_wavefunction_resident(bspatom_handle h, int iprob, int ivec0, int nvec, double ra, double rb,
                                  int npts, double *r_out, double *psi_out);

/* ---- statistics of the last run (for bench.py) ----------------------------- *
 * out[0] kernel launches, out[1] multisection rounds, out[2] refinement
 * iterations, out[3] ms in assembly, out[4] ms eigenvalue stage, out[5] ms
 * eigenvector stage, out[6] ms finalize, out[7] total device ms,
 * out[8..11] summed device ms of the multisection / factor / back-substitution /
 * assembly kernels (CUDA events around each launch), out[12..15] their launch counts */
int bspatom_get_stats(bspatom_handle h, double *out, int nout);

#ifdef __cplusplus
}
#endif
#endif /* BSPATOM_H */
