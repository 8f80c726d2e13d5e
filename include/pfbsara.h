/*
 * pfbsara.h — C ABI of the device backward steps of the deconvolution major cycle:
 *   - SARA (SURVEY.md §8 row f2): the wavelet dictionary Psi (analysis `dot`, synthesis `hdot`), the fused l21 dual
 *     update, and the element-wise pieces of the primal-dual iteration;
 *   - the Clark CLEAN minor cycle of `pfb kclean` (core/kclean.py:203-218 -> deconv/clark.py).
 * Same conventions as pfbgrid.h: every entry point returns 0 or a PFBG_ERR_* code, pfbg_last_error() holds the
 * message, plain pointers and sizes only.
 *
 * Reference interfaces replaced (paths relative to /root/reference/src/pfb_imaging):
 *   - Psi / PsiNocopyt .dot / .hdot  (operators/psi.py:549-664; PsiBand :231-372, PsiBandNocopyt :466-530;
 *     transforms wavelets/wavelets.py:40-343, convolutions wavelets/convolutions.py)        -> pfbs_psi_dot / _hdot
 *   - dual_update_numba_fast (prox/prox_21m.py:104-135)                                     -> pfbs_dual_update
 *   - prox_21m_numba (prox/prox_21m.py:30-62)                                               -> pfbs_prox_21m
 *   - _nb_extrapolate_dual, _nb_primal_step, _nb_norm_diff (opt/primal_dual.py:16-61),
 *     positivity / positivity_band (prox/positivity.py:13-38)                               -> pfbs_extrapolate /
 *                                                                                              pfbs_primal_step / pfbs_norm_diff
 *   - clark (deconv/clark.py), semantics as restated in oracle/clark_np.py                  -> pfbs_clark_run
 *   - pcg on HessPSF / HessianTree (operators/hessian.py:357-522, opt/pcg.py:202-314)       -> pfbs_tree_cg
 */
#ifndef PFBSARA_H
#define PFBSARA_H

#include <stdint.h>

#include "pfbgrid.h"

#ifdef __cplusplus
extern "C" {
#endif

#define PFBS_KMAX 10          /* longest filter (db5) */
#define PFBS_TRANSPOSED 8u    /* coefficient arrays are (…, nymax, nxmax) (`Psi`) instead of (…, nxmax, nymax) (`PsiNocopyt`) */

typedef struct pfbs_psi pfbs_psi;

/*
 * One dictionary for `nband` images of (nx, ny).  Per basis b: K[b] = filter length (0 = 'self', the identity),
 * filters[b][4][PFBS_KMAX] = dec_lo, dec_hi, rec_lo, rec_hi (zero padded).  The packing arrays are those of
 * operators/psi.py:24-137: ix, iy (nbasis, nlevel, 2); sx, sy, spx, spy (nbasis, nlevel); ntotx, ntoty (nbasis).
 */
int pfbs_psi_create(int32_t precision, int32_t device, int32_t nband, int32_t nx, int32_t ny, int32_t nbasis,
                    int32_t nlevel, const int32_t* K, const double* filters, const int64_t* ix, const int64_t* iy,
                    const int64_t* sx, const int64_t* sy, const int64_t* spx, const int64_t* spy,
                    const int64_t* ntotx, const int64_t* ntoty, int32_t nxmax, int32_t nymax, pfbs_psi** out);
int pfbs_psi_destroy(pfbs_psi* psi);
/* x (nband, nx, ny) -> alpha (nband, nbasis, nxmax, nymax); alpha is fully overwritten (unused cells = 0). */
int pfbs_psi_dot(pfbs_psi* psi, const void* x, void* alpha, uint32_t flags, void* stream);
/* alpha -> x (nband, nx, ny) = sum over bases of the inverse transforms (overwritten). */
int pfbs_psi_hdot(pfbs_psi* psi, const void* alpha, void* x, uint32_t flags, void* stream);

/*
 * Fused dual update on device arrays: v (nband, ncoef) holds Psi^T xp on entry;
 *   vtilde = vp + sigma v;  s = |sum_band vtilde|;  v = vtilde * min(1, lam w / s)
 * phase 0: all in one kernel (every band on this device).
 * phase 1: v = vtilde and bsum (ncoef) = sum over the LOCAL bands;   [caller all-reduces bsum across ranks]
 * phase 2: v *= min(1, lam w / |bsum|).
 * vbar (optional, phases 0 and 2; needs vp): also receives the extrapolated dual 2 v - vp (_nb_extrapolate_dual,
 * opt/primal_dual.py:16-23) in the same pass.
 */
int pfbs_dual_update(int32_t precision, int32_t device, const void* vp, void* v, const void* weight, double lam,
                     double sigma, int32_t nband, int64_t ncoef, void* bsum, int32_t phase, void* vbar, void* stream);
/* result = v * max(|sum_band v / sigma| - lam w / sigma, 0) / |sum_band v / sigma| / sigma   (0 where the sum is 0) */
int pfbs_prox_21m(int32_t precision, int32_t device, const void* v, void* result, const void* weight, double lam,
                  double sigma, int32_t nband, int64_t ncoef, void* stream);
/* out = a x + b y on device arrays (out may alias x or y): the element-wise steps of the forward-backward loop
 * (opt/forward_backward.py:84-121) */
int pfbs_axpby(int32_t precision, int32_t device, void* out, double a, const void* x, double b, const void* y,
               int64_t n, void* stream);
/* vp = 2 v - vp */
int pfbs_extrapolate(int32_t precision, int32_t device, const void* v, void* vp, int64_t n, void* stream);
/* x = xp - tau * xout, then positivity: 0 none, 1 clamp negatives, 2 zero a pixel in all (local) bands if any band <= 0 */
int pfbs_primal_step(int32_t precision, int32_t device, void* x, const void* xp, const void* xout, double tau,
                     int32_t positivity, int32_t nband, int64_t npix, void* stream);
/* num_den[0] = sum (x - xp)^2, num_den[1] = sum x^2 (host output; synchronises the stream) */
int pfbs_norm_diff(int32_t precision, int32_t device, const void* x, const void* xp, int64_t n, double* num_den,
                   void* stream);

/* out2[0] = <a, b>, out2[1] = <c, d> on device arrays (host output; synchronises the stream): the scalar products of
 * the device-resident conjugate gradients (opt/pcg.py:35-41, 77-85) */
int pfbs_dot2(int32_t precision, int32_t device, const void* a, const void* b, const void* c, const void* d, int64_t n,
              double* out2, void* stream);

/*
 * Clark CLEAN minor cycle (fp64 only).  Images are (nband, nx, ny), raster index p = i*ny + j; the PSF is
 * (nband, nx_psf, ny_psf) with its centre at (nx_psf/2, ny_psf/2), nx <= nx_psf, ny <= ny_psf.  `psfhat` is its
 * r2c half spectrum rfft2(ifftshift(PSF)), (nband, nx_psf, ny_psf/2+1) complex128.  create uploads both once (one PSF
 * convolver per band) so that a handle serves every major cycle of a deconvolution; psf / psfhat are device pointers
 * when `flags` has PFBG_DEVICE_PTRS.
 *
 * run: R = dirty, model = 0; per major iteration k (at most maxit):
 *   s(p) = |sum_b R_b(p)| over pixels with mask[p] != 0 (mask NULL: all), Rmax = max s, on the first pass
 *   tol = max(pf Rmax, threshold); stop when Rmax <= tol;  A = {masked p : s(p) >= subpf Rmax} (raster order);
 *   subminor components while the peak of s over A > max(subpf Rmax, threshold), at most submaxit: a* = first
 *   maximum, d_b = gamma R_b(a*) / peak_b (0 where peak_b <= 0), model_b(a*) += d_b, R_b(a) -= d_b PSF_b(c + a - a*)
 *   on A;  then R = dirty - PSF (*) model through psfhat.
 * dirty, model, residual (nband, nx, ny) and mask (nx, ny) uint8 are device pointers with PFBG_DEVICE_PTRS (the call is
 * then asynchronous after its last host decision), else host pointers.  Info, host arrays: niter; per major iteration
 * rmax[k], nactive[k] = |A|, nsub[k] components; peaks (capacity peaks_cap >= maxit * submaxit) the raster index of
 * every component in order; times_ms (optional, 3 per major iteration): search + compaction, subminor (with the
 * model update), residual step, from CUDA events.
 */
#define PFBS_CLARK_MAX_BANDS 1024

typedef struct pfbs_clark pfbs_clark;

int pfbs_clark_create(int32_t precision, int32_t device, int32_t nband, int32_t nx, int32_t ny, int32_t nx_psf,
                      int32_t ny_psf, const void* psf, const void* psfhat, uint32_t flags, void* stream,
                      pfbs_clark** out);
int pfbs_clark_run(pfbs_clark* h, const void* dirty, const uint8_t* mask, void* model, void* residual,
                   double threshold, double gamma, double pf, int32_t maxit, double subpf, int32_t submaxit,
                   int32_t* niter, double* rmax, int64_t* nactive, int32_t* nsub, int64_t* peaks, int64_t peaks_cap,
                   float* times_ms, uint32_t flags, void* stream);
int pfbs_clark_destroy(pfbs_clark* h);

/*
 * Conjugate gradients on grouped PSF-convolution Hessians, every system at once, fp64 only: the corr-0 operator of a
 * band's HessianTree (operators/hessian.py:439-522), a sum over the beam groups g = group_start[s] ..
 * group_start[s+1]-1 of system s,
 *     A_s v = scale_s sum_g beam_g conv_g(beam_g v) + eta_s v      (scale_s = 1 / wsum_s)
 * applied with pfbg_conv_apply_scaled, accumulating through one scratch image.  HessPSF.idot(mode="psf")
 * (operators/hessian.py:357-436) is the case of one group per system and scale 1, A_b v = pfbg_conv_apply(conv[b], v,
 * beam[b], eta[b]).  conv[] and beam[] are the flattened group lists (beam[g] may be NULL), scale[] and eta[] have one
 * entry per system.  The convolvers are borrowed (any kernel mode) and must share (nx, ny) and `device`.
 * rhs and x are (nsys, nx, ny) device arrays, npix = nx * ny; x holds the starting point on entry and the solution on
 * return.  Per system, solvers.pcg with no preconditioner: iterate while (eps > tol or k < minit) and k < maxit and
 * stalls < 5, each system on its own; a system that stops is frozen and its convolutions are skipped.  Host outputs
 * per system: iters, eps and stop, one of the PFBS_CG_* codes below.  All reductions are deterministic.  Synchronises
 * `stream` once per iteration.  PFBG_ERR_ARG also for group_start[0] != 0, a system without a group, and a scale that
 * is not finite and > 0.
 * work: device memory of at least pfbs_tree_cg_work_bytes(nsys, group_start, npix) bytes (r, p, Ap, the reductions,
 * and one more image when some system has two or more groups; -1 for nsys < 1, npix < 1 or no group_start).
 */
#define PFBS_CG_CONVERGED 1
#define PFBS_CG_MAXIT 2
#define PFBS_CG_STALLED 3
#define PFBS_CG_ZERO_RESIDUAL 4 /* r = A x - b had r.r not > 0: x is left as it was */
#define PFBS_CG_EXACT 5         /* rho == 0 and p.Ap == 0: the iterate is the solution */

int64_t pfbs_tree_cg_work_bytes(int32_t nsys, const int32_t* group_start, int64_t npix);
int pfbs_tree_cg(int32_t device, int32_t nsys, const int32_t* group_start, pfbg_conv* const* conv,
                 const void* const* beam, const double* scale, const double* eta, const void* rhs, void* x,
                 int64_t npix, double tol, int32_t maxit, int32_t minit, void* work, int64_t work_bytes,
                 int32_t* iters, double* eps, int32_t* stop, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PFBSARA_H */
