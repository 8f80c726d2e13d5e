/*
 * pfbgrid.h — C ABI of the B200-native w-stacked gridder / degridder and
 * Hessian apply that replaces pfb-imaging's calls into ducc0.wgridder.
 *
 * Every entry point returns 0 on success and a non-zero status otherwise; the
 * message of the last failure on the calling thread is pfbg_last_error().
 * Nothing aborts or throws across this boundary.  All pointers are plain host
 * or device pointers (selected by PFBG_DEVICE_PTRS in `flags`); no torch /
 * numpy types appear in the signatures.
 *
 * Reference interfaces replaced (paths relative to /root/reference):
 *   - ducc0.wgridder.experimental.vis2dirty as called at
 *       src/pfb_imaging/operators/gridder.py:78-100, 590-613, 633-656,
 *       672-695, 709-732, 852-875, 888-911, 990-1013, 1087-1111 and
 *       src/pfb_imaging/operators/hessian.py:68-89         -> pfbg_grid
 *   - ducc0.wgridder.experimental.dirty2vis as called at
 *       operators/gridder.py:128-143, 350-365, 485-503, 972-989, 1067-1085
 *       and operators/hessian.py:50-66                      -> pfbg_degrid
 *   - hessian_slice (operators/hessian.py:15-100)           -> pfbg_hessian
 *   - the per-band pinned state of _BandWorkerImpl.load_band
 *       (operators/band_worker.py:61-106)                   -> pfbg_bind_vis /
 *                                                              pfbg_bind_weights
 *   - _compute_counts / counts_to_weights
 *       (utils/weighting.py:81-140, 143-208)                -> pfbg_counts /
 *                                                              pfbg_counts_to_weights
 *   - the same per snapshot of `pfb hci`
 *       (utils/stokes2im.py:563-604)                        -> pfbg_counts_to_weights_batch /
 *                                                              pfbg_bind_weights_robust
 *   - the l2 re-weighting block of image_data_products
 *       (operators/gridder.py:509-532)                      -> pfbg_l2_reweight
 */
#ifndef PFBGRID_H
#define PFBGRID_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFBG_OK 0
#define PFBG_ERR_ARG 1
#define PFBG_ERR_CUDA 2
#define PFBG_ERR_CUFFT 3
#define PFBG_ERR_STATE 4
#define PFBG_ERR_NOMEM 5

/* precision of vis / weights / image and of all grid arithmetic */
#define PFBG_F32 0 /* vis complex64,  wgt float32, image float32 */
#define PFBG_F64 1 /* vis complex128, wgt float64, image float64 */

/* flags */
#define PFBG_HOST_PTRS 0u
#define PFBG_DEVICE_PTRS 1u   /* data pointers are device pointers; call is asynchronous on `stream` */
#define PFBG_APPLY_WGT 2u     /* degrid: multiply the output by the bound/passed weights */
#define PFBG_NO_MASK_ZERO 4u  /* degrid: leave masked output samples untouched instead of zeroing */
/* pfbg_plan_desc.flags */
#define PFBG_PLAN_EXTERNAL_STACK 1 /* do not allocate the plane stack: the caller lends one (pfbg_plan_set_stack) */

#define PFBG_PINNED_IN 16u    /* host-pointer calls: the input image(s) are page-locked (pfbg_host_register): DMA directly */
#define PFBG_PINNED_OUT 32u   /* host-pointer calls: the output image is page-locked */
#define PFBG_BEAM_CACHED 64u  /* pfbg_hessian, host pointers: `beam` equals the beam of the previous call on this plan
                               * (the caller vouches for it): use the device copy instead of uploading it again */

typedef struct pfbg_plan pfbg_plan;

/* Everything the host-side plan (pfb-imaging_b200/plan.py) decides. */
typedef struct pfbg_plan_desc {
  int32_t precision;     /* PFBG_F32 | PFBG_F64 */
  int32_t device;        /* CUDA device ordinal */
  int32_t nx, ny;        /* image size (even) */
  int32_t nu, nv;        /* oversampled grid (multiples of 32) */
  int32_t W;             /* kernel support, 4..16; 4..8 in fp32 */
  int32_t nplanes;       /* w-planes (1 when do_wgridding == 0) */
  int32_t do_wgridding;
  int32_t divide_by_n;
  double beta;           /* ES kernel shape */
  double pixsize_x, pixsize_y;
  double center_x, center_y; /* after the flip rule */
  double usign, vsign, wsign; /* +-1 */
  double w0, dw, nshift; /* plane p sits at w0 + p*dw; the planes must cover |w| f/c of all samples:
                          * samples with w < 0 are folded onto -(u,v,w) with the conjugate visibility */
  const double* corr_u;  /* host (nx): 1/psihat_u */
  const double* corr_v;  /* host (ny) */
  const double* gl_x;    /* host (n_gl): Gauss-Legendre nodes on (0,1) */
  const double* gl_w;    /* host (n_gl) */
  int32_t n_gl;
  int32_t pmirror;       /* 0, or the number of virtual planes below plane 0 (mirror planes): then w0 == dw/2, so
                          * plane -p-1 is the Hermitian mirror of plane p (G_{-p-1}(u,v) = conj G_p(-u,-v), the
                          * image being real) and samples near w = 0 use the mirrored cells of planes 0..pmirror-1
                          * instead of planes that would have to be stored and transformed */
  int32_t fast_screen;   /* fp32 plans only: w-screen phasors from the SFU (sin.approx / cos.approx after the fp64
                          * range reduction, abs. error ~5e-7) instead of sincospif; for epsilon >= 3e-6 */
  int32_t flags;         /* PFBG_PLAN_* bits */
} pfbg_plan_desc;

typedef struct pfbg_plan_info {
  int64_t nrow;
  int64_t nvis;          /* nrow * nchan */
  int64_t nactive;       /* samples with mask != 0 */
  int64_t grid_bytes;    /* plane stack */
  int64_t total_bytes;   /* all device allocations of the plan */
  int32_t nchan;
  int32_t nplanes;
  int32_t nu, nv, W;
  int32_t n_work_items;  /* tile work items of the gridding kernel */
} pfbg_plan_info;

const char* pfbg_last_error(void);
/* 102: pfbg_plan_create and pfbg_split_helper_create reject PFBG_F32 with W > 8 (PFBG_ERR_ARG) */
int pfbg_version(void);
int pfbg_device_count(int32_t* count);

int pfbg_plan_create(const pfbg_plan_desc* desc, pfbg_plan** out);
int pfbg_plan_destroy(pfbg_plan* plan);
int pfbg_plan_get_info(const pfbg_plan* plan, pfbg_plan_info* info);
/* Re-target a plan to another w-plane range (w0, nplanes, pmirror); everything that depends only on the image
 * geometry, sigma and W is kept.  Unbinds the visibilities.  Used to pool plans across the thousands of
 * small snapshot images of `pfb hci` (utils/stokes2im.py:635-683). */
int pfbg_plan_set_wrange(pfbg_plan* plan, double w0, int32_t nplanes, int32_t pmirror);
/*
 * Lend the plan a plane stack (device memory of the plan's device, 256-byte aligned, at least nplanes * nu * nv
 * complex cells).  The stack is scratch between calls, so the bands that share a GPU — the reference keeps one
 * worker per band, operators/band_worker.py:217-246 — can take turns on one stack per compute stream instead of
 * holding one each (config 4: 62 GB per band at 10240^2).  The caller keeps calls that share a stack on one stream.
 * dev_ptr == NULL takes the loan back.  Plans of a split band (pfbg_split_*) cannot borrow.
 */
int pfbg_plan_set_stack(pfbg_plan* plan, void* dev_ptr, uint64_t bytes);

/*
 * Batched snapshots (`pfb hci`: utils/stokes2im.py:635-683 makes two vis2dirty calls per 512^2 snapshot, thousands
 * of snapshots): nbatch images of ONE geometry (nx, ny, cell, centre, sigma, W, dw — everything in the plan desc)
 * go through one bin/sort, one launch of every kernel.  Snapshot s owns snap_np[s] planes starting at w = snap_w0[s]
 * (host arrays; the planes of all snapshots form one stack) and the rows [row_offsets[s], row_offsets[s+1]) of the
 * arrays given to pfbg_bind_vis_batch.  Afterwards the image arguments of pfbg_grid / pfbg_degrid / pfbg_hessian are
 * (nbatch, nx, ny).  The plan must be created without mirror planes (pmirror = 0).
 */
int pfbg_plan_set_batch(pfbg_plan* plan, int32_t nbatch, const double* snap_w0, const int32_t* snap_np);
int pfbg_bind_vis_batch(pfbg_plan* plan, const double* uvw, const double* fscale, const uint8_t* mask,
                        int64_t nrow, int32_t nchan, const int64_t* row_offsets, uint32_t flags, void* stream);

/*
 * Kernel 1: upload uvw (nrow,3) f64, fscale (nchan) f64 = freq/c, optional mask
 * (nrow,nchan) u8, compute the uv-tile / w-plane bucket of every sample and
 * sort the active samples by bucket.  Cached in the plan until re-bound.
 */
int pfbg_bind_vis(pfbg_plan* plan, const double* uvw, const double* fscale, const uint8_t* mask,
                  int64_t nrow, int32_t nchan, uint32_t flags, void* stream);

/* Optional cached imaging weights (nrow,nchan) of the plan's precision; NULL unbinds. */
int pfbg_bind_weights(pfbg_plan* plan, const void* wgt, uint32_t flags, void* stream);

/*
 * Bit-exact check of kernel 1.  Host outputs; any pointer may be NULL.
 * iu0/iv0/ip0/key have nvis entries (row-major, also for masked samples);
 * sorted_idx has nactive entries (flat sample index in bucket order).
 */
int pfbg_bin_dump(pfbg_plan* plan, int32_t* iu0, int32_t* iv0, int32_t* ip0, uint64_t* key,
                  uint32_t* sorted_idx);

/*
 * Kernel 2 (+4, cuFFT): dirty (nx,ny) = R^H (wgt * mask * vis).
 * vis has element strides (vis_rs, vis_cs) (both 0 = one broadcast value);
 * wgt may be NULL (then the bound weights, if any, are used).
 */
int pfbg_grid(pfbg_plan* plan, const void* vis, int64_t vis_rs, int64_t vis_cs, const void* wgt,
              void* dirty, uint32_t flags, void* stream);

/*
 * PSF of an off-centre field (operators/gridder.py:616-629, 877-911; utils/stokes2im.py:483-486, SURVEY §8 a13):
 * grids vis[r,c] = exp(sign * 2 pi i f_c/c0 (u x0 + v y0 - w (n0 - 1))), n0 = sqrt(1 - x0^2 - y0^2), with the
 * unflipped bound u, v, w.  The visibilities are generated on the device (the reference materialises an
 * (nrow, nchan) complex128 array on the host); sign = +1 at the gridder.py call sites, -1 at stokes2im.py's.
 */
int pfbg_grid_psf(pfbg_plan* plan, double x0, double y0, double sign, const void* wgt, void* dirty,
                  uint32_t flags, void* stream);

/* Kernel 3 (+4, cuFFT): vis (nrow,nchan) contiguous = R dirty; masked samples are zeroed. */
int pfbg_degrid(pfbg_plan* plan, const void* dirty, void* vis, const void* wgt, uint32_t flags,
                void* stream);

/*
 * Fused Hessian apply (operators/hessian.py:15-100):
 *   out = beam * R^H W M R (beam * x) / wsum + eta * x
 * beam may be NULL, wsum <= 0 means "no division", eta == 0 means "no ridge".
 * Uses the bound weights (or none).  Model visibilities never leave the device.
 */
int pfbg_hessian(pfbg_plan* plan, const void* x, const void* beam, double wsum, double eta,
                 void* out, uint32_t flags, void* stream);

/* Page-lock / unlock a caller-owned host range (cudaHostRegister) so that host-pointer calls flagged PFBG_PINNED_*
 * copy without the pinned staging buffer.  The range must be unregistered before its memory is freed. */
int pfbg_host_register(void* ptr, uint64_t bytes);
int pfbg_host_unregister(void* ptr);

/* 64-bit content hash of a host range (multi-threaded, a few ms per 100 MB).  The host-side plan cache of
 * pfb_imaging_b200.operators validates a cached band binding with it on every call: the reference keeps no state
 * between hessian_slice calls (operators/hessian.py:15-100), so an in-place edit of weights, flags or beam between
 * two calls must be seen. */
int pfbg_host_hash64(const void* ptr, uint64_t bytes, uint64_t* out);

/* Seconds spent in the phases of the last grid/degrid/hessian call when profiling is on. */
int pfbg_set_profiling(pfbg_plan* plan, int32_t on);
int pfbg_get_timings(pfbg_plan* plan, float* ms, int32_t n, int32_t* n_written);

/* Number of kernels this library has launched on the calling process so far. */
int64_t pfbg_launch_count(void);

/*
 * Imaging-weight kernels (utils/weighting.py:81-140, 143-208).
 * counts (ncorr,nx,ny) of `precision`; wgt (ncorr,nrow,nchan); mask (nrow,nchan) u8.
 */
int pfbg_counts(int32_t precision, int32_t device, const double* uvw, const double* freq,
                const uint8_t* mask, const void* wgt, int64_t nrow, int32_t nchan, int32_t ncorr,
                int32_t nx, int32_t ny, double cell_x, double cell_y, double usign, double vsign,
                void* counts, uint32_t flags, void* stream);
/* Bit-exact check of the counts cell index: cells (nrow,nchan,2) int32 host output,
 * (-1,-1) for masked / off-grid samples.  Host pointers only. */
int pfbg_counts_cells(int32_t device, const double* uvw, const double* freq, const uint8_t* mask,
                      int64_t nrow, int32_t nchan, int32_t nx, int32_t ny, double cell_x, double cell_y,
                      double usign, double vsign, int32_t* cells);
int pfbg_counts_to_weights(int32_t precision, int32_t device, void* counts, const double* uvw,
                           const double* freq, void* wgt, const uint8_t* mask, int64_t nrow,
                           int32_t nchan, int32_t ncorr, int32_t nx, int32_t ny, double cell_x,
                           double cell_y, double robust, double usign, double vsign, uint32_t flags,
                           void* stream);

/*
 * Briggs / uniform weights of a batch of snapshots (`pfb hci`, utils/stokes2im.py:563-604).  Snapshot b owns the rows
 * [row_offsets[b], row_offsets[b+1]) of uvw (nrow,3), mask (nrow,nchan) u8 or NULL and wgt (nrow,nchan) of
 * `precision` (one correlation); freq (nchan) is shared.  Each snapshot gets its own (nx_pad, ny_pad) counts grid,
 * its own sums and ssq, so wgt ends as it would after, for every snapshot on its own,
 *     pfbg_counts(rows of b) -> counts_b;  pfbg_counts_to_weights(counts_b, rows of b, robust)
 * A snapshot without any counts (no rows, all flagged, all off the grid) keeps its weights.  wgt is updated in place;
 * counts (nbatch, nx_pad, ny_pad) of `precision` receives the re-weighted grids when not NULL.  row_offsets is a host
 * array whatever `flags` says; it must rise monotonically from 0 to nrow.  Everything is checked before any launch.
 * Scratch held for the call: nbatch * nx_pad * ny_pad * sizeof(real) bytes of counts (2.1 GB for 256 snapshots on a
 * 1024^2 pad in fp64, 1.07 GB in fp32; none when `counts` is a device pointer), 24 B per snapshot and 4 B per row.
 */
int pfbg_counts_to_weights_batch(int32_t precision, int32_t device, int32_t nbatch, const int64_t* row_offsets,
                                 const double* uvw, const double* freq, const uint8_t* mask, void* wgt, int64_t nrow,
                                 int32_t nchan, int32_t nx_pad, int32_t ny_pad, double cell_x, double cell_y,
                                 double robust, double usign, double vsign, void* counts, uint32_t flags,
                                 void* stream);

/*
 * The same for the batch a plan holds (pfbg_plan_set_batch + pfbg_bind_vis_batch), on the device: wgt (nrow,nchan)
 * of the plan's precision is copied into the plan's bound weights and re-weighted there, per snapshot, from the
 * bound uvw, mask and rows; pfbg_grid / pfbg_degrid / pfbg_hessian with wgt == NULL then use them.  The cell of a
 * sample is the one pfbg_counts gives for freq when the bound fscale is the rounded quotient freq / c.  The plan keeps
 * nbatch * nx_pad * ny_pad * sizeof(real) + 24 nbatch bytes of counts scratch for the next call (2.1 GB for 256
 * snapshots on a 1024^2 pad in fp64, 1.07 GB in fp32).  PFBG_ERR_STATE for a plan without a bound batch.
 */
int pfbg_bind_weights_robust(pfbg_plan* plan, const void* wgt, int32_t nx_pad, int32_t ny_pad, double cell_x,
                             double cell_y, double robust, double usign, double vsign, uint32_t flags, void* stream);

/*
 * l2 (Student-t) re-weighting of the natural weights from residual visibilities — the block
 * `if l2_reweight_dof:` of image_data_products (operators/gridder.py:509-532):
 *     ressq = |resvis|^2 * wgtp;  ovar[c] = sum_{mask>0} ressq[c] / sum(mask);
 *     wgt[c] *= (dof + 2) / (dof + ressq[c] / ovar[c])          (every sample, flagged ones included)
 * resvis (ncorr,nrow,nchan) complex of `precision`, wgtp (ncorr,nrow,nchan) real or NULL (= 1),
 * mask (nrow,nchan) u8 or NULL, wgt (ncorr,nrow,nchan) real, updated in place.  ovar_out (ncorr doubles,
 * host) receives the per-correlation variance; when any of them is zero nothing is written to wgt and
 * *applied = 0 (the reference then sets the weights to None).
 */
int pfbg_l2_reweight(int32_t precision, int32_t device, const void* resvis, const void* wgtp,
                     const uint8_t* mask, void* wgt, int64_t nvis, int32_t ncorr, double dof,
                     double* ovar_out, int32_t* applied, uint32_t flags, void* stream);

/*
 * PSF-convolution Hessian on the device (SURVEY §8 f1; operators/hessian.py:103-143 hessian_psf_slice,
 * operators/psf.py:8-31 psf_convolve_slice):
 *     out = beam * crop( IFFT( FFT( pad(beam * x) ) * khat ) ) + eta * x
 * x, beam, out: (nx,ny) real of `precision`; khat: complex of `precision`, either the r2c half spectrum
 * (nx_psf, ny_psf/2+1) of a real kernel (PSFHAT / abspsf) or the full (nx_psf, ny_psf) spectrum.
 * Padded sizes may contain the factors 2, 3, 5, 7, 11 (ducc0.fft.good_size).
 */
typedef struct pfbg_conv pfbg_conv;
int pfbg_conv_create(int32_t precision, int32_t device, int32_t nx, int32_t ny, int32_t nx_psf, int32_t ny_psf,
                     pfbg_conv** out);
int pfbg_conv_destroy(pfbg_conv* conv);
int pfbg_conv_set_kernel(pfbg_conv* conv, const void* khat, int32_t half, uint32_t flags, void* stream);
int pfbg_conv_apply(pfbg_conv* conv, const void* x, const void* beam, double eta, void* out, uint32_t flags,
                    void* stream);
/* Read-only: the column-block width C (1, 2 or 4 columns per CTA of the column pass) and the CTA size of the
 * row passes that this convolver runs with.  Either output pointer may be NULL. */
int pfbg_conv_info(const pfbg_conv* conv, int32_t* col_block, int32_t* row_threads);
/*
 * Analytic kernel (`pfb restore`): the multiplier becomes the DFT on the padded grid of the periodised, pixel-sampled
 * Gaussian g(x, y) = exp(-4 ln 2 (x'^2 / emaj^2 + y'^2 / emin^2)), (x', y') the pixel offsets rotated by pa, evaluated
 * inside the column pass (no spectrum is stored).  Beams are (emaj, emin, pa): FWHMs in pixels, emaj >= emin >= 1,
 * the major axis along (cos pa, sin pa) in the (axis 0, axis 1) plane.  from == NULL: convolution with `to`; else the
 * ratio K_to / K_from that takes an image at resolution `from` to resolution `to`, which needs S_to - S_from positive
 * semi-definite (S the beam covariances).  The alias sums keep every term above 1e-18 of the peak (plain) or of the
 * largest term of each sum (ratio).  norm_kernel != 0: unit-sum kernels, else peak 1.  PFBG_ERR_ARG for a beam below
 * 1 px, emaj < emin, a `to` that does not contain `from`, or (ratio only) an axis ratio above about 30.
 * pfbg_conv_set_kernel switches back; the stored spectrum is allocated by set_kernel (so an out-of-memory failure
 * shows there, and leaves the previous kernel in place) and released here, after a device synchronisation.
 */
int pfbg_conv_set_gauss(pfbg_conv* conv, const double to[3], const double from[3], int32_t norm_kernel);
/* out = crop(IFFT(FFT(pad(x)) * K)) + add, the sum taken in the row epilogue; pointers as in pfbg_conv_apply.  With
 * PFBG_DEVICE_PTRS, `add` must not alias `out` (host pointers are staged, so there they may). */
int pfbg_conv_apply_add(pfbg_conv* conv, const void* x, const void* add, void* out, uint32_t flags, void* stream);
/*
 * Direct inverse of the Hessian (operators/hessian.py:213-248 hess_direct_slice) from the stored spectrum, fp64 only:
 *     out = taper * crop( IFFT( FFT( pad(taper * x) ) * (Re khat + c)^s ) ),   s = -1 if inverse else +1
 * taper may be NULL; no ridge term.  Re khat + c and its reciprocal are formed in fp64 with IEEE division, so the
 * output equals that of a convolver whose kernel was set to those doubles.  Pointers as in pfbg_conv_apply.
 * PFBG_ERR_STATE for a convolver without a stored spectrum (no kernel, or pfbg_conv_set_gauss).
 */
int pfbg_conv_apply_shifted(pfbg_conv* conv, const void* x, const void* taper, double c, int32_t inverse, void* out,
                            uint32_t flags, void* stream);
/*
 * One term of a sum-over-partitions Hessian (operators/hessian.py:439-522 HessianTree), device arrays only:
 *     out = scale * beam * crop( IFFT( FFT( pad(beam * x) ) * K ) ) + eta * xin
 * beam may be NULL; xin is not read when eta == 0 (it may then be NULL).  The epilogue multiplies by
 * scale / (nx_psf * ny_psf), so scale = 1 and xin = x give the bits of pfbg_conv_apply.  A sum over groups accumulates
 * through xin with eta = 1, ping-ponging between two buffers: xin must not alias out.  `flags` must hold
 * PFBG_DEVICE_PTRS; PFBG_ERR_ARG for host pointers, pointers on another device, or a scale that is not finite and > 0.
 */
int pfbg_conv_apply_scaled(pfbg_conv* conv, const void* x, const void* beam, const void* xin, double eta, double scale,
                           void* out, uint32_t flags, void* stream);

/*
 * Band split across two GPUs, one process per GPU (SURVEY §8e; the reference runs one actor per band,
 * operators/band_worker.py:217-246, and sums row partitions by linearity, operators/gridder.py:962-1016,
 * tests/test_imager_pass2.py:45-63).  When a job has as many bands as GPUs the heaviest band bounds the step, so
 * its owner hands the plane transforms of the LAST nq w-planes to a helper GPU.  The transfers are fused into the
 * transform kernels: the helper's forward column pass stores into the owner's peer-mapped plane stack, its inverse
 * column pass loads the gridded columns from there, and its fp64 partial image reaches the owner by one peer
 * copy.  Flags in device memory order the two streams; no host round trip, no collective.
 *
 * Set-up: owner  pfbg_split_owner_init(plan, nq, blobs[4])      -> ship blobs + plan desc + active window (host side)
 *         helper pfbg_split_helper_create(desc, nq, window, blobs, &hplan, &mailbox_blob) -> ship mailbox_blob back
 *         owner  pfbg_split_owner_connect(plan, &mailbox_blob)
 * Per apply: owner pfbg_hessian(plan, ..., PFBG_DEVICE_PTRS, stream); helper pfbg_split_helper_serve(hplan, stream),
 * once per owner call and in the same order.  A flag wait gives up after 20 s (pfbg_split_status reports it).
 */
#define PFBG_IPC_BLOB_BYTES 96
typedef struct pfbg_ipc_blob { unsigned char bytes[PFBG_IPC_BLOB_BYTES]; } pfbg_ipc_blob;
int pfbg_ipc_export(const void* dev_ptr, pfbg_ipc_blob* blob);
int pfbg_ipc_open(int32_t device, const pfbg_ipc_blob* blob, void** dev_ptr);
int pfbg_ipc_close_all(void);
int pfbg_split_owner_init(pfbg_plan* plan, int32_t nq, pfbg_ipc_blob* blobs4);
int pfbg_split_owner_connect(pfbg_plan* plan, const pfbg_ipc_blob* helper_mailbox);
/* window4 = {a_lo, a_len, b_lo, b_len}: the owner's active uv window (pfbg_plan_get_window) */
int pfbg_split_helper_create(const pfbg_plan_desc* desc, int32_t nq, const int32_t* window4,
                             const pfbg_ipc_blob* owner_blobs4, pfbg_plan** out, pfbg_ipc_blob* mailbox_out);
int pfbg_split_helper_serve(pfbg_plan* plan, void* stream);
int pfbg_split_status(pfbg_plan* plan, void* stream, int32_t* timed_out);
int pfbg_split_end(pfbg_plan* plan);
/* rows [a_lo, a_lo + a_len) x columns [b_lo, b_lo + b_len) (circular) of the grid any bound sample can touch */
int pfbg_plan_get_window(const pfbg_plan* plan, int32_t* window4);

/*
 * Visibilities and weights of one correlation behind diagonal Jones terms, as `pfb init` prepares them for the gridder.
 * Replaces: pfb_imaging.utils.correlations._weight_data_impl / wgt_func / vis_func
 * (src/pfb_imaging/utils/correlations.py:195-232):
 *   wgt[r, f] = Re(w0 gp gq conj(gp) conj(gq)),  vis[r, f] = w0 gq v0 conj(gp),
 *   gp = jones[row_t[r] * js_t + ant1[r] * js_a + f * js_c] (element strides of the complex Jones array), gq with ant2,
 *   (v0, w0) = correlation 0 of data / weight (nrow, nchan, ncorr).  row_t[r] < 0: the row is in no time bin and
 *   stays zero.  Products in the reference's order with every operation rounded separately: bit-identical to the
 *   numba loop.  The per-Stokes variant (utils/weighting.py:274-468) needs radiomesh's generated expressions and is
 *   not provided.  Host or device pointers (flags); host pointers: synchronous.
 */
int pfbg_weight_data_corr(int32_t precision, int32_t device, const void* data, const void* weight, const void* jones,
                          const int32_t* row_t, const int32_t* ant1, const int32_t* ant2, int64_t nrow, int32_t nchan,
                          int32_t ncorr, int64_t jones_elems, int64_t js_t, int64_t js_a, int64_t js_c, void* vis,
                          void* wgt, uint32_t flags, void* stream);

/*
 * Unit-test hook for the in-shared-memory FFT engine behind the fused plane transforms:
 * `batch` transforms of length n (2^a 3^b 5^c 7^d 11^e), complex of `precision`, host pointers.
 * mode 0 = decimation in frequency, 1 = decimation in time; inverse != 0 -> e^{+2 pi i nk/n}.
 */
int pfbg_debug_fft1d(int32_t precision, int32_t device, int32_t n, int32_t batch, const void* in,
                     void* out, int32_t mode, int32_t inverse);

/*
 * Unit-test hook for the fp64 exponential-of-semicircle tap of the DMMA run kernels (csrc/runs_mma.cuh):
 * out[i] = exp(beta (sqrt(1 - x[i]^2) - 1)) for n host values x in [-1, 1], evaluated by the kernels' own lean
 * exp / rsqrt (the quantity ducc0 tabulates by piecewise polynomials; tests compare with numpy).
 */
int pfbg_debug_es_fast64(int32_t device, int64_t n, const double* x, double beta, double* out);

/*
 * Unit-test hook for the fp32 pair engine (csrc/fft2.cuh) behind the TMA-fed column transforms: `batch` groups of
 * 2 np interleaved transforms of length n, in / out (batch, 2 np, n) complex64 on the host.  aos != 0: the first
 * stage reads the array-of-structures order the TMA unit delivers.
 */
int pfbg_debug_fft2(int32_t device, int32_t n, int32_t np, int32_t batch, const void* in, void* out,
                    int32_t inverse, int32_t aos);

#ifdef __cplusplus
}
#endif
#endif /* PFBGRID_H */
