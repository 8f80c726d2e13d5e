// PSF-convolution Hessian (psfconv.cuh): the convolver object, its tables and the pfbg_conv_* entry points of the
// C ABI (include/pfbgrid.h).
#include <algorithm>
#include <cmath>

#include "fft_host.h"
#include "host.h"
#include "psfconv.cuh"

struct pfbg_conv {
  int precision = 0, device = 0;
  ConvTabs ct{};
  int col_c = 1;
  void *tw_u = nullptr, *tw_v = nullptr, *rev_u = nullptr, *rev_v = nullptr, *pos_v = nullptr;
  void *khat = nullptr, *tmp = nullptr, *d_x = nullptr, *d_beam = nullptr, *d_out = nullptr;
  bool has_kernel = false;
  bool gauss = false;  // pfbg_conv_set_gauss: the analytic multiplier `gm`, no stored spectrum
  GaussMul gm{};
};

template <typename T>
static int conv_setup_t(pfbg_conv* cv) {
  const ConvTabs& c0 = cv->ct;
  FftDesc du, dv;
  if (!factorize(c0.nxp, du, sizeof(T) == 4 ? 16 : 8) || !factorize(c0.nyp, dv, sizeof(T) == 4 ? 16 : 8))
    return fail(PFBG_ERR_ARG, "padded sizes %d x %d must be 2^a 3^b 5^c 7^d 11^e", c0.nxp, c0.nyp);
  if (fft_smem_bytes<T>(c0.nyp) > kMaxSmem) return fail(PFBG_ERR_ARG, "ny_psf=%d too large for the shared-memory FFT", c0.nyp);
  int cc = (int)(32 / sizeof(cx2<T>));
  while (cc > 1 && (c0.nyp % cc || fft_smem_bytes<T>(c0.nxp * cc) > kMaxSmem)) cc /= 2;
  if (fft_smem_bytes<T>(c0.nxp * cc) > kMaxSmem) return fail(PFBG_ERR_ARG, "nx_psf=%d too large for the shared-memory FFT", c0.nxp);
  cv->col_c = cc;
  auto up = [&](void** dst, const void* src, size_t bytes) -> int {
    CK(cudaMalloc(dst, bytes));
    CK(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return PFBG_OK;
  };
  std::vector<int> rev, pos;
  const std::vector<cx2<T>> tw_u = twiddles<T>(c0.nxp), tw_v = twiddles<T>(c0.nyp);
  CKRC(up(&cv->tw_u, tw_u.data(), tw_u.size() * sizeof(cx2<T>)));
  CKRC(up(&cv->tw_v, tw_v.data(), tw_v.size() * sizeof(cx2<T>)));
  digit_tables(du, rev, pos);
  CKRC(up(&cv->rev_u, rev.data(), rev.size() * 4));
  digit_tables(dv, rev, pos);
  CKRC(up(&cv->rev_v, rev.data(), rev.size() * 4));
  CKRC(up(&cv->pos_v, pos.data(), pos.size() * 4));
  const size_t rb = sizeof(T);
  CK(cudaMalloc(&cv->tmp, (size_t)c0.nx * c0.nyp * 2 * rb));
  CK(cudaMalloc(&cv->d_x, (size_t)c0.nx * c0.ny * rb));
  CK(cudaMalloc(&cv->d_beam, (size_t)c0.nx * c0.ny * rb));
  CK(cudaMalloc(&cv->d_out, (size_t)c0.nx * c0.ny * rb));
  ConvTabs& ct = cv->ct;
  ct.du = du; ct.dv = dv;
  ct.tw_u = cv->tw_u; ct.tw_v = cv->tw_v;
  ct.rev_u = (const int*)cv->rev_u; ct.rev_v = (const int*)cv->rev_v; ct.pos_v = (const int*)cv->pos_v;
  CK(cudaFuncSetAttribute(k_conv_rows_fwd<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_rows_inv<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_cols<T, 4, KhatMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_cols<T, 2, KhatMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_cols<T, 1, KhatMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_cols<T, 4, GaussMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_cols<T, 2, GaussMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_conv_cols<T, 1, GaussMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  if constexpr (sizeof(T) == 8) {  // pfbg_conv_apply_shifted is fp64 only
    CK(cudaFuncSetAttribute(k_conv_cols<T, 4, ShiftMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CK(cudaFuncSetAttribute(k_conv_cols<T, 2, ShiftMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CK(cudaFuncSetAttribute(k_conv_cols<T, 1, ShiftMul>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  }
  return PFBG_OK;
}

extern "C" int pfbg_conv_destroy(pfbg_conv* cv) {
  if (!cv) return PFBG_OK;
  cudaSetDevice(cv->device);
  void* all[] = {cv->tw_u, cv->tw_v, cv->rev_u, cv->rev_v, cv->pos_v, cv->khat, cv->tmp, cv->d_x, cv->d_beam, cv->d_out};
  for (void* p : all)
    if (p) cudaFree(p);
  delete cv;
  return PFBG_OK;
}

extern "C" int pfbg_conv_create(int32_t precision, int32_t device, int32_t nx, int32_t ny, int32_t nx_psf,
                                int32_t ny_psf, pfbg_conv** out) {
  if (!out) return fail(PFBG_ERR_ARG, "null argument");
  *out = nullptr;
  if (precision != PFBG_F32 && precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  if (nx <= 0 || ny <= 0 || nx_psf < nx || ny_psf < ny) return fail(PFBG_ERR_ARG, "need 0 < nx <= nx_psf and 0 < ny <= ny_psf");
  CK(cudaSetDevice(device));
  pfbg_conv* cv = new pfbg_conv();
  cv->precision = precision; cv->device = device;
  cv->ct.nx = nx; cv->ct.ny = ny; cv->ct.nxp = nx_psf; cv->ct.nyp = ny_psf;
  int rc = precision == PFBG_F32 ? conv_setup_t<float>(cv) : conv_setup_t<double>(cv);
  if (rc) { pfbg_conv_destroy(cv); return rc; }
  *out = cv;
  return PFBG_OK;
}

// the column-block width and the row-pass CTA size conv_setup_t / conv_apply_t chose (read-only, for tests)
extern "C" int pfbg_conv_info(const pfbg_conv* cv, int32_t* col_block, int32_t* row_threads_out) {
  if (!cv) return fail(PFBG_ERR_ARG, "null argument");
  if (col_block) *col_block = cv->col_c;
  if (row_threads_out) *row_threads_out = row_threads(cv->ct.nyp, 256);
  return PFBG_OK;
}

// khat: complex multiplier of `precision`; half != 0: (nx_psf, ny_psf/2+1) half spectrum of a real kernel
// (r2c layout: PSFHAT / abspsf), else the full (nx_psf, ny_psf) spectrum.
extern "C" int pfbg_conv_set_kernel(pfbg_conv* cv, const void* khat, int32_t half, uint32_t flags, void* stream) {
  if (!cv || !khat) return fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(cv->device));
  cudaStream_t s = (cudaStream_t)stream;
  const ConvTabs& ct = cv->ct;
  const size_t cb = cv->precision == PFBG_F32 ? 8 : 16;
  const cudaMemcpyKind kind = (flags & PFBG_DEVICE_PTRS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  // the spectrum is allocated here, not at creation: a convolver that only ever runs the analytic kernel never holds it
  // (an out-of-memory failure therefore shows here, not at pfbg_conv_create; the previous kernel is kept)
  if (!cv->khat) CK(cudaMalloc(&cv->khat, (size_t)ct.nxp * ct.nyp * cb));
  if (!half) {
    // keep the Hermitian part only (all a real image can see; the column stage evaluates half the columns)
    const size_t fb = (size_t)ct.nxp * ct.nyp * cb;
    void* df = nullptr;
    CK(cudaMalloc(&df, fb));
    cudaError_t e = cudaMemcpyAsync(df, khat, fb, kind, s);
    if (e == cudaSuccess) {
      dim3 grd((ct.nyp + 127) / 128, ct.nxp);
      if (cv->precision == PFBG_F32) k_hermitize<float><<<grd, 128, 0, s>>>(ct.nxp, ct.nyp, (const cx2<float>*)df, (cx2<float>*)cv->khat);
      else k_hermitize<double><<<grd, 128, 0, s>>>(ct.nxp, ct.nyp, (const cx2<double>*)df, (cx2<double>*)cv->khat);
      LAUNCHED();
      e = cudaStreamSynchronize(s);
    }
    cudaFree(df);
    if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "set_kernel failed: %s", cudaGetErrorString(e));
  } else {
    const size_t hb = (size_t)ct.nxp * (ct.nyp / 2 + 1) * cb;
    void* dh = nullptr;
    CK(cudaMalloc(&dh, hb));
    cudaError_t e = cudaMemcpyAsync(dh, khat, hb, kind, s);
    if (e == cudaSuccess) {
      dim3 grd((ct.nyp + 127) / 128, ct.nxp);
      if (cv->precision == PFBG_F32) k_expand_half<float><<<grd, 128, 0, s>>>(ct.nxp, ct.nyp, (const cx2<float>*)dh, (cx2<float>*)cv->khat);
      else k_expand_half<double><<<grd, 128, 0, s>>>(ct.nxp, ct.nyp, (const cx2<double>*)dh, (cx2<double>*)cv->khat);
      LAUNCHED();
      e = cudaStreamSynchronize(s);
    }
    cudaFree(dh);
    if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "set_kernel failed: %s", cudaGetErrorString(e));
  }
  CK(cudaStreamSynchronize(s));
  cv->gauss = false;
  cv->has_kernel = true;
  return PFBG_OK;
}

// Beam (emaj, emin, pa) in pixels -> covariance S of exp(-x^T S^-1 x / 2); emaj, emin are FWHMs, the major axis points
// along (cos pa, sin pa) in the (axis 0, axis 1) plane.
static int gauss_cov(const double* b, const char* which, double S[3]) {
  const double emaj = b[0], emin = b[1], pa = b[2];
  if (!std::isfinite(emaj) || !std::isfinite(emin) || !std::isfinite(pa))
    return fail(PFBG_ERR_ARG, "%s beam is not finite", which);
  if (emin < 1.0) return fail(PFBG_ERR_ARG, "%s beam FWHM %g px is below 1 pixel", which, emin);
  if (emaj < emin) return fail(PFBG_ERR_ARG, "%s beam has emaj %g < emin %g", which, emaj, emin);
  const double k = 1.0 / (8.0 * M_LN2);  // sigma^2 = FWHM^2 / (8 ln 2)
  const double va = emaj * emaj * k, vb = emin * emin * k, c = cos(pa), sn = sin(pa);
  S[0] = va * c * c + vb * sn * sn;
  S[1] = (va - vb) * c * sn;
  S[2] = va * sn * sn + vb * c * c;
  return PFBG_OK;
}

static double sym2_min_eig(const double S[3]) {
  const double m = 0.5 * (S[0] + S[2]), d = hypot(0.5 * (S[0] - S[2]), S[1]);
  return m - d;
}

// Alias count of one sum of the ratio mode, where each sum must be accurate relative to its own largest term (the
// quotient divides the scale out), not to the peak at f = 0.  With m = 0 as the reference kept term, a dropped term m
// is small enough at every f of the zone [-1/2, 1/2]^2 when
//     (f + m)^T S (f + m) - f^T S f = m^T S m + 2 m^T S f >= m^T S m - |S m|_1 >= c,   c = -ln(1e-18) / (2 pi^2),
// so M is the largest |m|_inf of any m that fails this.  Outside |m|_inf <= r0, m^T S m >= lmin r^2 and
// |S m|_1 <= 2 lmax r make every m pass.  Returns -1 when r0 exceeds kMaxAliasScan (beams with an axis ratio above ~30).
static constexpr int kMaxAliasScan = 2048;
static int ratio_alias_M(const double S[3], double c) {
  const double lmin = sym2_min_eig(S), lmax = S[0] + S[2] - lmin;
  const double r0 = (lmax + sqrt(lmax * lmax + lmin * c)) / lmin;
  if (!(r0 <= kMaxAliasScan)) return -1;
  const int R = (int)ceil(r0);
  int M = 0;
  for (int mx = -R; mx <= R; ++mx)
    for (int my = -R; my <= R; ++my) {
      const double sx = S[0] * mx + S[1] * my, sy = S[1] * mx + S[2] * my;
      if (mx * sx + my * sy - fabs(sx) - fabs(sy) < c) M = std::max(M, std::max(std::abs(mx), std::abs(my)));
    }
  return M;
}

// the alias sum of GaussMul at f = 0 (host), for the unit-sum normalisation
static double gauss_sum0(const double q[3], int M) {
  double acc = 0.0;
  for (int mx = -M; mx <= M; ++mx)
    for (int my = -M; my <= M; ++my) acc += exp(q[0] * mx * mx + q[1] * mx * my + q[2] * my * my);
  return acc;
}

// to, from: (emaj, emin, pa) in pixels; from == NULL: plain convolution with the `to` Gaussian, else the ratio
// K_to / K_from.  norm_kernel != 0: unit sum, else peak 1 (for a ratio, both kernels are normalised the same way).
extern "C" int pfbg_conv_set_gauss(pfbg_conv* cv, const double* to, const double* from, int32_t norm_kernel) {
  if (!cv || !to) return fail(PFBG_ERR_ARG, "null argument");
  double St[3], Sf[3];
  CKRC(gauss_cov(to, "target", St));
  if (from) {
    CKRC(gauss_cov(from, "source", Sf));
    // converting to a narrower (or differently shaped) beam would divide by a vanishing transfer function
    const double D[3] = {St[0] - Sf[0], St[1] - Sf[1], St[2] - Sf[2]};
    const double tol = 1e-9 * fmax(St[0] + St[2], Sf[0] + Sf[2]);
    if (sym2_min_eig(D) < -tol)
      return fail(PFBG_ERR_ARG, "target beam (%g, %g, %g) does not contain source beam (%g, %g, %g): S_to - S_from "
                  "is not positive semi-definite", to[0], to[1], to[2], from[0], from[1], from[2]);
  }
  GaussMul g{};
  const double cdrop = -log(1e-18) / (2.0 * M_PI * M_PI);
  if (!from) {
    // plain: an absolute bound suffices.  The dropped alias terms have |f + m| >= M + 1/2, so
    // q <= -2 pi^2 lmin (M + 1/2)^2, below 1e-18 of the peak when that is <= ln(1e-18) (M = 3 at a 1 px FWHM)
    const double need = sqrt(cdrop / sym2_min_eig(St)) - 0.5;
    g.M = need <= 0.0 ? 0 : (int)ceil(need);
  } else {
    const int mt = ratio_alias_M(St, cdrop), mf = ratio_alias_M(Sf, cdrop);
    if (mt < 0 || mf < 0)
      return fail(PFBG_ERR_ARG, "beam axis ratio too large for a change of resolution (alias scan beyond %d)",
                  kMaxAliasScan);
    g.M = std::max(mt, mf);
  }
  g.ratio = from != nullptr;
  const double c2 = -2.0 * M_PI * M_PI;
  const double qt[3] = {c2 * St[0], 2.0 * c2 * St[1], c2 * St[2]};
  for (int i = 0; i < 3; ++i) g.q_to[i] = qt[i];
  auto amp_of = [&](const double* S, const double* q) {
    return norm_kernel ? 1.0 / gauss_sum0(q, g.M) : 2.0 * M_PI * sqrt(S[0] * S[2] - S[1] * S[1]);
  };
  g.amp = amp_of(St, qt);
  if (from) {
    const double qf[3] = {c2 * Sf[0], 2.0 * c2 * Sf[1], c2 * Sf[2]};
    for (int i = 0; i < 3; ++i) g.q_from[i] = qf[i];
    g.amp /= amp_of(Sf, qf);
  }
  if (cv->khat) {  // a Gaussian-mode convolver holds no spectrum
    CK(cudaSetDevice(cv->device));
    // an apply still in flight on any stream may read it.  set_gauss takes no stream, and cudaFree synchronises the
    // device anyway; this happens once per switch from a stored spectrum, never between bands of a Gaussian run.
    CK(cudaDeviceSynchronize());
    cudaFree(cv->khat);
    cv->khat = nullptr;
  }
  cv->gm = g;
  cv->gauss = true;
  cv->has_kernel = true;
  return PFBG_OK;
}

template <typename T, class Mul>
static void conv_cols_launch(const pfbg_conv* cv, const Mul& mul, cudaStream_t s) {
  const ConvTabs& ct = cv->ct;
  const int cc = cv->col_c;
  const size_t csm = fft_smem_bytes<T>(ct.nxp * cc);
  // Hermitian symmetry (real image, real kernel): only the columns l <= nyp/2 are transformed (psfconv.cuh)
  const int ncol = ct.nyp / 2 + 1;
  const cx2<T>* kh = (const cx2<T>*)cv->khat;
  cx2<T>* tmp = (cx2<T>*)cv->tmp;
  if (cc == 4) k_conv_cols<T, 4, Mul><<<(ncol + 3) / 4, 512, csm, s>>>(ct, kh, tmp, mul);
  else if (cc == 2) k_conv_cols<T, 2, Mul><<<(ncol + 1) / 2, 512, csm, s>>>(ct, kh, tmp, mul);
  else k_conv_cols<T, 1, Mul><<<ncol, 512, csm, s>>>(ct, kh, tmp, mul);
}

// xin != NULL: out += eta * xin in the row epilogue (the ridge term of the Hessian, or eta = 1 for apply_add).
// shift != NULL (fp64, stored spectrum): the column pass multiplies by ShiftMul instead of the convolver's own kernel.
// scale multiplies the convolution term: the epilogue factor is scale / (nxp nyp), the same double as 1 / (nxp nyp) at
// scale = 1.
template <typename T>
static int conv_apply_t(pfbg_conv* cv, const void* x, const void* beam, const void* xin, double eta, void* out,
                        cudaStream_t s, const ShiftMul* shift, double scale) {
  const ConvTabs& ct = cv->ct;
  const int rt = row_threads(ct.nyp, 256);
  k_conv_rows_fwd<T><<<(ct.nx + 1) / 2, rt, fft_smem_bytes<T>(ct.nyp), s>>>(ct, (const T*)x, (const T*)beam, (cx2<T>*)cv->tmp);
  LAUNCHED();
  if constexpr (sizeof(T) == 8) {
    if (shift) conv_cols_launch<T>(cv, *shift, s);
    else if (cv->gauss) conv_cols_launch<T>(cv, cv->gm, s);
    else conv_cols_launch<T>(cv, KhatMul{}, s);
  } else {
    if (cv->gauss) conv_cols_launch<T>(cv, cv->gm, s);
    else conv_cols_launch<T>(cv, KhatMul{}, s);
  }
  LAUNCHED();
  const double escale = scale / ((double)ct.nxp * (double)ct.nyp);
  k_conv_rows_inv<T><<<(ct.nx + 1) / 2, rt, fft_smem_bytes<T>(ct.nyp), s>>>(ct, (const cx2<T>*)cv->tmp, (const T*)beam,
                                                                 (const T*)xin, escale, eta, (T*)out);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

// out = beam * crop(IFFT(FFT(pad(beam * x)) * K)) + eta * xin; host pointers are staged through d_x / d_beam / d_out
// (apply_add passes no beam, so its `add` image rides in d_beam)
static int conv_apply_any(pfbg_conv* cv, const void* x, const void* beam, const void* xin, double eta, void* out,
                          uint32_t flags, void* stream, const ShiftMul* shift = nullptr, double scale = 1.0) {
  if (!cv || !x || !out) return fail(PFBG_ERR_ARG, "null argument");
  if (!cv->has_kernel) return fail(PFBG_ERR_STATE, "no kernel set");
  CK(cudaSetDevice(cv->device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t ib = (size_t)cv->ct.nx * cv->ct.ny * (cv->precision == PFBG_F32 ? 4 : 8);
  const void *dx = x, *db = beam, *dxin = xin;
  void* dout = out;
  if (!dev) {
    CK(cudaMemcpyAsync(cv->d_x, x, ib, cudaMemcpyHostToDevice, s));
    dx = cv->d_x;
    if (beam) { CK(cudaMemcpyAsync(cv->d_beam, beam, ib, cudaMemcpyHostToDevice, s)); db = cv->d_beam; }
    if (xin == x) dxin = dx;
    else if (xin) { CK(cudaMemcpyAsync(cv->d_beam, xin, ib, cudaMemcpyHostToDevice, s)); dxin = cv->d_beam; }
    dout = cv->d_out;
  }
  CKRC(cv->precision == PFBG_F32 ? conv_apply_t<float>(cv, dx, db, dxin, eta, dout, s, nullptr, scale)
                                 : conv_apply_t<double>(cv, dx, db, dxin, eta, dout, s, shift, scale));
  if (!dev) {
    CK(cudaMemcpyAsync(out, dout, ib, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  return PFBG_OK;
}

// out = beam * crop(IFFT(FFT(pad(beam * x)) * khat)) + eta * x      (beam may be NULL)
extern "C" int pfbg_conv_apply(pfbg_conv* cv, const void* x, const void* beam, double eta, void* out, uint32_t flags,
                               void* stream) {
  return conv_apply_any(cv, x, beam, eta != 0.0 ? x : nullptr, eta, out, flags, stream);
}

// out = crop(IFFT(FFT(pad(x)) * K)) + add, the add in the row epilogue (x + 1.0 * add rounds as the separate sum)
extern "C" int pfbg_conv_apply_add(pfbg_conv* cv, const void* x, const void* add, void* out, uint32_t flags,
                                   void* stream) {
  if (!add) return fail(PFBG_ERR_ARG, "null argument");
  return conv_apply_any(cv, x, nullptr, add, 1.0, out, flags, stream);
}

// a device array on `device` (or managed memory)
bool pfbg_on_device(const void* p, int device) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == device;
}

// the unchecked device-pointer body of pfbg_conv_apply_scaled, for the batched solvers (xin is ignored when eta == 0)
int pfbg_conv_apply_dev(pfbg_conv* cv, const void* x, const void* beam, const void* xin, double eta, double scale,
                        void* out, void* stream) {
  return conv_apply_any(cv, x, beam, eta != 0.0 ? xin : nullptr, eta, out, PFBG_DEVICE_PTRS, stream, nullptr, scale);
}

// out = scale * beam * crop(IFFT(FFT(pad(beam * x)) * K)) + eta * xin, device arrays only
extern "C" int pfbg_conv_apply_scaled(pfbg_conv* cv, const void* x, const void* beam, const void* xin, double eta,
                                      double scale, void* out, uint32_t flags, void* stream) {
  if (!cv || !x || !out || (eta != 0.0 && !xin)) return fail(PFBG_ERR_ARG, "null argument");
  if (!(flags & PFBG_DEVICE_PTRS)) return fail(PFBG_ERR_ARG, "pfbg_conv_apply_scaled takes device pointers only");
  if (!(scale > 0.0) || !std::isfinite(scale)) return fail(PFBG_ERR_ARG, "scale %g must be finite and > 0", scale);
  if (eta != 0.0 && xin == out) return fail(PFBG_ERR_ARG, "xin must not alias out (accumulate through a second buffer)");
  CK(cudaSetDevice(cv->device));
  const void* ptrs[] = {x, beam, eta != 0.0 ? xin : nullptr, out};
  for (const void* p : ptrs)
    if (p && !pfbg_on_device(p, cv->device))
      return fail(PFBG_ERR_ARG, "x, beam, xin and out must be device arrays on device %d", cv->device);
  return pfbg_conv_apply_dev(cv, x, beam, xin, eta, scale, out, stream);
}

// out = taper * crop(IFFT(FFT(pad(taper * x)) * (Re khat + c)^(+-1)))   (taper may be NULL; no ridge term)
extern "C" int pfbg_conv_apply_shifted(pfbg_conv* cv, const void* x, const void* taper, double c, int32_t inverse,
                                       void* out, uint32_t flags, void* stream) {
  if (!cv || !x || !out) return fail(PFBG_ERR_ARG, "null argument");
  if (cv->precision != PFBG_F64) return fail(PFBG_ERR_ARG, "the shifted spectrum is fp64 only");
  if (!cv->has_kernel || cv->gauss || !cv->khat)
    return fail(PFBG_ERR_STATE, "the shifted spectrum needs a stored spectrum (pfbg_conv_set_kernel)");
  const ShiftMul sh{c, inverse ? 1 : 0};
  return conv_apply_any(cv, x, taper, nullptr, 0.0, out, flags, stream, &sh);
}

// what the batched solvers of pfbsara.cu check before borrowing a convolver (not part of the C ABI)
int pfbg_conv_props(const pfbg_conv* cv, int* precision, int* device, int* nx, int* ny, int* has_kernel) {
  if (!cv) return fail(PFBG_ERR_ARG, "null convolver");
  *precision = cv->precision; *device = cv->device; *nx = cv->ct.nx; *ny = cv->ct.ny; *has_kernel = cv->has_kernel;
  return PFBG_OK;
}
