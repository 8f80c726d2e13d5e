// C-ABI of the device backward steps (include/pfbsara.h): SARA (kernels in sara.cuh), the Clark minor cycle
// (clean.cuh) and the batched conjugate gradients of HessPSF.idot and HessianTree (cg.cuh).
#include <cuda_runtime.h>

#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cub/device/device_select.cuh>
#include <vector>

#include "../../include/pfbsara.h"
#include "cg.cuh"
#include "clean.cuh"
#include "host.h"
#include "sara.cuh"

struct pfbs_psi {
  int precision = 0, device = 0;
  int nband = 0, nx = 0, ny = 0, nbasis = 0, nlevel = 0, nxmax = 0, nymax = 0;
  std::vector<int> K;
  std::vector<DwtFilt> dec, rec;
  std::vector<int64_t> ix, iy, sx, sy, spx, spy, ntotx, ntoty;
  void *approx[2] = {nullptr, nullptr};  // (nband, sx0max, sy0max) ping-pong: LL of the previous level
  void *img[2] = {nullptr, nullptr};     // (nband, nx+1, ny+1) ping-pong: inner reconstructions
  void *d_x = nullptr, *d_alpha = nullptr, *d_alpha_t = nullptr;  // staging for host-pointer / transposed calls
  size_t approx_elems = 0, img_elems = 0;
  int64_t L(const std::vector<int64_t>& a, int b, int l) const { return a[(size_t)b * nlevel + l]; }
};

static size_t rbytes(int precision) { return precision == PFBG_F32 ? 4 : 8; }

extern "C" int pfbs_psi_destroy(pfbs_psi* p) {
  if (!p) return PFBG_OK;
  cudaSetDevice(p->device);
  void* all[] = {p->approx[0], p->approx[1], p->img[0], p->img[1], p->d_x, p->d_alpha, p->d_alpha_t};
  for (void* q : all)
    if (q) cudaFree(q);
  delete p;
  return PFBG_OK;
}

extern "C" int pfbs_psi_create(int32_t precision, int32_t device, int32_t nband, int32_t nx, int32_t ny, int32_t nbasis,
                               int32_t nlevel, const int32_t* K, const double* filters, const int64_t* ix,
                               const int64_t* iy, const int64_t* sx, const int64_t* sy, const int64_t* spx,
                               const int64_t* spy, const int64_t* ntotx, const int64_t* ntoty, int32_t nxmax,
                               int32_t nymax, pfbs_psi** out) {
  if (!out || !K || !filters || !ix || !iy || !sx || !sy || !spx || !spy || !ntotx || !ntoty)
    return pfbg_fail(PFBG_ERR_ARG, "null argument");
  *out = nullptr;
  if (precision != PFBG_F32 && precision != PFBG_F64) return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  if (nband < 1 || nx < 1 || ny < 1 || nbasis < 1 || nlevel < 1 || nxmax < nx || nymax < ny)
    return pfbg_fail(PFBG_ERR_ARG, "bad sizes");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return pfbg_fail(PFBG_ERR_ARG, "device %d out of range", device);
  CK(cudaSetDevice(device));
  pfbs_psi* p = new pfbs_psi();
  p->precision = precision; p->device = device; p->nband = nband; p->nx = nx; p->ny = ny;
  p->nbasis = nbasis; p->nlevel = nlevel; p->nxmax = nxmax; p->nymax = nymax;
  p->K.assign(K, K + nbasis);
  p->dec.resize(nbasis); p->rec.resize(nbasis);
  const size_t nl = (size_t)nbasis * nlevel;
  p->ix.assign(ix, ix + 2 * nl); p->iy.assign(iy, iy + 2 * nl);
  p->sx.assign(sx, sx + nl); p->sy.assign(sy, sy + nl); p->spx.assign(spx, spx + nl); p->spy.assign(spy, spy + nl);
  p->ntotx.assign(ntotx, ntotx + nbasis); p->ntoty.assign(ntoty, ntoty + nbasis);
  size_t amax = 1;
  for (int b = 0; b < nbasis; ++b) {
    const int k = K[b];
    if (k == 0) continue;
    if (k < 2 || k > PFBS_KMAX || (k & 1)) { delete p; return pfbg_fail(PFBG_ERR_ARG, "filter length %d not in 2..%d (even)", k, PFBS_KMAX); }
    if (ntotx[b] > nxmax || ntoty[b] > nymax) { delete p; return pfbg_fail(PFBG_ERR_ARG, "basis %d does not fit (nxmax, nymax)", b); }
    const double* f = filters + (size_t)b * 4 * PFBS_KMAX;
    memset(&p->dec[b], 0, sizeof(DwtFilt)); memset(&p->rec[b], 0, sizeof(DwtFilt));
    p->dec[b].K = p->rec[b].K = k;
    for (int t = 0; t < k; ++t) {
      p->dec[b].lo[t] = f[t]; p->dec[b].hi[t] = f[PFBS_KMAX + t];
      p->rec[b].lo[t] = f[2 * PFBS_KMAX + t]; p->rec[b].hi[t] = f[3 * PFBS_KMAX + t];
    }
    for (int l = 0; l < nlevel; ++l) {
      const size_t a = (size_t)p->L(p->sx, b, l) * p->L(p->sy, b, l);
      if (a > amax) amax = a;
    }
  }
  const size_t rb = rbytes(precision);
  p->approx_elems = amax;
  p->img_elems = (size_t)(nx + 2) * (ny + 2);
  cudaError_t e = cudaSuccess;
  for (int t = 0; t < 2 && e == cudaSuccess; ++t) {
    e = cudaMalloc(&p->approx[t], (size_t)nband * p->approx_elems * rb);
    if (e == cudaSuccess) e = cudaMalloc(&p->img[t], (size_t)nband * p->img_elems * rb);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    pfbs_psi_destroy(p);
    return pfbg_fail(PFBG_ERR_NOMEM, "scratch allocation failed: %s", cudaGetErrorString(e));
  }
  *out = p;
  return PFBG_OK;
}

static int stage_alloc(void** buf, size_t bytes) {
  if (*buf) return PFBG_OK;
  cudaError_t e = cudaMalloc(buf, bytes);
  if (e != cudaSuccess) { *buf = nullptr; cudaGetLastError(); return pfbg_fail(PFBG_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); }
  return PFBG_OK;
}

template <typename T>
static int psi_dot_t(pfbs_psi* p, const T* x, T* alpha, cudaStream_t s) {
  const int64_t img = (int64_t)p->nx * p->ny, plane = (int64_t)p->nxmax * p->nymax;
  const int64_t astride = (int64_t)p->nbasis * plane;
  CK(cudaMemsetAsync(alpha, 0, (size_t)p->nband * astride * sizeof(T), s));
  for (int b = 0; b < p->nbasis; ++b) {
    T* ab = alpha + (int64_t)b * plane;
    if (p->K[b] == 0) {
      k_copy2d<T><<<dim3((p->ny + 127) / 128, p->nx, p->nband), 128, 0, s>>>(x, p->ny, img, ab, p->nymax, astride, p->nx, p->ny, 0);
      LAUNCHED();
      continue;
    }
    const T* in = x;
    int ld_in = p->ny, nxin = p->nx, nyin = p->ny;
    int64_t in_stride = img;
    for (int l = 0; l < p->nlevel; ++l) {
      const int sx = (int)p->L(p->sx, b, l), sy = (int)p->L(p->sy, b, l);
      const int hx = (int)p->ix[((size_t)b * p->nlevel + l) * 2 + 1], hy = (int)p->iy[((size_t)b * p->nlevel + l) * 2 + 1];
      const int lx = hx - 2 * sx, ly = hy - 2 * sy;
      T* ap = (l + 1 < p->nlevel) ? (T*)p->approx[l & 1] : nullptr;
      BandPtr bp{in_stride, astride, (int64_t)p->approx_elems};
      dim3 grd((sy + SW_TY - 1) / SW_TY, (sx + SW_TX - 1) / SW_TX, p->nband);
      T* blk = ab + (int64_t)lx * p->nymax + ly;
      switch (p->K[b]) {
        case 2: k_dwt_level<T, 2><<<grd, 256, 0, s>>>(in, ld_in, nxin, nyin, blk, p->nymax, sx, sy, ap, p->dec[b], bp); break;
        case 4: k_dwt_level<T, 4><<<grd, 256, 0, s>>>(in, ld_in, nxin, nyin, blk, p->nymax, sx, sy, ap, p->dec[b], bp); break;
        case 6: k_dwt_level<T, 6><<<grd, 256, 0, s>>>(in, ld_in, nxin, nyin, blk, p->nymax, sx, sy, ap, p->dec[b], bp); break;
        case 8: k_dwt_level<T, 8><<<grd, 256, 0, s>>>(in, ld_in, nxin, nyin, blk, p->nymax, sx, sy, ap, p->dec[b], bp); break;
        default: k_dwt_level<T, 10><<<grd, 256, 0, s>>>(in, ld_in, nxin, nyin, blk, p->nymax, sx, sy, ap, p->dec[b], bp); break;
      }
      LAUNCHED();
      in = ap; ld_in = sy; nxin = sx; nyin = sy; in_stride = (int64_t)p->approx_elems;
    }
  }
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int psi_hdot_t(pfbs_psi* p, const T* alpha, T* x, cudaStream_t s) {
  const int64_t img = (int64_t)p->nx * p->ny, plane = (int64_t)p->nxmax * p->nymax;
  const int64_t astride = (int64_t)p->nbasis * plane;
  CK(cudaMemsetAsync(x, 0, (size_t)p->nband * img * sizeof(T), s));
  for (int b = 0; b < p->nbasis; ++b) {
    const T* ab = alpha + (int64_t)b * plane;
    if (p->K[b] == 0) {
      k_copy2d<T><<<dim3((p->ny + 127) / 128, p->nx, p->nband), 128, 0, s>>>(ab, p->nymax, astride, x, p->ny, img, p->nx, p->ny, 1);
      LAUNCHED();
      continue;
    }
    const T* ll = nullptr;  // LL source of the current level: the block's own quadrant at the deepest level
    int ld_ll = 0;
    int64_t ll_stride = 0;
    for (int l = p->nlevel - 1; l >= 0; --l) {
      const int sx = (int)p->L(p->sx, b, l), sy = (int)p->L(p->sy, b, l);
      const int hx = (int)p->ix[((size_t)b * p->nlevel + l) * 2 + 1], hy = (int)p->iy[((size_t)b * p->nlevel + l) * 2 + 1];
      const int lx = hx - 2 * sx, ly = hy - 2 * sy;
      const T* blk = ab + (int64_t)lx * p->nymax + ly;
      if (l == p->nlevel - 1) { ll = blk; ld_ll = p->nymax; ll_stride = astride; }
      int nxo = (int)p->L(p->spx, b, l), nyo = (int)p->L(p->spy, b, l);
      if (nxo > p->nx) nxo = p->nx;
      if (nyo > p->ny) nyo = p->ny;
      T* dst; int ld_dst; int64_t dst_stride; int acc;
      if (l == 0) { dst = x; ld_dst = p->ny; dst_stride = img; acc = 1; }
      else { dst = (T*)p->img[l & 1]; ld_dst = p->ny + 2; dst_stride = (int64_t)p->img_elems; acc = 0; }
      BandPtr bp{astride, dst_stride, ll_stride};
      dim3 grd(((nyo + 1) / 2 + SW_TY - 1) / SW_TY, ((nxo + 1) / 2 + SW_TX - 1) / SW_TX, p->nband);
      switch (p->K[b]) {
        case 2: k_idwt_level<T, 2><<<grd, 256, 0, s>>>(ll, ld_ll, blk, p->nymax, sx, sy, dst, ld_dst, nxo, nyo, p->rec[b], acc, bp); break;
        case 4: k_idwt_level<T, 4><<<grd, 256, 0, s>>>(ll, ld_ll, blk, p->nymax, sx, sy, dst, ld_dst, nxo, nyo, p->rec[b], acc, bp); break;
        case 6: k_idwt_level<T, 6><<<grd, 256, 0, s>>>(ll, ld_ll, blk, p->nymax, sx, sy, dst, ld_dst, nxo, nyo, p->rec[b], acc, bp); break;
        case 8: k_idwt_level<T, 8><<<grd, 256, 0, s>>>(ll, ld_ll, blk, p->nymax, sx, sy, dst, ld_dst, nxo, nyo, p->rec[b], acc, bp); break;
        default: k_idwt_level<T, 10><<<grd, 256, 0, s>>>(ll, ld_ll, blk, p->nymax, sx, sy, dst, ld_dst, nxo, nyo, p->rec[b], acc, bp); break;
      }
      LAUNCHED();
      ll = dst; ld_ll = ld_dst; ll_stride = dst_stride;
    }
  }
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int transpose_planes(const T* src, T* dst, int nplanes, int n0, int n1, cudaStream_t s) {
  for (int z0 = 0; z0 < nplanes; z0 += 65535) {
    const int nz = nplanes - z0 < 65535 ? nplanes - z0 : 65535;
    k_transpose<T><<<dim3((n1 + 31) / 32, (n0 + 31) / 32, nz), dim3(32, 8), 0, s>>>(src + (int64_t)z0 * n0 * n1, dst + (int64_t)z0 * n0 * n1, n0, n1);
    LAUNCHED();
  }
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int psi_apply(pfbs_psi* p, const void* in, void* out, uint32_t flags, cudaStream_t s, bool fwd) {
  const bool dev = flags & PFBG_DEVICE_PTRS, tr = flags & PFBS_TRANSPOSED;
  const size_t xb = (size_t)p->nband * p->nx * p->ny * sizeof(T);
  const size_t ab = (size_t)p->nband * p->nbasis * p->nxmax * p->nymax * sizeof(T);
  const int nplanes = p->nband * p->nbasis;
  if (fwd) {
    const T* dx = (const T*)in;
    if (!dev) { CKRC(stage_alloc(&p->d_x, xb)); CK(cudaMemcpyAsync(p->d_x, in, xb, cudaMemcpyHostToDevice, s)); dx = (const T*)p->d_x; }
    T* da = (T*)out;
    if (!dev || tr) { CKRC(stage_alloc(&p->d_alpha, ab)); da = (T*)p->d_alpha; }
    CKRC(psi_dot_t<T>(p, dx, da, s));
    if (tr) {
      T* dt = (T*)out;
      if (!dev) { CKRC(stage_alloc(&p->d_alpha_t, ab)); dt = (T*)p->d_alpha_t; }
      CKRC(transpose_planes<T>(da, dt, nplanes, p->nxmax, p->nymax, s));
      da = dt;
    }
    if (!dev) { CK(cudaMemcpyAsync(out, da, ab, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s)); }
  } else {
    const T* da = (const T*)in;
    if (!dev) { CKRC(stage_alloc(tr ? &p->d_alpha_t : &p->d_alpha, ab)); void* st = tr ? p->d_alpha_t : p->d_alpha; CK(cudaMemcpyAsync(st, in, ab, cudaMemcpyHostToDevice, s)); da = (const T*)st; }
    if (tr) {
      CKRC(stage_alloc(&p->d_alpha, ab));
      CKRC(transpose_planes<T>(da, (T*)p->d_alpha, nplanes, p->nymax, p->nxmax, s));
      da = (const T*)p->d_alpha;
    }
    T* dx = (T*)out;
    if (!dev) { CKRC(stage_alloc(&p->d_x, xb)); dx = (T*)p->d_x; }
    CKRC(psi_hdot_t<T>(p, da, dx, s));
    if (!dev) { CK(cudaMemcpyAsync(out, dx, xb, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s)); }
  }
  return PFBG_OK;
}

extern "C" int pfbs_psi_dot(pfbs_psi* p, const void* x, void* alpha, uint32_t flags, void* stream) {
  if (!p || !x || !alpha) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(p->device));
  return p->precision == PFBG_F32 ? psi_apply<float>(p, x, alpha, flags, (cudaStream_t)stream, true)
                                  : psi_apply<double>(p, x, alpha, flags, (cudaStream_t)stream, true);
}

extern "C" int pfbs_psi_hdot(pfbs_psi* p, const void* alpha, void* x, uint32_t flags, void* stream) {
  if (!p || !x || !alpha) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(p->device));
  return p->precision == PFBG_F32 ? psi_apply<float>(p, alpha, x, flags, (cudaStream_t)stream, false)
                                  : psi_apply<double>(p, alpha, x, flags, (cudaStream_t)stream, false);
}

// ---------------------------------------------------------------------------
// element-wise pieces (device pointers only: they live inside the device-resident primal-dual loop)
// ---------------------------------------------------------------------------
static unsigned nblk(int64_t n) { return (unsigned)((n + 255) / 256); }

extern "C" int pfbs_dual_update(int32_t precision, int32_t device, const void* vp, void* v, const void* weight,
                                double lam, double sigma, int32_t nband, int64_t ncoef, void* bsum, int32_t phase,
                                void* vbar, void* stream) {
  if (!v || !weight || (phase != 2 && !vp) || (phase != 0 && !bsum) || (vbar && !vp))
    return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (vbar && phase == 1) return pfbg_fail(PFBG_ERR_ARG, "the extrapolated dual is written by phase 0 or 2");
  if (phase < 0 || phase > 2 || nband < 1 || ncoef < 0) return pfbg_fail(PFBG_ERR_ARG, "bad phase / sizes");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  if (ncoef == 0) return PFBG_OK;
  if (precision == PFBG_F32)
    k_dual_update<float><<<nblk(ncoef), 256, 0, s>>>((const float*)vp, (float*)v, (const float*)weight, (float)lam, (float)sigma, nband, ncoef, (float*)bsum, phase, (float*)vbar);
  else if (precision == PFBG_F64)
    k_dual_update<double><<<nblk(ncoef), 256, 0, s>>>((const double*)vp, (double*)v, (const double*)weight, lam, sigma, nband, ncoef, (double*)bsum, phase, (double*)vbar);
  else return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

extern "C" int pfbs_prox_21m(int32_t precision, int32_t device, const void* v, void* result, const void* weight,
                             double lam, double sigma, int32_t nband, int64_t ncoef, void* stream) {
  if (!v || !result || !weight) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (nband < 1 || ncoef < 0 || !(sigma > 0)) return pfbg_fail(PFBG_ERR_ARG, "bad sizes / sigma");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  if (ncoef == 0) return PFBG_OK;
  if (precision == PFBG_F32)
    k_prox_21m<float><<<nblk(ncoef), 256, 0, s>>>((const float*)v, (float*)result, (const float*)weight, (float)lam, (float)sigma, nband, ncoef);
  else if (precision == PFBG_F64)
    k_prox_21m<double><<<nblk(ncoef), 256, 0, s>>>((const double*)v, (double*)result, (const double*)weight, lam, sigma, nband, ncoef);
  else return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

extern "C" int pfbs_extrapolate(int32_t precision, int32_t device, const void* v, void* vp, int64_t n, void* stream) {
  if (!v || !vp) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  if (n <= 0) return PFBG_OK;
  if (precision == PFBG_F32) k_extrapolate<float><<<nblk(n), 256, 0, s>>>((const float*)v, (float*)vp, n);
  else if (precision == PFBG_F64) k_extrapolate<double><<<nblk(n), 256, 0, s>>>((const double*)v, (double*)vp, n);
  else return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

extern "C" int pfbs_axpby(int32_t precision, int32_t device, void* out, double a, const void* x, double b, const void* y,
                          int64_t n, void* stream) {
  if (!out || !x || !y) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  if (n <= 0) return PFBG_OK;
  if (precision == PFBG_F32) k_axpby<float><<<nblk(n), 256, 0, s>>>((float*)out, (float)a, (const float*)x, (float)b, (const float*)y, n);
  else if (precision == PFBG_F64) k_axpby<double><<<nblk(n), 256, 0, s>>>((double*)out, a, (const double*)x, b, (const double*)y, n);
  else return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

extern "C" int pfbs_primal_step(int32_t precision, int32_t device, void* x, const void* xp, const void* xout, double tau,
                                int32_t positivity, int32_t nband, int64_t npix, void* stream) {
  if (!x || !xp || !xout) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (positivity < 0 || positivity > 2 || nband < 1) return pfbg_fail(PFBG_ERR_ARG, "bad positivity mode / nband");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  if (npix <= 0) return PFBG_OK;
  if (precision == PFBG_F32)
    k_primal_step<float><<<nblk(npix), 256, 0, s>>>((float*)x, (const float*)xp, (const float*)xout, (float)tau, positivity, nband, npix);
  else if (precision == PFBG_F64)
    k_primal_step<double><<<nblk(npix), 256, 0, s>>>((double*)x, (const double*)xp, (const double*)xout, tau, positivity, nband, npix);
  else return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

// two doubles of device scratch for the reductions, held for the duration of the call (pfbgrid.cu: recycled blocks,
// one per concurrent caller, so host threads / streams on one device never share an accumulator; no cudaMalloc /
// cudaFree, which synchronises the device, inside the solver loops)

template <typename K>
static int reduce2(int device, cudaStream_t s, double* out2, K launch) {
  struct Hold {
    int dev; void* p;
    ~Hold() { pfbg_scratch_put(dev, p); }
  } hold{device, pfbg_scratch_get(device)};
  double* acc = (double*)hold.p;
  if (!acc) return pfbg_fail(PFBG_ERR_NOMEM, "no reduction scratch on device %d", device);
  CK(cudaMemsetAsync(acc, 0, 16, s));
  launch(acc);
  LAUNCHED();
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out2, acc, 16, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return PFBG_OK;
}

extern "C" int pfbs_norm_diff(int32_t precision, int32_t device, const void* x, const void* xp, int64_t n,
                              double* num_den, void* stream) {
  if (!x || !xp || !num_den) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (precision != PFBG_F32 && precision != PFBG_F64) return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  num_den[0] = num_den[1] = 0.0;
  if (n <= 0) return PFBG_OK;
  const unsigned grd = n < (int64_t)1184 * 256 ? nblk(n) : 1184;  // 148 SMs x 8 CTAs
  return reduce2(device, s, num_den, [&](double* acc) {
    if (precision == PFBG_F32) k_norm_diff<float><<<grd, 256, 0, s>>>((const float*)x, (const float*)xp, n, acc);
    else k_norm_diff<double><<<grd, 256, 0, s>>>((const double*)x, (const double*)xp, n, acc);
  });
}

extern "C" int pfbs_dot2(int32_t precision, int32_t device, const void* a, const void* b, const void* c, const void* d,
                         int64_t n, double* out2, void* stream) {
  if (!a || !b || !c || !d || !out2) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (precision != PFBG_F32 && precision != PFBG_F64) return pfbg_fail(PFBG_ERR_ARG, "bad precision");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  out2[0] = out2[1] = 0.0;
  if (n <= 0) return PFBG_OK;
  const unsigned grd = n < (int64_t)1184 * 256 ? nblk(n) : 1184;
  return reduce2(device, s, out2, [&](double* acc) {
    if (precision == PFBG_F32) k_dot2<float><<<grd, 256, 0, s>>>((const float*)a, (const float*)b, (const float*)c, (const float*)d, n, acc);
    else k_dot2<double><<<grd, 256, 0, s>>>((const double*)a, (const double*)b, (const double*)c, (const double*)d, n, acc);
  });
}

// ---------------------------------------------------------------------------
// Clark CLEAN minor cycle (clean.cuh)
// ---------------------------------------------------------------------------
struct pfbs_clark {
  int device = 0, nband = 0, nx = 0, ny = 0, nxp = 0, nyp = 0;
  int npix = 0, search_grid = 0, sub_grid = 0, log_cap = 0;
  std::vector<double> peak;
  std::vector<pfbg_conv*> conv;
  double *psf = nullptr, *peak_d = nullptr, *ID = nullptr, *R = nullptr, *model = nullptr, *s = nullptr;
  double *RA = nullptr, *SA = nullptr, *cand_s = nullptr, *slot_s = nullptr, *slot_r = nullptr, *log_d = nullptr;
  int *idx = nullptr, *cand_i = nullptr, *slot_a = nullptr, *log_p = nullptr, *ints = nullptr;  // ints: best_i, nsel, count
  int2* ij = nullptr;
  uint8_t* mask = nullptr;
  void* cub_tmp = nullptr;
  size_t cub_bytes = 0;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

extern "C" int pfbs_clark_destroy(pfbs_clark* h) {
  if (!h) return PFBG_OK;
  cudaSetDevice(h->device);
  for (pfbg_conv* cv : h->conv) pfbg_conv_destroy(cv);
  void* all[] = {h->psf, h->peak_d, h->ID, h->R, h->model, h->s, h->RA, h->SA, h->cand_s, h->slot_s, h->slot_r,
                 h->log_d, h->idx, h->cand_i, h->slot_a, h->log_p, h->ints, h->ij, h->mask, h->cub_tmp};
  for (void* q : all)
    if (q) cudaFree(q);
  for (cudaEvent_t e : h->ev)
    if (e) cudaEventDestroy(e);
  delete h;
  return PFBG_OK;
}

extern "C" int pfbs_clark_create(int32_t precision, int32_t device, int32_t nband, int32_t nx, int32_t ny,
                                 int32_t nx_psf, int32_t ny_psf, const void* psf, const void* psfhat, uint32_t flags,
                                 void* stream, pfbs_clark** out) {
  if (!out || !psf || !psfhat) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  *out = nullptr;
  if (precision != PFBG_F64) return pfbg_fail(PFBG_ERR_ARG, "the Clark minor cycle is fp64 only");
  if (nband < 1 || nband > PFBS_CLARK_MAX_BANDS) return pfbg_fail(PFBG_ERR_ARG, "nband %d not in 1..%d", nband, PFBS_CLARK_MAX_BANDS);
  if (nx < 1 || ny < 1 || nx_psf < nx || ny_psf < ny)
    return pfbg_fail(PFBG_ERR_ARG, "need 0 < nx <= nx_psf and 0 < ny <= ny_psf (got %d x %d, PSF %d x %d)", nx, ny, nx_psf, ny_psf);
  if ((int64_t)nx * ny > INT32_MAX) return pfbg_fail(PFBG_ERR_ARG, "nx * ny must be below 2^31");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return pfbg_fail(PFBG_ERR_ARG, "device %d out of range", device);
  CK(cudaSetDevice(device));
  int coop = 0, nsm = 0, occ = 0;
  CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
  if (!coop) return pfbg_fail(PFBG_ERR_CUDA, "device %d does not support cooperative launches", device);
  CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_clark_subminor, CLK_THREADS, (size_t)nband * sizeof(double)));
  if (occ < 1) return pfbg_fail(PFBG_ERR_CUDA, "the subminor kernel cannot be resident");
  cudaStream_t s = (cudaStream_t)stream;
  const cudaMemcpyKind kind = (flags & PFBG_DEVICE_PTRS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  pfbs_clark* h = new pfbs_clark();
  h->device = device; h->nband = nband; h->nx = nx; h->ny = ny; h->nxp = nx_psf; h->nyp = ny_psf;
  h->npix = nx * ny;
  // at most 2 CTAs per SM: every CTA reads every candidate slot once per component, so the slot traffic grows with
  // the square of the grid, while 2 x 148 x 256 threads already give each thread < 2 entries at |A| ~ 10^5
  h->sub_grid = nsm * (occ < 2 ? occ : 2);
  h->search_grid = nsm * 4;
  const size_t npix = h->npix, nb = nband;
  const size_t plane = (size_t)nx_psf * ny_psf;
  auto fail_free = [&](int rc) { pfbs_clark_destroy(h); return rc; };
  auto alloc = [&](void** p, size_t bytes) -> int {
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) { *p = nullptr; cudaGetLastError(); return pfbg_fail(PFBG_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e)); }
    return PFBG_OK;
  };
  int rc = PFBG_OK;
  void** bufs[] = {(void**)&h->psf, (void**)&h->ID, (void**)&h->R, (void**)&h->model, (void**)&h->s, (void**)&h->RA,
                   (void**)&h->SA, (void**)&h->idx, (void**)&h->ij, (void**)&h->mask, (void**)&h->peak_d,
                   (void**)&h->cand_s, (void**)&h->cand_i, (void**)&h->slot_s, (void**)&h->slot_a, (void**)&h->slot_r,
                   (void**)&h->ints};
  const size_t sizes[] = {nb * plane * 8, nb * npix * 8, nb * npix * 8, nb * npix * 8, npix * 8, nb * npix * 8,
                          npix * 8, npix * 4, npix * 8, npix, nb * 8,
                          (size_t)(h->search_grid + 1) * 8, (size_t)h->search_grid * 4, 2 * (size_t)h->sub_grid * 8,
                          2 * (size_t)h->sub_grid * 4, 2 * (size_t)h->sub_grid * nb * 8, 4 * 4};
  for (size_t k = 0; k < sizeof(sizes) / sizeof(sizes[0]) && rc == PFBG_OK; ++k) rc = alloc(bufs[k], sizes[k]);
  if (rc) return fail_free(rc);
  ClarkActive pred{h->s, 0.0};
  cudaError_t e = cub::DeviceSelect::If(nullptr, h->cub_bytes, thrust::counting_iterator<int>(0), h->idx, h->ints + 1,
                                        h->npix, pred, s);
  if (e != cudaSuccess) { cudaGetLastError(); return fail_free(pfbg_fail(PFBG_ERR_CUDA, "cub select sizing failed: %s", cudaGetErrorString(e))); }
  if ((rc = alloc(&h->cub_tmp, h->cub_bytes))) return fail_free(rc);
  e = cudaMemcpyAsync(h->psf, psf, nb * plane * 8, kind, s);
  h->peak.resize(nband);
  const size_t centre = (size_t)(nx_psf / 2) * ny_psf + ny_psf / 2;
  for (int b = 0; b < nband && e == cudaSuccess; ++b)
    e = cudaMemcpyAsync(&h->peak[b], h->psf + b * plane + centre, 8, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaMemcpy(h->peak_d, h->peak.data(), nb * 8, cudaMemcpyHostToDevice);
  for (int k = 0; k < 4 && e == cudaSuccess; ++k) e = cudaEventCreate(&h->ev[k]);
  if (e != cudaSuccess) { cudaGetLastError(); return fail_free(pfbg_fail(PFBG_ERR_CUDA, "PSF upload failed: %s", cudaGetErrorString(e))); }
  h->conv.assign(nband, nullptr);
  const size_t half = (size_t)nx_psf * (ny_psf / 2 + 1) * 16;
  for (int b = 0; b < nband; ++b) {
    if ((rc = pfbg_conv_create(PFBG_F64, device, nx, ny, nx_psf, ny_psf, &h->conv[b]))) return fail_free(rc);
    if ((rc = pfbg_conv_set_kernel(h->conv[b], (const char*)psfhat + b * half, 1, flags & PFBG_DEVICE_PTRS, stream)))
      return fail_free(rc);
  }
  *out = h;
  return PFBG_OK;
}

static int clark_log_reserve(pfbs_clark* h, int n) {
  if (n <= h->log_cap) return PFBG_OK;
  if (h->log_p) cudaFree(h->log_p);
  if (h->log_d) cudaFree(h->log_d);
  h->log_p = nullptr; h->log_d = nullptr; h->log_cap = 0;
  CKRC(stage_alloc((void**)&h->log_p, (size_t)n * 4));
  CKRC(stage_alloc((void**)&h->log_d, (size_t)n * h->nband * 8));
  h->log_cap = n;
  return PFBG_OK;
}

extern "C" int pfbs_clark_run(pfbs_clark* h, const void* dirty, const uint8_t* mask, void* model, void* residual,
                              double threshold, double gamma, double pf, int32_t maxit, double subpf, int32_t submaxit,
                              int32_t* niter, double* rmax, int64_t* nactive, int32_t* nsub, int64_t* peaks,
                              int64_t peaks_cap, float* times_ms, uint32_t flags, void* stream) {
  if (!h || !dirty || !model || !residual || !niter) return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (!(threshold >= 0.0) || threshold == HUGE_VAL) return pfbg_fail(PFBG_ERR_ARG, "threshold must be finite and >= 0");
  if (!(gamma > 0.0 && gamma <= 1.0)) return pfbg_fail(PFBG_ERR_ARG, "gamma must be in (0, 1]");
  if (!(pf >= 0.0) || pf == HUGE_VAL) return pfbg_fail(PFBG_ERR_ARG, "pf must be finite and >= 0");
  if (!(subpf > 0.0 && subpf < 1.0)) return pfbg_fail(PFBG_ERR_ARG, "subpf must be in (0, 1)");
  if (maxit < 0 || submaxit < 1) return pfbg_fail(PFBG_ERR_ARG, "need maxit >= 0 and submaxit >= 1");
  if (maxit > 0 && (!rmax || !nactive || !nsub || !peaks)) return pfbg_fail(PFBG_ERR_ARG, "null info buffer");
  if (peaks_cap < (int64_t)maxit * submaxit) return pfbg_fail(PFBG_ERR_ARG, "peaks holds %lld entries, maxit * submaxit = %lld",
                                                              (long long)peaks_cap, (long long)maxit * submaxit);
  CK(cudaSetDevice(h->device));
  CKRC(clark_log_reserve(h, submaxit));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const int npix = h->npix, nband = h->nband;
  const size_t ib = (size_t)nband * npix * 8;
  CK(cudaMemcpyAsync(h->ID, dirty, ib, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  if (mask) CK(cudaMemcpyAsync(h->mask, mask, npix, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->R, h->ID, ib, cudaMemcpyDeviceToDevice, s));
  CK(cudaMemsetAsync(h->model, 0, ib, s));
  double tol = -1.0;
  int k = 0;
  int64_t npeaks = 0;
  for (;; ++k) {
    if (times_ms) CK(cudaEventRecord(h->ev[0], s));
    k_clark_search<<<h->search_grid, CLK_THREADS, 0, s>>>(h->R, nband, npix, mask ? h->mask : nullptr, h->s, h->cand_s, h->cand_i);
    k_clark_best<<<1, CLK_THREADS, 0, s>>>(h->cand_s, h->cand_i, h->search_grid, h->cand_s + h->search_grid, h->ints);
    LAUNCHED(); LAUNCHED();
    CK(cudaGetLastError());
    double Rmax = 0.0;
    CK(cudaMemcpyAsync(&Rmax, h->cand_s + h->search_grid, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (Rmax < 0.0) Rmax = 0.0;  // no pixel is searched
    if (k == 0) tol = std::max(pf * Rmax, threshold);
    if (!(Rmax > tol) || k >= maxit) break;
    const ClarkActive pred{h->s, subpf * Rmax};
    CK(cub::DeviceSelect::If(h->cub_tmp, h->cub_bytes, thrust::counting_iterator<int>(0), h->idx, h->ints + 1, npix, pred, s));
    int nA = 0;
    CK(cudaMemcpyAsync(&nA, h->ints + 1, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const int ga = std::min((nA + CLK_THREADS - 1) / CLK_THREADS, h->search_grid);
    k_clark_gather<<<std::max(ga, 1), CLK_THREADS, 0, s>>>(h->R, h->s, nband, npix, h->ny, h->idx, nA, h->RA, h->SA, h->ij);
    LAUNCHED();
    CK(cudaGetLastError());
    if (times_ms) CK(cudaEventRecord(h->ev[1], s));
    ClarkSub c{h->RA, h->SA, h->ij, nA, nband, h->ny, h->psf, h->peak_d, h->nxp, h->nyp, h->nxp / 2, h->nyp / 2,
               gamma, std::max(subpf * Rmax, threshold), submaxit, h->slot_s, h->slot_a, h->slot_r, h->log_p, h->log_d,
               h->ints + 2};
    const int grid = std::max(1, std::min((nA + CLK_THREADS - 1) / CLK_THREADS, h->sub_grid));
    void* args[] = {&c};
    CK(cudaLaunchCooperativeKernel((const void*)k_clark_subminor, dim3(grid), dim3(CLK_THREADS), args,
                                    (size_t)nband * sizeof(double), s));
    LAUNCHED();
    k_clark_replay<<<(nband + 31) / 32, 32, 0, s>>>(h->model, nband, npix, h->log_p, h->log_d, h->ints + 2);
    LAUNCHED();
    CK(cudaGetLastError());
    if (times_ms) CK(cudaEventRecord(h->ev[2], s));
    for (int b = 0; b < nband; ++b)
      CKRC(pfbg_conv_apply(h->conv[b], h->model + (int64_t)b * npix, nullptr, 0.0, h->R + (int64_t)b * npix, PFBG_DEVICE_PTRS, stream));
    k_clark_resid<<<h->search_grid, CLK_THREADS, 0, s>>>(h->ID, h->R, (int64_t)nband * npix);
    LAUNCHED();
    CK(cudaGetLastError());
    if (times_ms) CK(cudaEventRecord(h->ev[3], s));
    int cnt = 0;
    CK(cudaMemcpyAsync(&cnt, h->ints + 2, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    std::vector<int> lp(cnt);
    if (cnt) CK(cudaMemcpy(lp.data(), h->log_p, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
    for (int t = 0; t < cnt; ++t) peaks[npeaks + t] = lp[t];
    npeaks += cnt;
    rmax[k] = Rmax;
    nactive[k] = nA;
    nsub[k] = cnt;
    if (times_ms)
      for (int t = 0; t < 3; ++t) CK(cudaEventElapsedTime(&times_ms[3 * k + t], h->ev[t], h->ev[t + 1]));
  }
  *niter = k;
  const cudaMemcpyKind back = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  CK(cudaMemcpyAsync(model, h->model, ib, back, s));
  CK(cudaMemcpyAsync(residual, h->R, ib, back, s));
  if (!dev) CK(cudaStreamSynchronize(s));
  return PFBG_OK;
}

// ---------------------------------------------------------------------------
// Batched conjugate gradients on sums of PSF-convolution terms (cg.cuh): the one CG driver of the library.
// pfbs_psf_cg is the case of one group per system and scale 1.
// ---------------------------------------------------------------------------

static const int64_t kCgAlign = 256;
static int64_t cg_round(int64_t b) { return (b + kCgAlign - 1) / kCgAlign * kCgAlign; }
static int cg_grid(int64_t npix) { return (int)std::min<int64_t>((npix + CG_THREADS - 1) / CG_THREADS, CG_GMAX); }

// r, p, Ap, the partial sums and the CgCtl of every system, then (pingpong) one image for the running sum of a
// system with two or more groups: the systems are applied one after another on one stream, so they share it
static int64_t cg_work_bytes(int64_t nsys, int64_t npix, bool pingpong) {
  return 3 * cg_round(nsys * npix * 8) + cg_round(nsys * CG_GMAX * 2 * 8) + cg_round(nsys * (int64_t)sizeof(CgCtl)) +
         (pingpong ? cg_round(npix * 8) : 0);
}

extern "C" int64_t pfbs_psf_cg_work_bytes(int32_t nband, int64_t npix) {
  if (nband < 1 || npix < 1) return -1;
  return cg_work_bytes(nband, npix, false);
}

extern "C" int64_t pfbs_tree_cg_work_bytes(int32_t nsys, const int32_t* group_start, int64_t npix) {
  if (nsys < 1 || npix < 1 || !group_start) return -1;
  bool pingpong = false;
  for (int s = 0; s < nsys; ++s) pingpong |= group_start[s + 1] - group_start[s] >= 2;
  return cg_work_bytes(nsys, npix, pingpong);
}

extern "C" int pfbs_tree_cg(int32_t device, int32_t nsys, const int32_t* group_start, pfbg_conv* const* conv,
                            const void* const* beam, const double* scale, const double* eta, const void* rhs, void* x,
                            int64_t npix, double tol, int32_t maxit, int32_t minit, void* work, int64_t work_bytes,
                            int32_t* iters, double* eps, int32_t* stop, void* stream) {
  if (!group_start || !conv || !beam || !scale || !eta || !rhs || !x || !work || !iters || !eps || !stop)
    return pfbg_fail(PFBG_ERR_ARG, "null argument");
  if (nsys < 1 || nsys > 65535) return pfbg_fail(PFBG_ERR_ARG, "nsys %d not in 1..65535", nsys);
  if (!(tol >= 0.0) || maxit < 0 || minit < 0) return pfbg_fail(PFBG_ERR_ARG, "need tol >= 0, maxit >= 0, minit >= 0");
  if (group_start[0] != 0) return pfbg_fail(PFBG_ERR_ARG, "group_start[0] = %d, not 0", group_start[0]);
  for (int s = 0; s < nsys; ++s) {
    if (group_start[s + 1] <= group_start[s])
      return pfbg_fail(PFBG_ERR_ARG, "system %d has no group (group_start[%d] = %d, group_start[%d] = %d)", s, s,
                       group_start[s], s + 1, group_start[s + 1]);
    if (!(scale[s] > 0.0) || !std::isfinite(scale[s]))
      return pfbg_fail(PFBG_ERR_ARG, "scale[%d] = %g must be finite and > 0", s, scale[s]);
  }
  const int ngroup = group_start[nsys];
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return pfbg_fail(PFBG_ERR_ARG, "device %d out of range", device);
  int nx0 = 0, ny0 = 0;
  for (int g = 0; g < ngroup; ++g) {
    int prec = 0, dev = 0, nx = 0, ny = 0, hk = 0;
    if (!conv[g]) return pfbg_fail(PFBG_ERR_ARG, "convolver %d is NULL", g);
    CKRC(pfbg_conv_props(conv[g], &prec, &dev, &nx, &ny, &hk));
    if (prec != PFBG_F64) return pfbg_fail(PFBG_ERR_ARG, "convolver %d is not fp64", g);
    if (dev != device) return pfbg_fail(PFBG_ERR_ARG, "convolver %d is on device %d, not %d", g, dev, device);
    if (!hk) return pfbg_fail(PFBG_ERR_STATE, "convolver %d has no kernel", g);
    if (g == 0) { nx0 = nx; ny0 = ny; }
    else if (nx != nx0 || ny != ny0)
      return pfbg_fail(PFBG_ERR_ARG, "convolver %d images are %d x %d, convolver 0's %d x %d", g, nx, ny, nx0, ny0);
  }
  if (npix != (int64_t)nx0 * ny0) return pfbg_fail(PFBG_ERR_ARG, "npix %lld != nx * ny = %lld", (long long)npix, (long long)nx0 * ny0);
  const int64_t need = pfbs_tree_cg_work_bytes(nsys, group_start, npix);
  if (work_bytes < need) return pfbg_fail(PFBG_ERR_ARG, "work holds %lld bytes, %lld needed", (long long)work_bytes, (long long)need);
  CK(cudaSetDevice(device));
  if (!pfbg_on_device(rhs, device) || !pfbg_on_device(x, device) || !pfbg_on_device(work, device))
    return pfbg_fail(PFBG_ERR_ARG, "rhs, x and work must be device arrays on device %d", device);
  for (int g = 0; g < ngroup; ++g)
    if (beam[g] && !pfbg_on_device(beam[g], device)) return pfbg_fail(PFBG_ERR_ARG, "beam %d is not a device array on device %d", g, device);

  cudaStream_t s = (cudaStream_t)stream;
  const int64_t vb = cg_round((int64_t)nsys * npix * 8);
  double* r = (double*)work;
  double* p = (double*)((char*)work + vb);
  double* ap = (double*)((char*)work + 2 * vb);
  double* part = (double*)((char*)work + 3 * vb);
  CgCtl* ctl = (CgCtl*)((char*)part + cg_round((int64_t)nsys * CG_GMAX * 2 * 8));
  double* pong = (double*)((char*)ctl + cg_round((int64_t)nsys * (int64_t)sizeof(CgCtl)));
  const int G = cg_grid(npix);
  const dim3 grd(G, nsys);
  const double* xd = (const double*)x;
  std::vector<CgCtl> h(nsys);
  // out_s = scale_s sum_g beam_g conv_g(beam_g in_s) + eta_s in_s: the first group adds the ridge term, each later one
  // adds the running sum (eta = 1) from the other buffer, and the parity puts the last group's output in out_s
  auto apply = [&](const double* in, double* out, int sys) -> int {
    const double* xs = in + sys * npix;
    const double* prev = nullptr;
    const int g0 = group_start[sys], g1 = group_start[sys + 1];
    for (int g = g0; g < g1; ++g) {
      double* dst = ((g1 - 1 - g) & 1) ? pong : out + sys * npix;
      CKRC(pfbg_conv_apply_dev(conv[g], xs, beam[g], g == g0 ? xs : prev, g == g0 ? eta[sys] : 1.0, scale[sys], dst,
                               stream));
      prev = dst;
    }
    return PFBG_OK;
  };
  auto read_ctl = [&]() -> int {
    CK(cudaMemcpyAsync(h.data(), ctl, (size_t)nsys * sizeof(CgCtl), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return PFBG_OK;
  };

  for (int b = 0; b < nsys; ++b) CKRC(apply(xd, r, b));  // r = A x
  k_cg_init<<<grd, CG_THREADS, 0, s>>>((const double*)rhs, r, p, npix, part);
  k_cg_init_fin<<<nsys, CG_THREADS, 0, s>>>(ctl, part, G, tol, maxit, minit);
  LAUNCHED(); LAUNCHED();
  CK(cudaGetLastError());
  CKRC(read_ctl());
  for (;;) {
    bool any = false;
    for (int b = 0; b < nsys; ++b)
      if (h[b].stop == CG_RUNNING) { any = true; CKRC(apply(p, ap, b)); }  // stopped systems skip their convolutions
    if (!any) break;
    k_cg_dots<<<grd, CG_THREADS, 0, s>>>(ctl, p, ap, npix, part);
    k_cg_dots_fin<<<nsys, CG_THREADS, 0, s>>>(ctl, part, G);
    k_cg_update<<<grd, CG_THREADS, 0, s>>>(ctl, (double*)x, r, p, ap, npix, part);
    k_cg_update_fin<<<nsys, CG_THREADS, 0, s>>>(ctl, part, G, tol, maxit, minit);
    k_cg_direction<<<grd, CG_THREADS, 0, s>>>(ctl, p, r, npix);
    for (int t = 0; t < 5; ++t) LAUNCHED();
    CK(cudaGetLastError());
    CKRC(read_ctl());
  }
  for (int b = 0; b < nsys; ++b) {
    iters[b] = h[b].k;
    eps[b] = h[b].eps;
    stop[b] = h[b].stop;
  }
  return PFBG_OK;
}

extern "C" int pfbs_psf_cg(int32_t device, int32_t nband, pfbg_conv* const* conv, const void* const* beam,
                           const double* eta, const void* rhs, void* x, int64_t npix, double tol, int32_t maxit,
                           int32_t minit, void* work, int64_t work_bytes, int32_t* iters, double* eps, int32_t* stop,
                           void* stream) {
  if (nband < 1 || nband > 65535) return pfbg_fail(PFBG_ERR_ARG, "nband %d not in 1..65535", nband);
  std::vector<int32_t> group_start(nband + 1);
  for (int b = 0; b <= nband; ++b) group_start[b] = b;
  const std::vector<double> scale(nband, 1.0);
  return pfbs_tree_cg(device, nband, group_start.data(), conv, beam, scale.data(), eta, rhs, x, npix, tol, maxit, minit,
                      work, work_bytes, iters, eps, stop, stream);
}
