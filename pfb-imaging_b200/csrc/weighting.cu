// Imaging-weight entry points of the C ABI (include/pfbgrid.h; kernels in weighting.cuh): counts, Briggs / uniform
// re-weighting (utils/weighting.py:81-140, 143-208), the l2 re-weighting and the data / weights of one correlation.
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "host.h"
#include "weighting.cuh"

static constexpr double kLightspeed = 299792458.0;

static WParams make_wparams(int64_t nrow, int nchan, int ncorr, int nx, int ny, double cell_x, double cell_y,
                            double usign, double vsign) {
  WParams w;
  w.nrow = nrow; w.nchan = nchan; w.ncorr = ncorr; w.nx = nx; w.ny = ny;
  w.u_cell = 1.0 / ((double)nx * cell_x);
  w.umax = fabs(1.0 / cell_x / 2.0);
  w.v_cell = 1.0 / ((double)ny * cell_y);
  w.vmax = fabs(1.0 / cell_y / 2.0);
  w.usign = usign; w.vsign = vsign; w.lightspeed = kLightspeed;
  return w;
}

// reduction launch of the counts kernels: blockIdx.y over up to kCountsGridsPerLaunch grids, ~1184 CTAs in all
static dim3 counts_rgrid(int64_t ngrid) {
  const int gy = (int)std::min<int64_t>(ngrid, kCountsGridsPerLaunch);
  return dim3((unsigned)std::max(8, 1184 / gy), (unsigned)gy);
}

template <typename T>
static int launch_counts(cudaStream_t s, const WParams& w, const double* uvw, const double* scale, const uint8_t* mask,
                         const int* row_snap, const T* wgt, T* counts, size_t cbytes) {
  CK(cudaMemsetAsync(counts, 0, cbytes, s));
  const int64_t nvis = w.nrow * w.nchan;
  if (nvis > 0) {
    k_counts<T><<<(unsigned)((nvis + 255) / 256), 256, 0, s>>>(w, uvw, scale, mask, row_snap, wgt, counts, nullptr);
    LAUNCHED();
    CK(cudaGetLastError());
  }
  return PFBG_OK;
}

// counts (nsnap * ncorr grids) -> Briggs / uniform weights, in place on counts and wgt (weighting.py:143-208);
// sums: 3 * nsnap * ncorr doubles of scratch.  No host synchronisation.
template <typename T>
static int launch_reweight(cudaStream_t s, const WParams& w, const double* uvw, const double* scale,
                           const uint8_t* mask, const int* row_snap, int64_t nsnap, T* counts, double* sums,
                           double robust, T* wgt) {
  const int64_t ncell = (int64_t)w.nx * w.ny, ngrid = nsnap * w.ncorr, nvis = w.nrow * w.nchan;
  const dim3 rg = counts_rgrid(ngrid);
  CK(cudaMemsetAsync(sums, 0, (size_t)ngrid * 3 * sizeof(double), s));
  k_counts_sums<T><<<rg, 256, 0, s>>>(counts, ncell, (int)ngrid, sums);
  LAUNCHED();
  if (robust > -2.0) {
    const double numsqrt = 5.0 * pow(10.0, -robust);
    k_counts_scale<T><<<rg, 256, 0, s>>>(counts, ncell, w.ncorr, (int)ngrid, sums, numsqrt * numsqrt);
    LAUNCHED();
  }
  if (nvis > 0) {
    k_apply_counts<T><<<(unsigned)((nvis + 255) / 256), 256, 0, s>>>(w, uvw, scale, mask, row_snap, counts, wgt);
    LAUNCHED();
  }
  CK(cudaGetLastError());
  return PFBG_OK;
}

int pfbg_counts_reweight(int precision, cudaStream_t s, int64_t nrow, int nchan, int nx, int ny, double cell_x,
                         double cell_y, double usign, double vsign, double lightspeed, const double* uvw,
                         const double* scale, const uint8_t* mask, const int* row_snap, int64_t nsnap, double robust,
                         void* counts, double* sums, void* wgt) {
  WParams w = make_wparams(nrow, nchan, 1, nx, ny, cell_x, cell_y, usign, vsign);
  w.lightspeed = lightspeed;
  const size_t cbytes = (size_t)nsnap * nx * ny * (precision == PFBG_F32 ? 4 : 8);
  if (precision == PFBG_F32) {
    CKRC(launch_counts<float>(s, w, uvw, scale, mask, row_snap, (const float*)wgt, (float*)counts, cbytes));
    return launch_reweight<float>(s, w, uvw, scale, mask, row_snap, nsnap, (float*)counts, sums, robust, (float*)wgt);
  }
  CKRC(launch_counts<double>(s, w, uvw, scale, mask, row_snap, (const double*)wgt, (double*)counts, cbytes));
  return launch_reweight<double>(s, w, uvw, scale, mask, row_snap, nsnap, (double*)counts, sums, robust, (double*)wgt);
}

extern "C" int pfbg_counts(int32_t precision, int32_t device, const double* uvw, const double* freq,
                           const uint8_t* mask, const void* wgt, int64_t nrow, int32_t nchan, int32_t ncorr,
                           int32_t nx, int32_t ny, double cell_x, double cell_y, double usign, double vsign,
                           void* counts, uint32_t flags, void* stream) {
  if (!uvw || !freq || !wgt || !counts) return fail(PFBG_ERR_ARG, "null argument");
  if (nrow < 0 || nchan <= 0 || ncorr <= 0 || nx <= 0 || ny <= 0) return fail(PFBG_ERR_ARG, "bad sizes");
  if (precision != PFBG_F32 && precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = precision == PFBG_F32 ? 4 : 8;
  const int64_t nvis = nrow * nchan;
  const size_t cbytes = (size_t)ncorr * nx * ny * rb;
  TmpBufs t;
  void *duvw, *dfreq, *dmask = nullptr, *dwgt, *dcounts;
  CKRC(t.get(&duvw, uvw, (size_t)nrow * 24, dev, true, s));
  CKRC(t.get(&dfreq, freq, (size_t)nchan * 8, dev, true, s));
  if (mask) CKRC(t.get(&dmask, mask, (size_t)nvis, dev, true, s));
  CKRC(t.get(&dwgt, wgt, (size_t)ncorr * nvis * rb, dev, true, s));
  CKRC(t.get(&dcounts, counts, cbytes, dev, false, s));
  WParams w = make_wparams(nrow, nchan, ncorr, nx, ny, cell_x, cell_y, usign, vsign);
  if (precision == PFBG_F32)
    CKRC(launch_counts<float>(s, w, (const double*)duvw, (const double*)dfreq, (const uint8_t*)dmask, nullptr, (const float*)dwgt, (float*)dcounts, cbytes));
  else
    CKRC(launch_counts<double>(s, w, (const double*)duvw, (const double*)dfreq, (const uint8_t*)dmask, nullptr, (const double*)dwgt, (double*)dcounts, cbytes));
  if (!dev) {
    CK(cudaMemcpyAsync(counts, dcounts, cbytes, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  return PFBG_OK;
}

// cell index dump for the bit-exact check: cells (nrow,nchan,2) int32, -1 = skipped
extern "C" int pfbg_counts_cells(int32_t device, const double* uvw, const double* freq, const uint8_t* mask,
                                 int64_t nrow, int32_t nchan, int32_t nx, int32_t ny, double cell_x, double cell_y,
                                 double usign, double vsign, int32_t* cells) {
  if (!uvw || !freq || !cells) return fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(device));
  const int64_t nvis = nrow * nchan;
  TmpBufs t;
  void *duvw, *dfreq, *dmask = nullptr, *dcells;
  CKRC(t.get(&duvw, uvw, (size_t)nrow * 24, false, true, 0));
  CKRC(t.get(&dfreq, freq, (size_t)nchan * 8, false, true, 0));
  if (mask) CKRC(t.get(&dmask, mask, (size_t)nvis, false, true, 0));
  CKRC(t.get(&dcells, cells, (size_t)nvis * 8, false, false, 0));
  WParams w = make_wparams(nrow, nchan, 1, nx, ny, cell_x, cell_y, usign, vsign);
  if (nvis > 0) {
    k_counts<float><<<(unsigned)((nvis + 255) / 256), 256>>>(w, (const double*)duvw, (const double*)dfreq, (const uint8_t*)dmask, nullptr, nullptr, nullptr, (int32_t*)dcells);
    LAUNCHED();
    CK(cudaGetLastError());
    CK(cudaMemcpy(cells, dcells, (size_t)nvis * 8, cudaMemcpyDeviceToHost));
  }
  return PFBG_OK;
}

extern "C" int pfbg_counts_to_weights(int32_t precision, int32_t device, void* counts, const double* uvw,
                                      const double* freq, void* wgt, const uint8_t* mask, int64_t nrow,
                                      int32_t nchan, int32_t ncorr, int32_t nx, int32_t ny, double cell_x,
                                      double cell_y, double robust, double usign, double vsign, uint32_t flags,
                                      void* stream) {
  if (!uvw || !freq || !wgt || !counts) return fail(PFBG_ERR_ARG, "null argument");
  if (nrow < 0 || nchan <= 0 || ncorr <= 0 || ncorr > 16 || nx <= 0 || ny <= 0) return fail(PFBG_ERR_ARG, "bad sizes");
  if (precision != PFBG_F32 && precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = precision == PFBG_F32 ? 4 : 8;
  const int64_t nvis = nrow * nchan, ncell = (int64_t)nx * ny;
  const size_t cbytes = (size_t)ncorr * ncell * rb, wbytes = (size_t)ncorr * nvis * rb;
  TmpBufs t;
  void *duvw, *dfreq, *dmask = nullptr, *dwgt, *dcounts, *dsums;
  CKRC(t.get(&duvw, uvw, (size_t)nrow * 24, dev, true, s));
  CKRC(t.get(&dfreq, freq, (size_t)nchan * 8, dev, true, s));
  if (mask) CKRC(t.get(&dmask, mask, (size_t)nvis, dev, true, s));
  CKRC(t.get(&dwgt, wgt, wbytes, dev, true, s));
  CKRC(t.get(&dcounts, counts, cbytes, dev, true, s));
  CKRC(t.get(&dsums, nullptr, (size_t)ncorr * 3 * 8, false, false, s));
  WParams w = make_wparams(nrow, nchan, ncorr, nx, ny, cell_x, cell_y, usign, vsign);
  if (precision == PFBG_F32)
    CKRC(launch_reweight<float>(s, w, (const double*)duvw, (const double*)dfreq, (const uint8_t*)dmask, nullptr, 1, (float*)dcounts, (double*)dsums, robust, (float*)dwgt));
  else
    CKRC(launch_reweight<double>(s, w, (const double*)duvw, (const double*)dfreq, (const uint8_t*)dmask, nullptr, 1, (double*)dcounts, (double*)dsums, robust, (double*)dwgt));
  if (!dev) {
    CK(cudaMemcpyAsync(wgt, dwgt, wbytes, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(counts, dcounts, cbytes, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return PFBG_OK;
}

// Arguments of the batched re-weighting, checked before anything is launched.
static int check_batch_weights(int64_t nbatch, const int64_t* row_offsets, int64_t nrow, int32_t nx_pad,
                               int32_t ny_pad, double cell_x, double cell_y) {
  if (nbatch < 1) return fail(PFBG_ERR_ARG, "nbatch must be positive");
  if (!row_offsets) return fail(PFBG_ERR_ARG, "null row_offsets");
  if (row_offsets[0] != 0 || row_offsets[nbatch] != nrow) return fail(PFBG_ERR_ARG, "row_offsets must run from 0 to nrow = %lld", (long long)nrow);
  for (int64_t b = 0; b < nbatch; ++b)
    if (row_offsets[b + 1] < row_offsets[b]) return fail(PFBG_ERR_ARG, "row_offsets must not decrease (snapshot %lld)", (long long)b);
  if (nx_pad <= 0 || ny_pad <= 0) return fail(PFBG_ERR_ARG, "pad sizes must be positive, got %d x %d", nx_pad, ny_pad);
  if (!std::isfinite(cell_x) || !std::isfinite(cell_y) || !(cell_x > 0) || !(cell_y > 0))
    return fail(PFBG_ERR_ARG, "cell sizes must be finite and positive");
  return PFBG_OK;
}

extern "C" int pfbg_counts_to_weights_batch(int32_t precision, int32_t device, int32_t nbatch, const int64_t* row_offsets,
                                            const double* uvw, const double* freq, const uint8_t* mask, void* wgt,
                                            int64_t nrow, int32_t nchan, int32_t nx_pad, int32_t ny_pad, double cell_x,
                                            double cell_y, double robust, double usign, double vsign, void* counts,
                                            uint32_t flags, void* stream) {
  if (precision != PFBG_F32 && precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  if (nrow < 0 || nchan <= 0) return fail(PFBG_ERR_ARG, "bad nrow / nchan");
  if (!freq || (nrow > 0 && (!uvw || !wgt))) return fail(PFBG_ERR_ARG, "null argument");
  CKRC(check_batch_weights(nbatch, row_offsets, nrow, nx_pad, ny_pad, cell_x, cell_y));
  std::vector<int> rs((size_t)(nrow > 0 ? nrow : 1));
  for (int b = 0; b < nbatch; ++b)
    for (int64_t r = row_offsets[b]; r < row_offsets[b + 1]; ++r) rs[(size_t)r] = b;
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = precision == PFBG_F32 ? 4 : 8;
  const int64_t nvis = nrow * nchan;
  const size_t cbytes = (size_t)nbatch * nx_pad * ny_pad * rb, wbytes = (size_t)nvis * rb;
  TmpBufs t;
  void *duvw, *dfreq, *dmask = nullptr, *dwgt, *dcounts, *dsums, *drs;
  CKRC(t.get(&duvw, uvw, (size_t)nrow * 24, dev, true, s));
  CKRC(t.get(&dfreq, freq, (size_t)nchan * 8, dev, true, s));
  if (mask) CKRC(t.get(&dmask, mask, (size_t)nvis, dev, true, s));
  CKRC(t.get(&dwgt, wgt, wbytes, dev, true, s));
  CKRC(t.get(&dcounts, counts, cbytes, dev && counts, false, s));
  CKRC(t.get(&dsums, nullptr, (size_t)nbatch * 3 * 8, false, false, s));
  CKRC(t.get(&drs, rs.data(), rs.size() * 4, false, true, s));
  CKRC(pfbg_counts_reweight(precision, s, nrow, nchan, nx_pad, ny_pad, cell_x, cell_y, usign, vsign, kLightspeed,
                            (const double*)duvw, (const double*)dfreq, (const uint8_t*)dmask, (const int*)drs, nbatch,
                            robust, dcounts, (double*)dsums, dwgt));
  if (!dev) {
    if (nvis > 0) CK(cudaMemcpyAsync(wgt, dwgt, wbytes, cudaMemcpyDeviceToHost, s));
    if (counts) CK(cudaMemcpyAsync(counts, dcounts, cbytes, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return PFBG_OK;
}

extern "C" int pfbg_l2_reweight(int32_t precision, int32_t device, const void* resvis, const void* wgtp,
                                const uint8_t* mask, void* wgt, int64_t nvis, int32_t ncorr, double dof,
                                double* ovar_out, int32_t* applied, uint32_t flags, void* stream) {
  if (!resvis || !wgt || !ovar_out || !applied) return fail(PFBG_ERR_ARG, "null argument");
  if (nvis < 0 || ncorr <= 0 || ncorr > 16) return fail(PFBG_ERR_ARG, "bad sizes");
  if (precision != PFBG_F32 && precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = precision == PFBG_F32 ? 4 : 8;
  const size_t wbytes = (size_t)ncorr * nvis * rb;
  *applied = 0;
  TmpBufs t;
  void *drv, *dp = nullptr, *dmask = nullptr, *dwgt, *dsums;
  CKRC(t.get(&drv, resvis, 2 * wbytes, dev, true, s));
  if (wgtp) CKRC(t.get(&dp, wgtp, wbytes, dev, true, s));
  if (mask) CKRC(t.get(&dmask, mask, (size_t)nvis, dev, true, s));
  CKRC(t.get(&dwgt, wgt, wbytes, dev, true, s));
  // 17 doubles of reduction scratch, held for this call (pfbg_scratch_get: recycled blocks, no cudaMalloc per call)
  struct Hold {
    int dev; void* p;
    ~Hold() { pfbg_scratch_put(dev, p); }
  } hold{device, pfbg_scratch_get(device)};
  if (!hold.p) return fail(PFBG_ERR_NOMEM, "no reduction scratch on device %d", device);
  dsums = hold.p;
  CK(cudaMemsetAsync(dsums, 0, 17 * 8, s));
  dim3 rgrid(592, ncorr);
  if (nvis > 0) {
    if (precision == PFBG_F32) k_l2_ssq<float><<<rgrid, 256, 0, s>>>((const float*)drv, (const float*)dp, (const uint8_t*)dmask, nvis, (double*)dsums);
    else k_l2_ssq<double><<<rgrid, 256, 0, s>>>((const double*)drv, (const double*)dp, (const uint8_t*)dmask, nvis, (double*)dsums);
    LAUNCHED();
  }
  double sums[17];
  CK(cudaMemcpyAsync(sums, dsums, sizeof sums, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  bool all_nonzero = true;
  for (int c = 0; c < ncorr; ++c) {
    ovar_out[c] = sums[c] / sums[ncorr];  // 0/0 -> NaN like numpy; NaN is truthy there too
    if (ovar_out[c] == 0.0) all_nonzero = false;
  }
  if (!all_nonzero) return PFBG_OK;
  CK(cudaMemcpyAsync(dsums, ovar_out, ncorr * 8, cudaMemcpyHostToDevice, s));
  if (nvis > 0) {
    if (precision == PFBG_F32) k_l2_apply<float><<<rgrid, 256, 0, s>>>((const float*)drv, (const float*)dp, (float*)dwgt, nvis, (const double*)dsums, dof, dof + 2.0);
    else k_l2_apply<double><<<rgrid, 256, 0, s>>>((const double*)drv, (const double*)dp, (double*)dwgt, nvis, (const double*)dsums, dof, dof + 2.0);
    LAUNCHED();
    CK(cudaGetLastError());
    if (!dev) CK(cudaMemcpyAsync(wgt, dwgt, wbytes, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  *applied = 1;
  return PFBG_OK;
}

extern "C" int pfbg_weight_data_corr(int32_t precision, int32_t device, const void* data, const void* weight,
                                     const void* jones, const int32_t* row_t, const int32_t* ant1, const int32_t* ant2,
                                     int64_t nrow, int32_t nchan, int32_t ncorr, int64_t jones_elems, int64_t js_t,
                                     int64_t js_a, int64_t js_c, void* vis, void* wgt, uint32_t flags, void* stream) {
  if (!data || !weight || !jones || !row_t || !ant1 || !ant2 || !vis || !wgt) return fail(PFBG_ERR_ARG, "null argument");
  if (nrow < 0 || nchan <= 0 || ncorr <= 0 || jones_elems <= 0) return fail(PFBG_ERR_ARG, "bad sizes");
  if (precision != PFBG_F32 && precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  CK(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = precision == PFBG_F32 ? 4 : 8;
  const int64_t nvis = nrow * nchan;
  TmpBufs t;
  void *dd, *dw, *dj, *dt, *d1, *d2, *dv, *dg;
  CKRC(t.get(&dd, data, (size_t)nvis * ncorr * 2 * rb, dev, true, s));
  CKRC(t.get(&dw, weight, (size_t)nvis * ncorr * rb, dev, true, s));
  CKRC(t.get(&dj, jones, (size_t)jones_elems * 2 * rb, dev, true, s));
  CKRC(t.get(&dt, row_t, (size_t)nrow * 4, dev, true, s));
  CKRC(t.get(&d1, ant1, (size_t)nrow * 4, dev, true, s));
  CKRC(t.get(&d2, ant2, (size_t)nrow * 4, dev, true, s));
  CKRC(t.get(&dv, vis, (size_t)nvis * 2 * rb, dev, false, s));
  CKRC(t.get(&dg, wgt, (size_t)nvis * rb, dev, false, s));
  CK(cudaMemsetAsync(dv, 0, (size_t)nvis * 2 * rb, s));
  CK(cudaMemsetAsync(dg, 0, (size_t)nvis * rb, s));
  if (nvis > 0) {
    const unsigned grd = (unsigned)((nvis + 255) / 256);
    if (precision == PFBG_F32)
      k_weight_data_corr<float><<<grd, 256, 0, s>>>((const float2*)dd, (const float*)dw, (const float2*)dj, (const int32_t*)dt,
                                                      (const int32_t*)d1, (const int32_t*)d2, nrow, nchan, ncorr, js_t, js_a, js_c,
                                                      (float2*)dv, (float*)dg);
    else
      k_weight_data_corr<double><<<grd, 256, 0, s>>>((const double2*)dd, (const double*)dw, (const double2*)dj, (const int32_t*)dt,
                                                       (const int32_t*)d1, (const int32_t*)d2, nrow, nchan, ncorr, js_t, js_a, js_c,
                                                       (double2*)dv, (double*)dg);
    LAUNCHED();
    CK(cudaGetLastError());
    if (!dev) {
      CK(cudaMemcpyAsync(vis, dv, (size_t)nvis * 2 * rb, cudaMemcpyDeviceToHost, s));
      CK(cudaMemcpyAsync(wgt, dg, (size_t)nvis * rb, cudaMemcpyDeviceToHost, s));
    }
  }
  if (!dev) CK(cudaStreamSynchronize(s));
  return PFBG_OK;
}
