// Imaging-weight kernels: nearest-cell weight histogram on the padded uv grid and
// the Briggs / uniform re-weighting that divides by it.  The integer cell index
// follows /root/reference/src/pfb_imaging/utils/weighting.py:115-135 operation
// for operation in fp64 without FMA contraction (bit-exact contract).
//
// Every kernel takes a batch of snapshots (pfb hci, utils/stokes2im.py:563-604): row r belongs to snapshot
// row_snap[r] (row_snap == NULL: one snapshot), whose ncorr grids start at grid snapshot * ncorr of the counts cube
// (nsnap * ncorr, nx, ny).  No sample reaches another snapshot's grids, and each grid has its own sums and ssq, so a
// batch computes what one call per snapshot computes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct WParams {
  int64_t nrow;
  int nchan, ncorr, nx, ny;
  // scale[f] / lightspeed is f/c: freq with lightspeed = c, or a bound fscale = fl(freq / c) with lightspeed = 1
  // (an exact division, so both give the same cell)
  double u_cell, v_cell, umax, vmax, usign, vsign, lightspeed;
};

// grids of one launch of the reduction kernels along blockIdx.y; the kernels stride over further grids
constexpr int kCountsGridsPerLaunch = 64;

// returns false when the sample falls off the grid
__device__ __forceinline__ bool uv_cell(const WParams& w, const double* __restrict__ uvw,
                                        const double* __restrict__ scale, int64_t r, int f, int& ui, int& vi) {
  double cn = __ddiv_rn(scale[f], w.lightspeed);
  double u = __dmul_rn(__dmul_rn(uvw[3 * r + 0], cn), w.usign);
  double v = __dmul_rn(__dmul_rn(uvw[3 * r + 1], cn), w.vsign);
  if (v < 0) { u = -u; v = -v; }
  double ug = __ddiv_rn(__dadd_rn(u, w.umax), w.u_cell);
  double vg = __ddiv_rn(__dadd_rn(v, w.vmax), w.v_cell);
  double fu = floor(ug), fv = floor(vg);
  if (!(fu >= 0.0) || !(fu < (double)w.nx) || !(fv >= 0.0) || !(fv < (double)w.ny)) return false;
  ui = (int)fu;
  vi = (int)fv;
  return true;
}

// first cell of correlation c of the snapshot of row r
__device__ __forceinline__ int64_t grid_base(const WParams& w, const int* __restrict__ row_snap, int64_t r, int c) {
  const int64_t snap = row_snap ? row_snap[r] : 0;
  return (snap * w.ncorr + c) * w.nx * (int64_t)w.ny;
}

template <typename T>
__global__ void k_counts(WParams w, const double* __restrict__ uvw, const double* __restrict__ scale,
                         const uint8_t* __restrict__ mask, const int* __restrict__ row_snap, const T* __restrict__ wgt,
                         T* __restrict__ counts, int32_t* __restrict__ cell_dump) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t nvis = w.nrow * w.nchan;
  if (k >= nvis) return;
  int64_t r = k / w.nchan;
  int f = (int)(k - r * w.nchan);
  if (cell_dump) { cell_dump[2 * k] = -1; cell_dump[2 * k + 1] = -1; }
  if (mask && !mask[k]) return;
  int ui, vi;
  if (!uv_cell(w, uvw, scale, r, f, ui, vi)) return;
  if (cell_dump) { cell_dump[2 * k] = ui; cell_dump[2 * k + 1] = vi; }
  if (!counts) return;
  for (int c = 0; c < w.ncorr; ++c) {
    T v = wgt[(int64_t)c * nvis + k];
    atomicAdd(&counts[grid_base(w, row_snap, r, c) + (int64_t)ui * w.ny + vi], v);
  }
}

// per grid g of ngrid: sum(c^2) -> sums[3g], sum(c) -> sums[3g+1], 1 -> sums[3g+2] when any cell is non-zero
template <typename T>
__global__ void k_counts_sums(const T* __restrict__ counts, int64_t ncell, int ngrid, double* __restrict__ sums) {
  for (int g = blockIdx.y; g < ngrid; g += gridDim.y) {
    const T* p = counts + (int64_t)g * ncell;
    double s2 = 0, s1 = 0;
    bool nz = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncell; i += (int64_t)gridDim.x * blockDim.x) {
      double v = (double)p[i];
      s2 += v * v;
      s1 += v;
      nz |= (v != 0.0);
    }
    for (int o = 16; o > 0; o >>= 1) {
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    nz = __any_sync(0xffffffffu, nz);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(&sums[3 * g], s2);
      atomicAdd(&sums[3 * g + 1], s1);
      if (nz) sums[3 * g + 2] = 1.0;
    }
  }
}

// Briggs: counts = counts * ssq + 1 with ssq = numsq * sum(c) / sum(c^2) of the grid (weighting.py:162-174).  A
// snapshot whose grids are all zero is left as it is (`if not counts.any(): return weight`), so its weights are too.
template <typename T>
__global__ void k_counts_scale(T* __restrict__ counts, int64_t ncell, int ncorr, int ngrid,
                               const double* __restrict__ sums, double numsq) {
  for (int g = blockIdx.y; g < ngrid; g += gridDim.y) {
    const int g0 = g - g % ncorr;
    bool any = false;
    for (int c = 0; c < ncorr; ++c) any |= sums[3 * (g0 + c) + 2] != 0.0;
    if (!any) continue;
    const T s = (T)(numsq * sums[3 * g + 1] / sums[3 * g]);
    T* p = counts + (int64_t)g * ncell;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncell; i += (int64_t)gridDim.x * blockDim.x)
      p[i] = p[i] * s + (T)1;
  }
}

template <typename T>
__global__ void k_apply_counts(WParams w, const double* __restrict__ uvw, const double* __restrict__ scale,
                               const uint8_t* __restrict__ mask, const int* __restrict__ row_snap,
                               const T* __restrict__ counts, T* __restrict__ wgt) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t nvis = w.nrow * w.nchan;
  if (k >= nvis) return;
  int64_t r = k / w.nchan;
  int f = (int)(k - r * w.nchan);
  if (mask && !mask[k]) return;
  int ui, vi;
  if (!uv_cell(w, uvw, scale, r, f, ui, vi)) return;
  for (int c = 0; c < w.ncorr; ++c) {
    T cv = counts[grid_base(w, row_snap, r, c) + (int64_t)ui * w.ny + vi];
    if (cv > (T)0) wgt[(int64_t)c * nvis + k] /= cv;
  }
}

// ---------------------------------------------------------------------------
// l2 (Student-t) re-weighting from residual visibilities
// (/root/reference/src/pfb_imaging/operators/gridder.py:509-532):
//   ressq = |r|^2 * wgtp ;  ovar[c] = sum_{mask>0} ressq[c] / sum(mask) ;  wgt *= (dof + 2) / (dof + ressq / ovar[c])
// HBM-bound streaming passes: pass 1 reads r (2p) + wgtp (p) + mask (1) per sample, pass 2 reads r, wgtp, wgt and
// writes wgt.  Vectorisation is left to the 32-lane coalescing (consecutive k -> consecutive addresses).
// ---------------------------------------------------------------------------
template <typename T>
__global__ void k_l2_ssq(const T* __restrict__ rv, const T* __restrict__ wgtp, const uint8_t* __restrict__ mask,
                         int64_t nvis, double* __restrict__ sums /* ncorr + 1: ssq[c], mask count */) {
  int c = blockIdx.y;
  const T* r = rv + (int64_t)c * nvis * 2;
  const T* p = wgtp ? wgtp + (int64_t)c * nvis : nullptr;
  double s = 0;
  unsigned long long cnt = 0;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nvis; k += (int64_t)gridDim.x * blockDim.x) {
    if (mask && !mask[k]) continue;
    T re = r[2 * k], im = r[2 * k + 1];
    T q = p ? (re * p[k]) * re + (im * p[k]) * im : re * re + im * im;
    s += (double)q;
    ++cnt;
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&sums[c], s);
    if (c == 0) atomicAdd(&sums[gridDim.y], (double)cnt);
  }
}

template <typename T>
__global__ void k_l2_apply(const T* __restrict__ rv, const T* __restrict__ wgtp, T* __restrict__ wgt, int64_t nvis,
                           const double* __restrict__ ovar, double dof, double numer) {
  int c = blockIdx.y;
  const T* r = rv + (int64_t)c * nvis * 2;
  const T* p = wgtp ? wgtp + (int64_t)c * nvis : nullptr;
  T* w = wgt + (int64_t)c * nvis;
  const double ov = ovar[c];  // ovar, the ratio and the product are float64 in the reference also for float32 data
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nvis; k += (int64_t)gridDim.x * blockDim.x) {
    T re = r[2 * k], im = r[2 * k + 1];
    T q = p ? (re * p[k]) * re + (im * p[k]) * im : re * re + im * im;
    w[k] = (T)((double)w[k] * (numer / (dof + (double)q / ov)));
  }
}


// ---------------------------------------------------------------------------
// Visibility / weight preparation of one correlation behind diagonal Jones terms (`pfb init`,
// utils/correlations.py:195-232): for row r of time bin t with antennas (p, q) and channel f
//   wgt[r, f] = Re( w0 gp gq conj(gp) conj(gq) )        vis[r, f] = w0 gq v0 conj(gp)
// with gp = jones[t, p, f, 0, 0], gq = jones[t, q, f, 0, 0], (v0, w0) = correlation 0 of data / weight.
// The products are formed in the reference's order, every operation rounded on its own (no FMA contraction), so the
// result is bit-identical to the numba loop.  HBM bound: (2 + ncorr) p + ... in, 3p out per sample.
// ---------------------------------------------------------------------------
template <typename T> struct wd_ops;
template <> struct wd_ops<float> {
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
};
template <> struct wd_ops<double> {
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
};
template <typename T, typename C2>
__device__ __forceinline__ C2 wd_cmul(C2 a, C2 b) {  // (ac - bd) + i (ad + bc), four products, two sums
  using O = wd_ops<T>;
  C2 r;
  r.x = O::sub(O::mul(a.x, b.x), O::mul(a.y, b.y));
  r.y = O::add(O::mul(a.x, b.y), O::mul(a.y, b.x));
  return r;
}

template <typename T>
__global__ void k_weight_data_corr(const typename cplx_of<T>::type* __restrict__ data, const T* __restrict__ weight,
                                   const typename cplx_of<T>::type* __restrict__ jones, const int32_t* __restrict__ row_t,
                                   const int32_t* __restrict__ ant1, const int32_t* __restrict__ ant2, int64_t nrow,
                                   int nchan, int ncorr, int64_t js_t, int64_t js_a, int64_t js_c,
                                   typename cplx_of<T>::type* __restrict__ vis, T* __restrict__ wgt) {
  using C2 = typename cplx_of<T>::type;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrow * nchan) return;
  const int64_t row = i / nchan;
  const int chan = (int)(i - row * nchan);
  const int t = row_t[row];
  if (t < 0) return;  // a row outside every time bin keeps the zeros it was initialised with
  const C2 gp = jones[t * js_t + ant1[row] * js_a + chan * js_c];
  const C2 gq = jones[t * js_t + ant2[row] * js_a + chan * js_c];
  const T w0 = weight[i * ncorr];
  const C2 v0 = data[i * ncorr];
  C2 w0c; w0c.x = w0; w0c.y = (T)0;  // the reference multiplies by the real weight as a complex number
  const C2 gpc = {gp.x, -gp.y}, gqc = {gq.x, -gq.y};
  C2 a = wd_cmul<T, C2>(w0c, gp);
  a = wd_cmul<T, C2>(a, gq);
  a = wd_cmul<T, C2>(a, gpc);
  a = wd_cmul<T, C2>(a, gqc);
  wgt[i] = a.x;
  C2 b = wd_cmul<T, C2>(w0c, gq);
  b = wd_cmul<T, C2>(b, v0);
  b = wd_cmul<T, C2>(b, gpc);
  vis[i] = b;
}
