// Clark CLEAN minor cycle on the device (the backward step of `pfb kclean`, reference core/kclean.py:203-218 ->
// deconv/clark.py).  fp64 only; images (nband, nx, ny), raster index p = i*ny + j; contract restated in
// oracle/clark_np.py.  Per major iteration:
//   k_clark_search + k_clark_best   s(p) = |sum_b R_b(p)| (band order) on masked pixels, global max
//   cub::DeviceSelect::If            active set A = {p : s(p) >= subpf Rmax} in raster order
//   k_clark_gather                   R_b(A) into a band-major SoA, s(A), (i, j)(A)
//   k_clark_subminor                 the serial subminor loop in ONE cooperative launch, one grid.sync per component
//   k_clark_replay                   the component log into the model, in log order (no atomics)
// The residual step R = ID - PSF (*) model runs through the PSF convolver (psfconv.cuh) and k_clark_resid.
// Every multiply / add / subtract that the contract spells out uses __dmul_rn / __dadd_rn / __dsub_rn so that no
// FMA contraction changes its rounding (the numpy restatement rounds each operation).
#pragma once
#include <cooperative_groups.h>

#include <climits>
#include <cstdint>

constexpr int CLK_THREADS = 256;

// (s, index) order of the search: larger s wins, equal s goes to the smaller (raster-earlier) index — numpy argmax
__device__ __forceinline__ bool clk_better(double s, int i, double bs, int bi) { return s > bs || (s == bs && i < bi); }

__device__ __forceinline__ void clk_warp_best(double& s, int& i) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const double so = __shfl_down_sync(0xffffffffu, s, o);
    const int io = __shfl_down_sync(0xffffffffu, i, o);
    if (clk_better(so, io, s, i)) { s = so; i = io; }
  }
}

// block-wide best (s, i), returned to every thread; red_s / red_i are shared arrays of 32
__device__ __forceinline__ void clk_block_best(double& s, int& i, double* red_s, int* red_i) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  clk_warp_best(s, i);
  if (lane == 0) { red_s[w] = s; red_i[w] = i; }
  __syncthreads();
  if (w == 0) {
    s = lane < nw ? red_s[lane] : -1.0;
    i = lane < nw ? red_i[lane] : INT_MAX;
    clk_warp_best(s, i);
    if (lane == 0) { red_s[0] = s; red_i[0] = i; }
  }
  __syncthreads();
  s = red_s[0];
  i = red_i[0];
  __syncthreads();  // red_* may be reused
}

// s(p) for every pixel (-1 where the mask excludes it: never selected, never the maximum) and one (s, p) candidate
// per CTA
__global__ void __launch_bounds__(CLK_THREADS) k_clark_search(const double* __restrict__ R, int nband, int npix,
                                                              const uint8_t* __restrict__ mask, double* __restrict__ s,
                                                              double* __restrict__ cand_s, int* __restrict__ cand_i) {
  __shared__ double red_s[32];
  __shared__ int red_i[32];
  double bs = -1.0;
  int bi = INT_MAX;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += gridDim.x * blockDim.x) {
    double v = -1.0;
    if (!mask || mask[p]) {
      double acc = R[p];
      for (int b = 1; b < nband; ++b) acc = __dadd_rn(acc, R[(int64_t)b * npix + p]);
      v = fabs(acc);
      if (clk_better(v, p, bs, bi)) { bs = v; bi = p; }
    }
    s[p] = v;
  }
  clk_block_best(bs, bi, red_s, red_i);
  if (threadIdx.x == 0) { cand_s[blockIdx.x] = bs; cand_i[blockIdx.x] = bi; }
}

// one CTA: the best of n candidates -> best_s[0], best_i[0]
__global__ void __launch_bounds__(CLK_THREADS) k_clark_best(const double* __restrict__ cand_s, const int* __restrict__ cand_i,
                                                            int n, double* __restrict__ best_s, int* __restrict__ best_i) {
  __shared__ double red_s[32];
  __shared__ int red_i[32];
  double bs = -1.0;
  int bi = INT_MAX;
  for (int k = threadIdx.x; k < n; k += blockDim.x)
    if (clk_better(cand_s[k], cand_i[k], bs, bi)) { bs = cand_s[k]; bi = cand_i[k]; }
  clk_block_best(bs, bi, red_s, red_i);
  if (threadIdx.x == 0) { *best_s = bs; *best_i = bi; }
}

// selection predicate of the active set (masked-out pixels carry s = -1 < thr)
struct ClarkActive {
  const double* s;
  double thr;
  __device__ __forceinline__ bool operator()(int p) const { return s[p] >= thr; }
};

__global__ void k_clark_gather(const double* __restrict__ R, const double* __restrict__ s, int nband, int npix, int ny,
                               const int* __restrict__ idx, int nA, double* __restrict__ RA, double* __restrict__ SA,
                               int2* __restrict__ ij) {
  for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < nA; a += gridDim.x * blockDim.x) {
    const int p = idx[a];
    ij[a] = make_int2(p / ny, p % ny);
    SA[a] = s[p];
    for (int b = 0; b < nband; ++b) RA[(int64_t)b * nA + a] = R[(int64_t)b * npix + p];
  }
}

struct ClarkSub {
  double* RA;          // (nband, nA) residual of the active set
  double* SA;          // (nA) its search value
  const int2* ij;      // (nA) pixel coordinates
  int nA, nband, ny;
  const double* psf;   // (nband, nxp, nyp)
  const double* peak;  // (nband) PSF centre values
  int nxp, nyp, cx, cy;
  double gamma, thr;   // thr = max(subpf Rmax, threshold)
  int submaxit;
  double* slot_s;      // (2, grid) per-CTA candidates, double-buffered by iteration parity
  int* slot_a;         // (2, grid)
  double* slot_r;      // (2, grid, nband) R_b at each CTA's candidate
  int* log_p;          // (submaxit) raster index of each component
  double* log_d;       // (submaxit, nband) its d_b
  int* count;          // number of components
};

// The subminor loop.  Entry a belongs to thread a mod (grid threads) for the whole launch, so RA / SA need no
// synchronisation; pass `it` subtracts component it-1 from the thread's entries inside its PSF support and tracks the
// best (s, a) in the same sweep.  After the grid sync every CTA reduces ALL candidate slots itself and so reaches the
// same a*, the same d_b and the same stop decision: the control flow is identical in every CTA (one that left the
// loop alone would deadlock grid.sync), and the loop is bounded by submaxit.
__global__ void __launch_bounds__(CLK_THREADS) k_clark_subminor(ClarkSub c) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  extern __shared__ double d_sh[];  // d_b of the previous component
  __shared__ double red_s[32];
  __shared__ int red_i[32];
  const int nthr = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t plane = (int64_t)c.nxp * c.nyp;
  int pi = 0, pj = 0;
  bool have = false;
  for (int it = 0;; ++it) {
    const int64_t slot = (int64_t)(it & 1) * gridDim.x;
    double bs = -1.0;
    int bi = INT_MAX;
    for (int a = t0; a < c.nA; a += nthr) {
      double sv;
      const int2 q = c.ij[a];
      const int x = c.cx + q.x - pi, y = c.cy + q.y - pj;
      if (have && (unsigned)x < (unsigned)c.nxp && (unsigned)y < (unsigned)c.nyp) {
        const double* pp = c.psf + (int64_t)x * c.nyp + y;
        double acc = 0.0;
        for (int b = 0; b < c.nband; ++b) {
          double* r = c.RA + (int64_t)b * c.nA + a;
          const double v = __dsub_rn(*r, __dmul_rn(d_sh[b], pp[b * plane]));
          *r = v;
          acc = b == 0 ? v : __dadd_rn(acc, v);
        }
        sv = fabs(acc);
        c.SA[a] = sv;
      } else {
        sv = c.SA[a];
      }
      if (clk_better(sv, a, bs, bi)) { bs = sv; bi = a; }
    }
    clk_block_best(bs, bi, red_s, red_i);  // its barriers also make this CTA's RA writes visible to its own threads
    if (threadIdx.x == 0) { c.slot_s[slot + blockIdx.x] = bs; c.slot_a[slot + blockIdx.x] = bi; }
    if (bi != INT_MAX)
      for (int b = threadIdx.x; b < c.nband; b += blockDim.x) c.slot_r[(slot + blockIdx.x) * c.nband + b] = c.RA[(int64_t)b * c.nA + bi];
    grid.sync();
    bs = -1.0;
    bi = INT_MAX;
    for (int k = threadIdx.x; k < gridDim.x; k += blockDim.x) {
      const double so = c.slot_s[slot + k];
      const int io = c.slot_a[slot + k];
      if (clk_better(so, io, bs, bi)) { bs = so; bi = io; }
    }
    clk_block_best(bs, bi, red_s, red_i);
    if (!(bs > c.thr) || it >= c.submaxit) {
      if (blockIdx.x == 0 && threadIdx.x == 0) *c.count = it;
      break;
    }
    const int owner = (bi % nthr) / blockDim.x;  // the CTA whose slot holds R_b(a*)
    const int2 q = c.ij[bi];
    for (int b = threadIdx.x; b < c.nband; b += blockDim.x) {
      const double pk = c.peak[b];
      const double d = pk > 0.0 ? __ddiv_rn(__dmul_rn(c.gamma, c.slot_r[(slot + owner) * c.nband + b]), pk) : 0.0;
      d_sh[b] = d;
      if (blockIdx.x == 0) c.log_d[(int64_t)it * c.nband + b] = d;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) c.log_p[it] = q.x * c.ny + q.y;
    pi = q.x;
    pj = q.y;
    have = true;
    __syncthreads();
  }
}

// model_b(p_k) += d_{k,b} for k in log order; one thread per band
__global__ void k_clark_replay(double* __restrict__ model, int nband, int npix, const int* __restrict__ log_p,
                               const double* __restrict__ log_d, const int* __restrict__ count) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nband) return;
  const int n = *count;
  double* m = model + (int64_t)b * npix;
  for (int k = 0; k < n; ++k) {
    const int p = log_p[k];
    m[p] = __dadd_rn(m[p], log_d[(int64_t)k * nband + b]);
  }
}

// R = ID - R, where R holds PSF (*) model on entry
__global__ void k_clark_resid(const double* __restrict__ ID, double* __restrict__ R, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    R[i] = __dsub_rn(ID[i], R[i]);
}
