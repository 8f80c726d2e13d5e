// Batched conjugate gradients on the PSF-convolution Hessian (pfbs_psf_cg): the vector work of solvers.pcg
// (solvers.py:35-82, no preconditioner) for every band of a cube in one launch per step.  Band = blockIdx.y; each band
// keeps its own scalars in a CgCtl, and a band whose `stop` is set is skipped by every kernel (frozen).
//
// Reductions are deterministic: each CTA writes its partial sums (grid-stride serial sum, then a fixed shuffle tree),
// and one CTA per band adds the partials in a fixed order.  No floating-point atomics, so two runs give the same bits.
// The element-wise updates round as numpy does (product, then sum: no FMA contraction), so the device iterates differ
// from the host ones only through the order of the dot-product sums.
#pragma once
#include <cstdint>

enum { CG_RUNNING = 0, CG_CONVERGED = 1, CG_MAXIT = 2, CG_STALLED = 3, CG_ZERO = 4, CG_EXACT = 5 };

struct CgCtl {
  double rho;    // r.r of the current residual
  double alpha;  // rho / p.Ap of this iteration
  double beta;   // rho' / rho
  double eps;    // |alpha| ||p|| / ||x||
  double pp;     // p.p of this iteration
  int k, stalls, stop, pad;
};

constexpr int CG_THREADS = 256;
constexpr int CG_GMAX = 1024;  // partial sums per band and quantity

// sum of a and b over the CTA (result valid in thread 0); fixed order
__device__ __forceinline__ void cg_block_sum2(double& a, double& b) {
  __shared__ double sh[2][CG_THREADS / 32];
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_down_sync(0xffffffffu, a, o);
    b += __shfl_down_sync(0xffffffffu, b, o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { sh[0][w] = a; sh[1][w] = b; }
  __syncthreads();
  if (w == 0) {
    a = lane < CG_THREADS / 32 ? sh[0][lane] : 0.0;
    b = lane < CG_THREADS / 32 ? sh[1][lane] : 0.0;
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_down_sync(0xffffffffu, a, o);
      b += __shfl_down_sync(0xffffffffu, b, o);
    }
  }
}

// the loop condition of pcg, and which of its three exits was taken when it fails
__device__ __forceinline__ int cg_stop_code(const CgCtl& c, double tol, int maxit, int minit) {
  if ((c.eps > tol || c.k < minit) && c.k < maxit && c.stalls < 5) return CG_RUNNING;
  return c.k >= maxit ? CG_MAXIT : c.stalls >= 5 ? CG_STALLED : CG_CONVERGED;
}

// partial sums of one band: part[(b * G + cta) * 2 + {0, 1}]
__device__ __forceinline__ void cg_put2(double* part, int G, double a, double b) {
  cg_block_sum2(a, b);
  if (threadIdx.x == 0) {
    double* q = part + ((int64_t)blockIdx.y * G + blockIdx.x) * 2;
    q[0] = a;
    q[1] = b;
  }
}

// fixed-order sum of band blockIdx.x's G partial pairs (valid in thread 0)
__device__ __forceinline__ void cg_get2(const double* part, int G, double& a, double& b) {
  a = 0.0; b = 0.0;
  const double* q = part + (int64_t)blockIdx.x * G * 2;
  for (int i = threadIdx.x; i < G; i += CG_THREADS) { a += q[2 * i]; b += q[2 * i + 1]; }
  cg_block_sum2(a, b);
}

#define CG_BAND_LOOP(i) for (int64_t i = (int64_t)blockIdx.x * CG_THREADS + threadIdx.x; i < npix; i += (int64_t)gridDim.x * CG_THREADS)

// r = A x - b (A x already in r), p = -r; partials of r.r
__global__ void __launch_bounds__(CG_THREADS) k_cg_init(const double* __restrict__ rhs, double* __restrict__ r,
                                                        double* __restrict__ p, int64_t npix, double* part) {
  const int64_t o = (int64_t)blockIdx.y * npix;
  double rr = 0.0, unused = 0.0;
  CG_BAND_LOOP(i) {
    const double v = __dsub_rn(r[o + i], rhs[o + i]);
    r[o + i] = v;
    p[o + i] = -v;
    rr += v * v;
  }
  cg_put2(part, gridDim.x, rr, unused);
}

__global__ void __launch_bounds__(CG_THREADS) k_cg_init_fin(CgCtl* ctl, const double* part, int G, double tol,
                                                            int maxit, int minit) {
  double rr, unused;
  cg_get2(part, G, rr, unused);
  if (threadIdx.x) return;
  CgCtl c{};
  c.rho = rr;
  if (!(rr > 0.0)) {
    c.stop = CG_ZERO;
  } else {
    c.eps = 1.0;
    c.stop = cg_stop_code(c, tol, maxit, minit);
  }
  ctl[blockIdx.x] = c;
}

// partials of p.Ap and p.p
__global__ void __launch_bounds__(CG_THREADS) k_cg_dots(const CgCtl* ctl, const double* __restrict__ p,
                                                        const double* __restrict__ ap, int64_t npix, double* part) {
  if (ctl[blockIdx.y].stop) return;
  const int64_t o = (int64_t)blockIdx.y * npix;
  double pap = 0.0, pp = 0.0;
  CG_BAND_LOOP(i) {
    const double pv = p[o + i];
    pap += pv * ap[o + i];
    pp += pv * pv;
  }
  cg_put2(part, gridDim.x, pap, pp);
}

// alpha = rho / p.Ap, or the exact stop of pcg (rho == 0 and p.Ap == 0: the iterate is already the solution)
__global__ void __launch_bounds__(CG_THREADS) k_cg_dots_fin(CgCtl* ctl, const double* part, int G) {
  if (ctl[blockIdx.x].stop) return;
  double pap, pp;
  cg_get2(part, G, pap, pp);
  if (threadIdx.x) return;
  CgCtl& c = ctl[blockIdx.x];
  if (c.rho == 0.0 && pap == 0.0) {
    c.stop = CG_EXACT;
    return;
  }
  c.alpha = c.rho / pap;
  c.pp = pp;
}

// x += alpha p, r += alpha Ap; partials of r.r and x.x
__global__ void __launch_bounds__(CG_THREADS) k_cg_update(const CgCtl* ctl, double* __restrict__ x,
                                                          double* __restrict__ r, const double* __restrict__ p,
                                                          const double* __restrict__ ap, int64_t npix, double* part) {
  if (ctl[blockIdx.y].stop) return;
  const double alpha = ctl[blockIdx.y].alpha;
  const int64_t o = (int64_t)blockIdx.y * npix;
  double rr = 0.0, xx = 0.0;
  CG_BAND_LOOP(i) {
    const double xv = __dadd_rn(x[o + i], __dmul_rn(alpha, p[o + i]));
    const double rv = __dadd_rn(r[o + i], __dmul_rn(alpha, ap[o + i]));
    x[o + i] = xv;
    r[o + i] = rv;
    rr += rv * rv;
    xx += xv * xv;
  }
  cg_put2(part, gridDim.x, rr, xx);
}

// rho' and beta, eps = |alpha| ||p|| / ||x|| (0 when ||x|| = 0), the stall count and the loop condition
__global__ void __launch_bounds__(CG_THREADS) k_cg_update_fin(CgCtl* ctl, const double* part, int G, double tol,
                                                              int maxit, int minit) {
  if (ctl[blockIdx.x].stop) return;
  double rr, xx;
  cg_get2(part, G, rr, xx);
  if (threadIdx.x) return;
  CgCtl c = ctl[blockIdx.x];
  c.beta = rr / c.rho;
  c.rho = rr;
  c.k += 1;
  const double eps_prev = c.eps;
  c.eps = xx > 0.0 ? fabs(c.alpha) * sqrt(c.pp / xx) : 0.0;
  if (fabs(eps_prev - c.eps) < 1e-3 * tol) c.stalls += 1;
  c.stop = cg_stop_code(c, tol, maxit, minit);
  ctl[blockIdx.x] = c;
}

// p = beta p - r
__global__ void __launch_bounds__(CG_THREADS) k_cg_direction(const CgCtl* ctl, double* __restrict__ p,
                                                             const double* __restrict__ r, int64_t npix) {
  if (ctl[blockIdx.y].stop) return;
  const double beta = ctl[blockIdx.y].beta;
  const int64_t o = (int64_t)blockIdx.y * npix;
  CG_BAND_LOOP(i) p[o + i] = __dsub_rn(__dmul_rn(beta, p[o + i]), r[o + i]);
}

#undef CG_BAND_LOOP
