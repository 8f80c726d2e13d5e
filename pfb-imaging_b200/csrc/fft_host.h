// Host-side tables of the shared-memory FFT engine (fft.cuh): radix plans, digit-reversal tables, twiddles and the
// row-pass CTA size, used by the plane transforms (pfbgrid.cu), the PSF convolver (psfconv.cu) and the engine unit
// tests (colsfft.cu).
#pragma once
#include <cmath>
#include <vector>

#include "fft.cuh"

static constexpr size_t kMaxSmem = 232448;  // 227 KB opt-in dynamic shared memory per CTA on sm_100

// maxr: largest power-of-two radix (16 in fp32; 8 in fp64, whose radix-16 butterfly needs ~250 registers and
// leaves one 8-warp CTA per SM)
inline bool factorize(int n, FftDesc& d, int maxr = 16) {
  d.n = n;
  d.nstage = 0;
  int m = n;
  const int odd[4] = {11, 7, 5, 3};
  for (int r : odd)
    while (m % r == 0) {
      if (d.nstage >= FFT_MAX_STAGES) return false;
      d.radix[d.nstage++] = r;
      m /= r;
    }
  int a = 0;
  while (m % 2 == 0) { m /= 2; ++a; }
  if (m != 1) return false;
  const int lg = maxr >= 16 ? 4 : 3;
  while (a >= lg) {
    if (d.nstage >= FFT_MAX_STAGES) return false;
    d.radix[d.nstage++] = 1 << lg;
    a -= lg;
  }
  if (a > 0) {
    if (d.nstage >= FFT_MAX_STAGES) return false;
    d.radix[d.nstage++] = 1 << a;
  }
  return true;
}

inline void digit_tables(const FftDesc& d, std::vector<int>& rev, std::vector<int>& pos) {
  rev.assign(d.n, 0);
  pos.assign(d.n, 0);
  for (int k = 0; k < d.n; ++k) {
    int kk = k, M = d.n, p = 0;
    for (int s = 0; s < d.nstage; ++s) {
      M /= d.radix[s];
      p += (kk % d.radix[s]) * M;
      kk /= d.radix[s];
    }
    pos[k] = p;
    rev[p] = k;
  }
}

// exp(-2 pi i t / n), t < n, evaluated in fp64 and rounded to T
template <typename T>
std::vector<cx2<T>> twiddles(int n) {
  std::vector<cx2<T>> tw(n);
  for (int t = 0; t < n; ++t) {
    double ang = -2.0 * M_PI * (double)t / (double)n;
    tw[t].x = (T)cos(ang);
    tw[t].y = (T)sin(ang);
  }
  return tw;
}

// threads per CTA for a row transform: the multiple of 32 (<= cap, >= cap/2) that balances the
// radix-16 stage best (n/16 butterflies)
inline int row_threads(int n, int cap, int radix = 16) {
  int nb = n / radix, best = cap;
  double best_eff = 0.0;
  for (int t = cap; t >= cap / 2; t -= 32) {
    int per = (nb + t - 1) / t;
    double eff = (double)nb / ((double)per * t);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = t; }
  }
  return best;
}
