// PSF-convolution Hessian on the device (SURVEY §8 f1): the operator pfb-imaging iterates inside
// pcg / power method / primal-dual,
//     out = beam * crop( IFFT( FFT( pad(beam * x) ) * khat ) ) + eta * x
// (/root/reference/src/pfb_imaging/operators/hessian.py:103-143 hessian_psf_slice,
//  operators/psf.py:8-31 psf_convolve_slice), built from the same shared-memory FFT engine as the
// plane transforms: a row pass, ONE column kernel that transforms, multiplies and transforms back
// without leaving shared memory (DIF forward -> multiply in digit-reversed order -> DIT inverse), and
// a row pass back.  The zero-padded rows / columns are never read or written.
#pragma once
#include "fft.cuh"

struct ConvTabs {
  FftDesc du, dv;      // along u (length nxp) and v (length nyp)
  const void* tw_u;
  const void* tw_v;
  const int* rev_u;
  const int* rev_v;
  const int* pos_v;
  int nx, ny, nxp, nyp;
};

// image rows -> tmp (nx, nyp): FFT along v of the zero-padded rows, image placed at columns 0..ny-1.
// The rows are real, so TWO of them share one complex transform: z = x_a + i x_b,
//   X_a[l] = (Z[l] + conj Z[N-l]) / 2,   X_b[l] = (Z[l] - conj Z[N-l]) / (2i),
// and only the half spectrum l <= nyp/2 is written (column nyp - l of every later stage is the conjugate of column l
// because x and the kernel are real).  CTA i handles rows 2i and 2i+1.
template <typename T>
__global__ void __launch_bounds__(256, (sizeof(T) == 4 ? 3 : 2))
k_conv_rows_fwd(ConvTabs ct, const T* __restrict__ x, const T* __restrict__ beam, cx2<T>* __restrict__ tmp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int ia = 2 * blockIdx.x, ib = ia + 1;
  const bool has_b = ib < ct.nx;
  for (int n = tid; n < ct.nyp; n += nthr) s[fft_pad<T>(n)] = {(T)0, (T)0};
  __syncthreads();
  constexpr int U = 4;
  const int64_t ra = (int64_t)ia * ct.ny, rb = (int64_t)ib * ct.ny;
  for (int j0 = tid; j0 < ct.ny; j0 += U * nthr) {
    T va[U], vb[U];
    int pv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = j0 + u * nthr;
      if (j < ct.ny) {
        va[u] = x[ra + j];
        vb[u] = has_b ? x[rb + j] : (T)0;
        if (beam) { va[u] *= beam[ra + j]; if (has_b) vb[u] *= beam[rb + j]; }
        pv[u] = ct.pos_v[j];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (j0 + u * nthr < ct.ny) s[fft_pad<T>(pv[u])] = {va[u], vb[u]};
  }
  __syncthreads();
  fft_dit<T, 1>(s, (const cx2<T>*)ct.tw_v, ct.dv, tid, nthr);
  cx2<T>* da = tmp + (int64_t)ia * ct.nyp;
  cx2<T>* db = tmp + (int64_t)ib * ct.nyp;
  const int nkeep = min(ct.nyp, ((ct.nyp / 2 + 1 + 3) / 4) * 4);  // half spectrum, rounded up to a column block
#pragma unroll 2
  for (int l = tid; l < nkeep; l += nthr) {
    const cx2<T> zl = s[fft_pad<T>(l)], zm = s[fft_pad<T>(l == 0 ? 0 : ct.nyp - l)];
    da[l] = {(T)0.5 * (zl.x + zm.x), (T)0.5 * (zl.y - zm.y)};
    if (has_b) db[l] = {(T)0.5 * (zl.y + zm.y), (T)0.5 * (zm.x - zl.x)};
  }
}

// The multiplier of the column pass at spectral cell (k, b0 + c): k is the row of the full spectrum (the digit-reversed
// position already resolved), b0 + c the column.  KhatMul reads the stored spectrum; GaussMul evaluates the transfer
// function of a pixel-sampled Gaussian where it is used, so nothing is stored.
struct KhatMul {
  template <typename T>
  __device__ __forceinline__ cx2<T> operator()(const ConvTabs& ct, const cx2<T>* __restrict__ khat, int k, int b0,
                                               int c) const {
    return khat[(int64_t)k * ct.nyp + b0 + c];
  }
};

// DFT on the padded grid of the periodised, pixel-sampled Gaussian g(x) = exp(-x^T S^-1 x / 2), by Poisson summation:
//     K(f) = amp * sum_{m in Z^2, |m_i| <= M} exp(q(f + m)),   q(f) = -2 pi^2 f^T S f,
// f = (k~ / nxp, l~ / nyp) the signed frequencies.  q[] holds (-2 pi^2 S00, -4 pi^2 S01, -2 pi^2 S11), so
// q(f) = q[0] fx^2 + q[1] fx fy + q[2] fy^2.  Every alias term is the exp of its own exponent (a product of separately
// exponentiated factors overflows for wide beams).  ratio != 0: K_to / K_from, each sum scaled by the exp of its
// largest exponent (the m = 0 term whenever f is S-nearest to the origin), so that neither sum underflows and the
// quotient of the two scales, exp(qmax_to - qmax_from) <= 1 for S_to - S_from positive semi-definite, cannot overflow.
struct GaussMul {
  double q_to[3], q_from[3];
  double amp;  // plain: 2 pi sqrt(det S) (peak 1) or 1 / sum (unit sum); ratio: amp_to / amp_from
  int M, ratio;

  __device__ __forceinline__ double qform(const double* q, double fx, double fy) const {
    return q[0] * fx * fx + q[1] * fx * fy + q[2] * fy * fy;
  }
  // sum_m exp(q(f + m) - shift), shift = max_m q(f + m) when scaled
  __device__ __forceinline__ double alias_sum(const double* q, double fx, double fy, bool scaled, double& shift) const {
    shift = 0.0;
    if (scaled) {
      shift = -INFINITY;
      for (int mx = -M; mx <= M; ++mx)
        for (int my = -M; my <= M; ++my) shift = fmax(shift, qform(q, fx + mx, fy + my));
    }
    double acc = 0.0;
    for (int mx = -M; mx <= M; ++mx)
      for (int my = -M; my <= M; ++my) acc += exp(qform(q, fx + mx, fy + my) - shift);
    return acc;
  }
  template <typename T>
  __device__ __forceinline__ cx2<T> operator()(const ConvTabs& ct, const cx2<T>* __restrict__, int k, int b0,
                                               int c) const {
    const int l = b0 + c;
    const double fx = (double)(2 * k > ct.nxp ? k - ct.nxp : k) / (double)ct.nxp;
    const double fy = (double)(2 * l > ct.nyp ? l - ct.nyp : l) / (double)ct.nyp;
    double v;
    if (!ratio) {
      double s0;
      v = amp * alias_sum(q_to, fx, fy, false, s0);
    } else {
      double st, sf;
      const double nt = alias_sum(q_to, fx, fy, true, st);
      const double nf = alias_sum(q_from, fx, fy, true, sf);
      v = amp * exp(st - sf) * (nt / nf);
    }
    return {(T)v, (T)0};
  }
};

// (Re khat + c) or its reciprocal as a real multiplier: the direct inverse of the Hessian (hess_direct_slice) from the
// convolver's own spectrum, without a second stored one.  fp64 sum and IEEE quotient, the doubles numpy forms.
struct ShiftMul {
  double c;
  int inverse;
  template <typename T>
  __device__ __forceinline__ cx2<T> operator()(const ConvTabs& ct, const cx2<T>* __restrict__ khat, int k, int b0,
                                               int col) const {
    const double v = (double)khat[(int64_t)k * ct.nyp + b0 + col].x + c;
    return {(T)(inverse ? 1.0 / v : v), (T)0};
  }
};

// column block: forward along u, multiply by mul(k, b), inverse along u, keep rows < nx
template <typename T, int C, class Mul>
__global__ void __launch_bounds__(512)
k_conv_cols(ConvTabs ct, const cx2<T>* __restrict__ khat, cx2<T>* __restrict__ tmp, Mul mul) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int b0 = blockIdx.x * C;
  cx2<T>* g = tmp + b0;
  constexpr int U = 8;
  for (int w = ct.nx * C + tid; w < ct.nxp * C; w += nthr) s[fft_pad<T>(w)] = {(T)0, (T)0};
  for (int w0 = tid; w0 < ct.nx * C; w0 += U * nthr) {
    cx2<T> v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int w = w0 + u * nthr;
      if (w < ct.nx * C) v[u] = g[(int64_t)(w / C) * ct.nyp + (w % C)];
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int w = w0 + u * nthr;
      if (w < ct.nx * C) s[fft_pad<T>(w)] = v[u];
    }
  }
  __syncthreads();
  fft_dif<T, C>(s, (const cx2<T>*)ct.tw_u, ct.du, tid, nthr);
  for (int w0 = tid; w0 < ct.nxp * C; w0 += U * nthr) {
    cx2<T> kv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int w = w0 + u * nthr;
      if (w < ct.nxp * C) kv[u] = mul(ct, khat, ct.rev_u[w / C], b0, w % C);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int w = w0 + u * nthr;
      if (w < ct.nxp * C) {
        cx2<T> v = cmul(s[fft_pad<T>(w)], kv[u]);
        v.y = -v.y;  // conj: the inverse transform is conj o forward o conj
        s[fft_pad<T>(w)] = v;
      }
    }
  }
  __syncthreads();
  fft_dit<T, C>(s, (const cx2<T>*)ct.tw_u, ct.du, tid, nthr);
  for (int w = tid; w < ct.nx * C; w += nthr) {
    const int a = w / C, c = w - a * C;
    cx2<T> v = s[fft_pad<T>(w)];
    v.y = -v.y;
    g[(int64_t)a * ct.nyp + c] = v;
  }
}

// tmp rows -> image: inverse FFT along v, crop, normalise, beam, ridge.  Two rows per transform again: with the half
// spectra Y_a, Y_b of the two (real) output rows, S[l] = Y_a[l] + i Y_b[l], S[N-l] = conj Y_a[l] + i conj Y_b[l], and
// the inverse transform of S is y_a + i y_b.  (The inverse is evaluated as conj o forward o conj.)
template <typename T>
__global__ void __launch_bounds__(256, (sizeof(T) == 4 ? 3 : 2))
k_conv_rows_inv(ConvTabs ct, const cx2<T>* __restrict__ tmp, const T* __restrict__ beam, const T* __restrict__ xin,
                double scale, double eta, T* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int ia = 2 * blockIdx.x, ib = ia + 1;
  const bool has_b = ib < ct.nx;
  const cx2<T>* sa = tmp + (int64_t)ia * ct.nyp;
  const cx2<T>* sb = tmp + (int64_t)ib * ct.nyp;
  const int nh = ct.nyp / 2;
#pragma unroll 2
  for (int l = tid; l <= nh; l += nthr) {
    const cx2<T> ya = sa[l];
    const cx2<T> yb = has_b ? sb[l] : cx2<T>{(T)0, (T)0};
    s[fft_pad<T>(l)] = {ya.x - yb.y, -(ya.y + yb.x)};                                   // conj S[l]
    if (l > 0 && 2 * l < ct.nyp) s[fft_pad<T>(ct.nyp - l)] = {ya.x + yb.y, ya.y - yb.x};  // conj S[N-l]
  }
  __syncthreads();
  fft_dif<T, 1>(s, (const cx2<T>*)ct.tw_v, ct.dv, tid, nthr);
  for (int j = tid; j < ct.ny; j += nthr) {
    const cx2<T> v = s[fft_pad<T>(ct.pos_v[j])];  // conj of the inverse transform: (y_a, -y_b)
    {
      const int64_t pix = (int64_t)ia * ct.ny + j;
      double r = (double)v.x * scale;
      if (beam) r *= (double)beam[pix];
      if (xin) r += eta * (double)xin[pix];
      out[pix] = (T)r;
    }
    if (has_b) {
      const int64_t pix = (int64_t)ib * ct.ny + j;
      double r = -(double)v.y * scale;
      if (beam) r *= (double)beam[pix];
      if (xin) r += eta * (double)xin[pix];
      out[pix] = (T)r;
    }
  }
}

// khat_full[k][l] from the half spectrum (nxp, nyp/2+1) of a real kernel: Hermitian mirror
template <typename T>
__global__ void k_expand_half(int nxp, int nyp, const cx2<T>* __restrict__ half, cx2<T>* __restrict__ full) {
  int l = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
  if (l >= nyp) return;
  const int nh = nyp / 2 + 1;
  cx2<T> v;
  if (l < nh) v = half[(int64_t)k * nh + l];
  else {
    const int km = k == 0 ? 0 : nxp - k;
    v = half[(int64_t)km * nh + (nyp - l)];
    v.y = -v.y;
  }
  full[(int64_t)k * nyp + l] = v;
}

// Hermitian part of a full spectrum: Re(IFFT(FFT(x) k)) for real x only sees (k[a,b] + conj k[-a,-b]) / 2, which is
// what the half-column evaluation above assumes.  out may not alias in.
template <typename T>
__global__ void k_hermitize(int nxp, int nyp, const cx2<T>* __restrict__ in, cx2<T>* __restrict__ out) {
  int l = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
  if (l >= nyp) return;
  const int km = k == 0 ? 0 : nxp - k, lm = l == 0 ? 0 : nyp - l;
  const cx2<T> a = in[(int64_t)k * nyp + l], b = in[(int64_t)km * nyp + lm];
  out[(int64_t)k * nyp + l] = {(T)0.5 * (a.x + b.x), (T)0.5 * (a.y - b.y)};
}
