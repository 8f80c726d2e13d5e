// Row passes of the fused plane transforms on the pair engine (fft2.cuh): one CTA transforms the SAME image row of
// TWO neighbouring w-planes (q, q + 1) as one packed transform.
//   * the image row, the correction, the beam and the n-1 table are read once for both planes (they were read once
//     per plane by k_rows_fwd / k_rows_inv of fused_fft.cuh),
//   * the butterflies run two-wide (FADD2 / FMUL2 / FFMA2): half the math instructions per plane,
//   * the grid direction adds the two planes' contributions to the fp64 image with ONE RED.F64 per pixel instead of two.
// Shared memory: nv pair elements of 16 bytes {re_q, re_q+1, im_q, im_q+1} (XOR-swizzled) + the two-level twiddle table;
// two CTAs per SM at nv = 6144.  A launch covers an even number of planes (the last plane of an odd count goes to the
// one-plane kernel).
//
//   k_rows2_fwd (degrid direction): pad + beam + correction + w-screen of both planes built in shared memory at the
//                                   digit-reversed positions, DIT transform (natural-order output), the active columns
//                                   of the two grid rows written
//   k_rows2_inv (grid direction)  : the active columns of the two grid rows read (swap-in = inverse transform), DIF,
//                                   conjugate screens applied to the ny kept outputs, real parts summed and added to
//                                   the fp64 accumulation image
#pragma once
#include "fused_common.cuh"
#include "fft2.cuh"

#define ROWS2_THREADS 192    // radix-16 stages: 128 registers per thread, two CTAs of 6 warps per SM

template <bool FAST>
__global__ void __launch_bounds__(ROWS2_THREADS, 2)
k_rows2_fwd(GParams p, FusedTabs ft, const float* __restrict__ x, const float* __restrict__ beam,
            const float* __restrict__ corr, float2* __restrict__ grid) {
  extern __shared__ __align__(1024) unsigned char smem_raw1k[];
  float4* s = reinterpret_cast<float4*>(smem_raw1k);
  const int tid = threadIdx.x, nthr = blockDim.x, i = blockIdx.y;
  const int nv = p.nv, hy = p.ny / 2;
  const FftDesc& dv = ft.dv;
  const int* __restrict__ pos_v = ft.pos_v;
  const int qa = 2 * blockIdx.x + ft.q0, qb = qa + 1;
  const P2Tw tw = p2_tw_fill(reinterpret_cast<float2*>(s + nv), (const float2*)ft.tw_v, nv, tid, nthr);
  const int ip = i - p.nx / 2;
  const int a = ip < 0 ? ip + p.nu : ip;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int n = tid; n < nv; n += nthr) s[n] = z;
  __syncthreads();
  const double wa = ft.plane_w ? ft.plane_w[qa] : p.w0 + qa * p.dw;
  const double wb = ft.plane_w ? ft.plane_w[qb] : p.w0 + qb * p.dw;
  const int64_t row = (int64_t)i * p.ny;
  const float* xa = x;
  const float* xb = x;
  const float* ba = beam;
  const float* bb = beam;
  if (ft.plane_img) {  // batched snapshots: every plane has its own image and beam
    const int64_t oa = (int64_t)ft.plane_img[qa] * p.nx * p.ny, ob = (int64_t)ft.plane_img[qb] * p.nx * p.ny;
    xa += oa;
    xb += ob;
    if (beam) { ba += oa; bb += ob; }
  }
  const bool same_x = xa == xb;  // (then ba == bb too)
  const bool vec_ok = (p.ny & 7) == 0 && (((uintptr_t)x | (uintptr_t)corr | (uintptr_t)beam) & 15) == 0;
  if (vec_ok) {
    // 4 consecutive pixels per step (hy % 4 == 0, so a group never straddles the wrap), two steps in flight
    const int ng = p.ny >> 2;
    for (int g0 = tid; g0 < ng; g0 += 2 * nthr) {
      float xv[2][4], yv[2][4], cv[2][4], bv[2][4], bw[2][4];
      double nuv[2][4];
      int pv[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int g = g0 + u * nthr;
        if (g < ng) {
          const int j = 4 * g;
          load4(xa + row + j, xv[u]);
          if (!same_x) load4(xb + row + j, yv[u]);
          load4(corr + row + j, cv[u]);
          if (beam) {
            load4(ba + row + j, bv[u]);
            if (!same_x) load4(bb + row + j, bw[u]);
          }
          if (p.do_wgridding) load4(ft.nutab + row + j, nuv[u]);
          const int jp = j - hy;
          load4(pos_v + (jp < 0 ? jp + nv : jp), pv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (g0 + u * nthr < ng) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float cb = cv[u][e], cbb = cb;
            if (beam) {
              cb *= bv[u][e];
              cbb = same_x ? cb : cbb * bw[u][e];
            }
            const float va = xv[u][e] * cb;
            const float vb = (same_x ? xv[u][e] : yv[u][e]) * cbb;
            if (va == 0.f && vb == 0.f) continue;  // the buffer is zero already
            float4 v = make_float4(va, vb, 0.f, 0.f);
            if (p.do_wgridding) {
              float ca, sa, c2, s2;
              cis_screen<FAST>(wa * nuv[u][e], ca, sa);
              cis_screen<FAST>(wb * nuv[u][e], c2, s2);
              v = make_float4(va * ca, vb * c2, va * sa, vb * s2);
            }
            s[sw2(pv[u][e])] = v;
          }
        }
      }
    }
  } else {
    for (int j = tid; j < p.ny; j += nthr) {
      const int64_t pix = row + j;
      const float c = corr[pix];
      const float va = xa[pix] * (beam ? c * ba[pix] : c), vb = xb[pix] * (beam ? c * bb[pix] : c);
      float4 v = make_float4(va, vb, 0.f, 0.f);
      if (p.do_wgridding) {
        float ca, sa, c2, s2;
        cis_screen<FAST>(wa * ft.nutab[pix], ca, sa);
        cis_screen<FAST>(wb * ft.nutab[pix], c2, s2);
        v = make_float4(va * ca, vb * c2, va * sa, vb * s2);
      }
      const int jp = j - hy;
      s[sw2(pos_v[jp < 0 ? jp + nv : jp])] = v;
    }
  }
  __syncthreads();
  p2_fft_dit<1>(s, tw, dv, tid, nthr);
  // only the active columns are written (window bounds are multiples of 32): two columns per step and plane
  float2* da = grid + ((int64_t)qa * p.nu + a) * nv;
  float2* db = grid + ((int64_t)qb * p.nu + a) * nv;
  const int npair = ft.b_len >> 1;
#pragma unroll 4
  for (int r = tid; r < npair; r += nthr) {
    int n = ft.b_lo + 2 * r;
    if (n >= nv) n -= nv;
    const float4 v0 = s[sw2(n)], v1 = s[sw2(n + 1)];  // {re_a, re_b, im_a, im_b}
    *reinterpret_cast<float4*>(da + n) = make_float4(v0.x, v0.z, v1.x, v1.z);
    *reinterpret_cast<float4*>(db + n) = make_float4(v0.y, v0.w, v1.y, v1.w);
  }
}

template <bool FAST>
__global__ void __launch_bounds__(ROWS2_THREADS, 2)
k_rows2_inv(GParams p, FusedTabs ft, const float2* __restrict__ grid, double* __restrict__ accimg) {
  extern __shared__ __align__(1024) unsigned char smem_raw1k[];
  float4* s = reinterpret_cast<float4*>(smem_raw1k);
  const int tid = threadIdx.x, nthr = blockDim.x, i = blockIdx.y;
  const int nv = p.nv, hy = p.ny / 2;
  const FftDesc& dv = ft.dv;
  const int* __restrict__ pos_v = ft.pos_v;
  const int qa = 2 * blockIdx.x + ft.q0, qb = qa + 1;
  const P2Tw tw = p2_tw_fill(reinterpret_cast<float2*>(s + nv), (const float2*)ft.tw_v, nv, tid, nthr);
  const int ip = i - p.nx / 2;
  const int a = ip < 0 ? ip + p.nu : ip;
  const float2* sa_ = grid + ((int64_t)qa * p.nu + a) * nv;
  const float2* sb_ = grid + ((int64_t)qb * p.nu + a) * nv;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  // columns outside the window are known to be zero
  for (int r = tid; r < nv - ft.b_len; r += nthr) {
    int n = ft.b_lo + ft.b_len + r;
    if (n >= nv) n -= nv;
    s[sw2(n)] = z;
  }
  const int npair = ft.b_len >> 1;
#pragma unroll 4
  for (int r = tid; r < npair; r += nthr) {
    int n = ft.b_lo + 2 * r;
    if (n >= nv) n -= nv;
    const float4 va = *reinterpret_cast<const float4*>(sa_ + n);  // {re(n), im(n), re(n+1), im(n+1)} of plane a
    const float4 vb = *reinterpret_cast<const float4*>(sb_ + n);
    // swap-in: the engine transforms (im, re), which makes the forward transform the inverse one
    s[sw2(n)] = make_float4(va.y, vb.y, va.x, vb.x);
    s[sw2(n + 1)] = make_float4(va.w, vb.w, va.z, vb.z);
  }
  __syncthreads();
  p2_fft_dif<1>(s, tw, dv, P2_IN_PAIR, tid, nthr);
  const double wa = ft.plane_w ? ft.plane_w[qa] : p.w0 + qa * p.dw;
  const double wb = ft.plane_w ? ft.plane_w[qb] : p.w0 + qb * p.dw;
  const int64_t row = (int64_t)i * p.ny;
  double* dsta = accimg + row + (ft.plane_img ? (int64_t)ft.plane_img[qa] * p.nx * p.ny : 0);
  double* dstb = accimg + row + (ft.plane_img ? (int64_t)ft.plane_img[qb] * p.nx * p.ny : 0);
  const bool same_img = dsta == dstb;
  // engine output = swap(IDFT): element {Im_a, Im_b, Re_a, Re_b}; contribution Re(IDFT e^{-i theta}) = Re c + Im s
  if ((p.ny & 7) == 0) {
    constexpr int RU = 3;  // groups of 4 pixels in flight per thread: the nu-table / position loads are L2 round trips
    const int ng = p.ny >> 2;
    for (int g0 = tid; g0 < ng; g0 += RU * nthr) {
      double nuv[RU][4];
      int pv[RU][4];
#pragma unroll
      for (int u = 0; u < RU; ++u) {
        const int g = g0 + u * nthr;
        if (g < ng) {
          const int j = 4 * g, jp = j - hy;
          if (p.do_wgridding) load4(ft.nutab + row + j, nuv[u]);
          load4(pos_v + (jp < 0 ? jp + nv : jp), pv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < RU; ++u) {
        const int g = g0 + u * nthr;
        if (g < ng) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float4 v = s[sw2(pv[u][e])];
            float ra, rb;
            if (p.do_wgridding) {
              float ca, sna, c2, sn2;
              cis_screen<FAST>(wa * nuv[u][e], ca, sna);
              cis_screen<FAST>(wb * nuv[u][e], c2, sn2);
              ra = v.z * ca + v.x * sna;
              rb = v.w * c2 + v.y * sn2;
            } else {
              ra = v.z;
              rb = v.w;
            }
            if (same_img) {
              atomicAdd(dsta + 4 * g + e, (double)ra + (double)rb);
            } else {
              atomicAdd(dsta + 4 * g + e, (double)ra);
              atomicAdd(dstb + 4 * g + e, (double)rb);
            }
          }
        }
      }
    }
  } else {
    for (int j = tid; j < p.ny; j += nthr) {
      const int jp = j - hy;
      const float4 v = s[sw2(pos_v[jp < 0 ? jp + nv : jp])];
      float ra, rb;
      if (p.do_wgridding) {
        float ca, sna, c2, sn2;
        cis_screen<FAST>(wa * ft.nutab[row + j], ca, sna);
        cis_screen<FAST>(wb * ft.nutab[row + j], c2, sn2);
        ra = v.z * ca + v.x * sna;
        rb = v.w * c2 + v.y * sn2;
      } else {
        ra = v.z;
        rb = v.w;
      }
      if (same_img) {
        atomicAdd(dsta + j, (double)ra + (double)rb);
      } else {
        atomicAdd(dsta + j, (double)ra);
        atomicAdd(dstb + j, (double)rb);
      }
    }
  }
}
