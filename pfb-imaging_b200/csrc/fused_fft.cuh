// Fused, pruned plane transforms (kernel 4 + the 2-D FFT in one): replaces
//   k_img2grid + cuFFT (degrid direction)   by  k_rows_fwd  + k_cols_fwd
//   cuFFT + k_grid2img (grid direction)     by  k_cols_inv  + k_rows_inv
//
// Per direction the plane stack is touched 2.3 times instead of 7 (SURVEY §8d counts 6):
//   rows_fwd : reads the image row (L2), builds pad + beam + correction + w-screen in shared memory,
//              FFT along v (DIT, natural output), writes ONLY the nx image rows of the plane
//   cols_fwd : reads ONLY those nx rows of a 32-byte wide column block, FFT along u, writes nu rows
//   cols_inv : reads nu rows of a column block, inverse FFT along u, writes ONLY the nx image rows
//   rows_inv : per image row, loops over the planes: reads the row, inverse FFT along v, applies the
//              conjugate w-screen to the ny kept outputs and accumulates them in fp64 registers;
//              one write of the image row with correction / beam / wsum / ridge fused
// Column blocks whose cells no bound visibility touches are skipped (cb_lo..cb_hi).
#pragma once
#include "common.cuh"
#include "fft.cuh"

#include "fused_common.cuh"

// --------------------------------------------------------------------------- degrid direction
// grid = (plane, image row), plane fastest: the CTAs sharing an image row (x, corr, nu table) are
// co-resident, so those rows are read from DRAM once instead of once per plane.
// BIG: rows so long that only one CTA fits an SM (> 113 KB of shared memory: fp32 rows beyond 14 k cells, config 4):
// three (fp32) / two (fp64) times the threads on the same transform, or 6 warps per SM would have to hide everything
template <typename T, bool FAST = false, bool BIG = false>
__global__ void __launch_bounds__(BIG ? (sizeof(T) == 4 ? ROWS_BIG_THREADS_F32 : ROWS_BIG_THREADS_F64) : ROWS_MAX_THREADS,
                                  BIG ? 1 : (sizeof(T) == 4 ? 3 : 2))
k_rows_fwd(GParams p, FusedTabs ft, const T* __restrict__ x, const T* __restrict__ beam, const T* __restrict__ corr,
           typename cplx_of<T>::type* __restrict__ grid) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  const int tid = threadIdx.x, nthr = blockDim.x, q = blockIdx.x + ft.q0, i = blockIdx.y;
  const int nv = p.nv, hy = p.ny / 2;
  const int ip = i - p.nx / 2;
  const int a = ip < 0 ? ip + p.nu : ip;
  for (int n = tid; n < nv; n += nthr) s[fft_pad<T>(n)] = {(T)0, (T)0};
  __syncthreads();
  const double wq = ft.plane_w ? ft.plane_w[q] : p.w0 + q * p.dw;
  const int64_t row = (int64_t)i * p.ny;
  if (ft.plane_img) {  // this plane's snapshot image and beam
    const int64_t off = (int64_t)ft.plane_img[q] * p.nx * p.ny;
    x += off;
    if (beam) beam += off;
  }
  const bool vec_ok = (p.ny & 7) == 0 &&
                      (((uintptr_t)x | (uintptr_t)corr | (uintptr_t)beam) & 15) == 0;  // caller-owned device pointers
  if (vec_ok) {
    // 4 consecutive pixels per step (hy % 4 == 0, so a group never straddles the wrap), two steps in flight
    const int ng = p.ny >> 2;
    for (int g0 = tid; g0 < ng; g0 += 2 * nthr) {
      T xv[2][4], cv[2][4], bv[2][4];
      double nuv[2][4];
      int pv[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int g = g0 + u * nthr;
        if (g < ng) {
          const int j = 4 * g;
          load4(x + row + j, xv[u]);
          load4(corr + row + j, cv[u]);
          if (beam) load4(beam + row + j, bv[u]);
          if (p.do_wgridding) load4(ft.nutab + row + j, nuv[u]);
          const int jp = j - hy;
          load4(ft.pos_v + (jp < 0 ? jp + nv : jp), pv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (g0 + u * nthr < ng) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            T val = xv[u][e] * cv[u][e];
            if (beam) val *= bv[u][e];
            cx2<T> v = {val, (T)0};
            if (p.do_wgridding && val != (T)0) {
              T c, sn;
              cis_screen<FAST>(wq * nuv[u][e], c, sn);
              v = {val * c, val * sn};
            }
            s[fft_pad<T>(pv[u][e])] = v;
          }
        }
      }
    }
  } else {
    for (int j = tid; j < p.ny; j += nthr) {
      const int64_t pix = row + j;
      T val = x[pix] * corr[pix];
      if (beam) val *= beam[pix];
      cx2<T> v = {val, (T)0};
      if (p.do_wgridding && val != (T)0) {
        T c, sn;
        cis_screen<FAST>(wq * ft.nutab[pix], c, sn);
        v = {val * c, val * sn};
      }
      const int jp = j - hy;
      s[fft_pad<T>(ft.pos_v[jp < 0 ? jp + nv : jp])] = v;
    }
  }
  __syncthreads();
  fft_dit<T, 1>(s, (const cx2<T>*)ft.tw_v, ft.dv, tid, nthr);
  // only the active columns are written (window bounds are multiples of 32)
  cx2<T>* dst = reinterpret_cast<cx2<T>*>(grid) + ((int64_t)q * p.nu + a) * nv;
  const int npair = ft.b_len >> 1;
#pragma unroll 4
  for (int r = tid; r < npair; r += nthr) {
    int n = ft.b_lo + 2 * r;
    if (n >= nv) n -= nv;
    store_pair(dst + n, s[fft_pad<T>(n)], s[fft_pad<T>(n + 1)]);
  }
}

// Column kernels: a CTA owns a block of C columns (one 32-byte sector per grid row).  Element w of the
// block maps to (row w / C, column w % C): consecutive lanes touch consecutive shared-memory words (no
// bank conflicts) and the 4 (2) lanes of a row share one global sector.  COLS_U independent global
// accesses are kept in flight per thread: with one CTA per SM nothing else hides the L2 / DRAM latency.
#define COLS_U 8

// column block of C columns starting at b0; rows of the image band only are read
template <typename T, int C>
__global__ void __launch_bounds__(512)
k_cols_fwd(GParams p, FusedTabs ft, const typename cplx_of<T>::type* grid, typename cplx_of<T>::type* grid_out) {
  // grid_out == grid for the in-place transform of a local stack; a helper GPU of a split band passes the
  // owner's peer-mapped stack: the transformed columns then go straight over NVLink (posted stores)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  constexpr int LGC = C == 1 ? 0 : (C == 2 ? 1 : 2);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int b0 = (ft.b_lo + blockIdx.x * C) % p.nv, q = blockIdx.y + ft.q0;
  const int nu = p.nu, nx = p.nx, hx = p.nx / 2;
  const cx2<T>* g = reinterpret_cast<const cx2<T>*>(grid) + (int64_t)q * nu * p.nv + b0;
  cx2<T>* go = reinterpret_cast<cx2<T>*>(grid_out) + (int64_t)q * nu * p.nv + b0;
  for (int w = tid; w < (nu - nx) * C; w += nthr) s[fft_pad<T>(hx * C + w)] = {(T)0, (T)0};
  const int nin = nx * C;
  for (int w0 = tid; w0 < nin; w0 += COLS_U * nthr) {
    cx2<T> v[COLS_U];
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nin) {
        const int r = w >> LGC, c = w & (C - 1);
        const int a = r < hx ? r : r + (nu - nx);
        v[u] = g[(int64_t)a * p.nv + c];
      }
    }
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nin) {
        const int r = w >> LGC, c = w & (C - 1);
        const int a = r < hx ? r : r + (nu - nx);
        s[fft_pad<T>(a * C + c)] = v[u];
      }
    }
  }
  __syncthreads();
  fft_dif<T, C>(s, (const cx2<T>*)ft.tw_u, ft.du, tid, nthr);
  const int nout = ft.a_len * C;
  for (int w0 = tid; w0 < nout; w0 += COLS_U * nthr) {
    int pos[COLS_U];
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nout) {
        int k = ft.a_lo + (w >> LGC);
        if (k >= nu) k -= nu;
        pos[u] = ft.pos_u[k];
      }
    }
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nout) {
        const int c = w & (C - 1);
        int k = ft.a_lo + (w >> LGC);
        if (k >= nu) k -= nu;
        go[(int64_t)k * p.nv + c] = s[fft_pad<T>(pos[u] * C + c)];
      }
    }
  }
}

// --------------------------------------------------------------------------- grid direction
template <typename T, int C>
__global__ void __launch_bounds__(512)
k_cols_inv(GParams p, FusedTabs ft, const typename cplx_of<T>::type* grid, typename cplx_of<T>::type* grid_out) {
  // grid may be the peer-mapped stack of the band's owner (helper GPU of a split band: the gridded columns are
  // read over NVLink, COLS_U loads in flight per thread), grid_out the local stack
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  constexpr int LGC = C == 1 ? 0 : (C == 2 ? 1 : 2);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int b0 = (ft.b_lo + blockIdx.x * C) % p.nv, q = blockIdx.y + ft.q0;
  const int nu = p.nu, nx = p.nx, hx = p.nx / 2;
  const cx2<T>* g = reinterpret_cast<const cx2<T>*>(grid) + (int64_t)q * nu * p.nv + b0;
  cx2<T>* go = reinterpret_cast<cx2<T>*>(grid_out) + (int64_t)q * nu * p.nv + b0;
  // rows outside the active window are known to be zero
  for (int w = tid; w < (nu - ft.a_len) * C; w += nthr) {
    int k = ft.a_lo + ft.a_len + (w >> LGC);
    if (k >= nu) k -= nu;
    s[fft_pad<T>(k * C + (w & (C - 1)))] = {(T)0, (T)0};
  }
  const int nin = ft.a_len * C;
  for (int w0 = tid; w0 < nin; w0 += COLS_U * nthr) {
    cx2<T> v[COLS_U];
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nin) {
        int k = ft.a_lo + (w >> LGC);
        if (k >= nu) k -= nu;
        v[u] = g[(int64_t)k * p.nv + (w & (C - 1))];
      }
    }
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nin) {
        int k = ft.a_lo + (w >> LGC);
        if (k >= nu) k -= nu;
        s[fft_pad<T>(k * C + (w & (C - 1)))] = {v[u].x, -v[u].y};  // inverse = conj o forward o conj
      }
    }
  }
  __syncthreads();
  fft_dif<T, C>(s, (const cx2<T>*)ft.tw_u, ft.du, tid, nthr);
  const int nout = nx * C;
  for (int w0 = tid; w0 < nout; w0 += COLS_U * nthr) {
    int pos[COLS_U];
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nout) {
        const int r = w >> LGC;
        pos[u] = ft.pos_u[r < hx ? r : r + (nu - nx)];
      }
    }
#pragma unroll
    for (int u = 0; u < COLS_U; ++u) {
      const int w = w0 + u * nthr;
      if (w < nout) {
        const int r = w >> LGC, c = w & (C - 1);
        const int k = r < hx ? r : r + (nu - nx);
        cx2<T> v = s[fft_pad<T>(pos[u] * C + c)];
        v.y = -v.y;
        go[(int64_t)k * p.nv + c] = v;
      }
    }
  }
}

// One CTA per (plane, image row): read the row (active window only), inverse FFT along v, apply the
// conjugate w-screen to the ny kept outputs and add their real parts to the fp64 accumulation image
// (RED.F64; CTAs of one row are adjacent in the grid, so the 32 KB image row stays in L2).
template <typename T, bool FAST = false, bool BIG = false>
__global__ void __launch_bounds__(BIG ? (sizeof(T) == 4 ? ROWS_BIG_THREADS_F32 : ROWS_BIG_THREADS_F64) : ROWS_MAX_THREADS,
                                  BIG ? 1 : (sizeof(T) == 4 ? 3 : 2))
k_rows_inv(GParams p, FusedTabs ft, const typename cplx_of<T>::type* __restrict__ grid, double* __restrict__ accimg) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cx2<T>* s = reinterpret_cast<cx2<T>*>(smem_raw);
  const int tid = threadIdx.x, nthr = blockDim.x, q = blockIdx.x + ft.q0, i = blockIdx.y;
  const int nv = p.nv, hy = p.ny / 2;
  const int ip = i - p.nx / 2;
  const int a = ip < 0 ? ip + p.nu : ip;
  const cx2<T>* src = reinterpret_cast<const cx2<T>*>(grid) + ((int64_t)q * p.nu + a) * nv;
  // columns outside the window are known to be zero
  for (int r = tid; r < nv - ft.b_len; r += nthr) {
    int n = ft.b_lo + ft.b_len + r;
    if (n >= nv) n -= nv;
    s[fft_pad<T>(n)] = {(T)0, (T)0};
  }
  const int npair = ft.b_len >> 1;
#pragma unroll 4
  for (int r = tid; r < npair; r += nthr) {
    int n = ft.b_lo + 2 * r;
    if (n >= nv) n -= nv;
    cx2<T> v0, v1;
    load_pair(src + n, v0, v1);
    s[fft_pad<T>(n)] = {v0.x, -v0.y};
    s[fft_pad<T>(n + 1)] = {v1.x, -v1.y};
  }
  __syncthreads();
  fft_dif<T, 1>(s, (const cx2<T>*)ft.tw_v, ft.dv, tid, nthr);
  const double wq = ft.plane_w ? ft.plane_w[q] : p.w0 + q * p.dw;
  const int64_t row = (int64_t)i * p.ny;
  double* dst = accimg + row + (ft.plane_img ? (int64_t)ft.plane_img[q] * p.nx * p.ny : 0);
  if ((p.ny & 7) == 0) {
    // RU groups of 4 pixels in flight per thread: the nu-table / position loads are L2 round trips
    constexpr int RU = PFBG_ROWS_INV_INFLIGHT;
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
          load4(ft.pos_v + (jp < 0 ? jp + nv : jp), pv[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < RU; ++u) {
        const int g = g0 + u * nthr;
        if (g < ng) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const cx2<T> v = s[fft_pad<T>(pv[u][e])];  // conj(v) is the inverse transform
            double r;
            if (p.do_wgridding) {
              T c, sn;
              cis_screen<FAST>(wq * nuv[u][e], c, sn);
              r = (double)(v.x * c - v.y * sn);  // Re( conj(v) e^{-i theta} )
            } else {
              r = (double)v.x;
            }
            atomicAdd(dst + 4 * g + e, r);
          }
        }
      }
    }
  } else {
    for (int j = tid; j < p.ny; j += nthr) {
      const int jp = j - hy;
      const cx2<T> v = s[fft_pad<T>(ft.pos_v[jp < 0 ? jp + nv : jp])];
      double r;
      if (p.do_wgridding) {
        T c, sn;
        cis_screen<FAST>(wq * ft.nutab[row + j], c, sn);
        r = (double)(v.x * c - v.y * sn);
      } else {
        r = (double)v.x;
      }
      atomicAdd(dst + j, r);
    }
  }
}

// out = (acc [+ acc2]) * corr [* beam] * inv_wsum [+ eta * xin]      (acc2: the planes a helper GPU transformed)
template <typename T>
__global__ void k_finish_image(int64_t npix, int64_t npix_img, const double* __restrict__ acc,
                               const double* __restrict__ acc2, const T* __restrict__ corr, const T* __restrict__ beam,
                               const T* __restrict__ xin, double inv_wsum, double eta, T* __restrict__ out) {
  // npix = nbatch * npix_img: the images of a batch share the correction of their common geometry; every snapshot
  // has its own beam
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= npix) return;
  const int64_t kc = npix == npix_img ? k : k % npix_img;
  double a = acc[k];
  if (acc2) a += acc2[k];
  double r = a * (double)corr[kc];
  if (beam) r *= (double)beam[k];
  r *= inv_wsum;
  if (xin) r += eta * (double)xin[k];
  out[k] = (T)r;
}

__global__ void k_nu_table(GParams p, double* __restrict__ nutab) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  int i = blockIdx.y;
  if (j >= p.ny) return;
  nutab[(int64_t)i * p.ny + j] = pixel_nm1(p, i, j) + p.nshift;
}

// mark the 32-cell groups of rows / columns touched by the bound samples (host derives the windows)
template <typename Rec>
__global__ void k_mark_cells(const Rec* __restrict__ recs, int64_t nact, int W, int nu, int nv,
                             int* __restrict__ uflag, int* __restrict__ vflag) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nact) return;
  int iu = recs[k].iu, iv = recs[k].iv;
  int iu2 = iu + W - 1, iv2 = iv + W - 1;
  if (iu2 >= nu) iu2 -= nu;
  if (iv2 >= nv) iv2 -= nv;
  uflag[iu >> 5] = 1; uflag[iu2 >> 5] = 1;
  vflag[iv >> 5] = 1; vflag[iv2 >> 5] = 1;
  if ((recs[k].ip & 0x3fffffff) < 64) {  // first plane < 0 (REC_IP_BIAS): the mirrored cells are touched too
    const int mu = iu ? nu - iu : 0, mu2 = iu2 ? nu - iu2 : 0, mv = iv ? nv - iv : 0, mv2 = iv2 ? nv - iv2 : 0;
    uflag[mu >> 5] = 1; uflag[mu2 >> 5] = 1;
    vflag[mv >> 5] = 1; vflag[mv2 >> 5] = 1;
  }
}

// zero the active window of every plane (instead of a memset of the whole stack)
template <typename C>
__global__ void k_zero_window(C* __restrict__ grid, int nu, int nv, int a_lo, int a_len, int b_lo, int b_len) {
  const int q = blockIdx.z;
  const int ra = blockIdx.y;
  int a = a_lo + ra;
  if (a >= nu) a -= nu;
  C* row = grid + ((int64_t)q * nu + a) * nv;
  C z; z.x = 0; z.y = 0;
  for (int rb = blockIdx.x * blockDim.x + threadIdx.x; rb < b_len; rb += gridDim.x * blockDim.x) {
    int b = b_lo + rb;
    if (b >= nv) b -= nv;
    row[b] = z;
  }
}

// ---- band split across GPUs: flags in peer-mapped memory order the kernels of the two processes ------------
// (one thread each; the waiter polls its OWN memory, the signaller writes over NVLink after a system fence)
__global__ void k_flag_signal(unsigned long long* flag, unsigned long long value) {
  __threadfence_system();
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(value) : "memory");
}
__global__ void k_flag_wait(const unsigned long long* flag, unsigned long long want, unsigned long long timeout_ns,
                            int* timed_out) {
  unsigned long long t0, t, v;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
    if (v >= want) break;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    if (t - t0 > timeout_ns) { *timed_out = 1; break; }  // never hang the GPU: the host reports the time-out
    __nanosleep(256);
  }
}
// xshare = x [* beam]: what the helper's row transforms start from
template <typename T>
__global__ void k_share_image(int64_t npix, const T* __restrict__ x, const T* __restrict__ beam, T* __restrict__ out) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < npix) out[k] = beam ? x[k] * beam[k] : x[k];
}
