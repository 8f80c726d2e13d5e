// Run-based gridding / degridding kernels (W <= 8).
//
// Kernel 1 sorts the samples by (uv tile, first w-plane, first cell inside the tile), so all
// samples whose W x W x W footprint starts at the same grid cell are contiguous ("a run").  On
// MeerKAT-like coverage > 90 % of consecutive samples belong to the same run, hence:
//
//   * one warp walks a slice of the sorted samples, a batch of NB samples at a time;
//   * the lanes own the footprint: lane = (j, q2) with j = v-offset (0..7) and q2 = plane slot
//     (planes q2 and q2+4); each lane keeps the 8 u-rows of its two planes in registers
//     (16 complex accumulators / grid values);
//   * per batch: (a) lane <-> sample: load the 32/64-byte record, form weight*phase*vis;
//     (b) lane <-> tap: evaluate the 24 ES taps of every sample of the batch into shared memory
//     (independent evaluations, full ILP, fast-math in fp32); (c) the FMA stage;
//   * gridding: accumulate in registers for the whole run, then flush the run ONCE with 16
//     vector REDs per lane (8 lanes x 8 B = 64 B contiguous per row);
//   * degridding: load the run's footprint ONCE, then every sample is 38 FMAs; the 32-lane sum
//     is taken per batch through a skewed shared-memory transpose instead of shuffles.
//
// Per-sample geometry comes from 32 B (fp32) / 64 B (fp64) records written in bucket order by
// kernel 1 (k_make_recs): no fp64 coordinate arithmetic and no scattered uvw loads here.
#pragma once
#include "common.cuh"

template <typename T> struct VisRec;
template <> struct __align__(16) VisRec<float> {
  float x0[3];        // first tap position relative to the sample, per axis: (i0 - g) in (-W/2, -W/2+1]
  uint32_t idx;       // flat (row, chan) index
  float pc, ps;       // e^{+2 pi i (u x0 + v y0 + w nshift)}
  uint16_t iu, iv;    // wrapped first cell
  int32_t ip;         // first plane + REC_IP_BIAS (it can be negative with mirror planes); bit 30 = folded sample
};
template <> struct __align__(16) VisRec<double> {
  double x0[3];
  double pc, ps;
  uint32_t idx;
  uint16_t iu, iv;
  int32_t ip;
  int32_t pad;
};
static_assert(sizeof(VisRec<float>) == 32, "VisRec<float> must be 32 bytes");
static_assert(sizeof(VisRec<double>) == 64, "VisRec<double> must be 64 bytes");

#define REC_CONJ_BIT 0x40000000
#define REC_IP_BIAS 64
__device__ __forceinline__ int origin_plane(uint64_t origin) { return (int)(origin >> 32) - REC_IP_BIAS; }
__device__ __forceinline__ uint64_t pack_origin(uint32_t iu, uint32_t iv, int32_t ip) {
  return ((uint64_t)(uint32_t)(ip & ~REC_CONJ_BIT) << 32) | ((uint64_t)iu << 16) | (uint64_t)iv;
}

// kernel 1b: per-sample records in bucket order
template <typename T>
__global__ void k_make_recs(GParams p, const double* __restrict__ uvw, const double* __restrict__ fscale,
                            const uint32_t* __restrict__ sorted_idx, int64_t nact, VisRec<T>* __restrict__ recs) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nact) return;
  uint32_t idx = sorted_idx[k];
  int64_t row = idx / p.nchan;
  int chan = (int)(idx - row * p.nchan);
  VisCoord c = vis_coord(p, uvw, fscale, row, chan);
  VisRec<T> r;
  r.x0[0] = (T)((double)c.iu0 - c.gu);
  r.x0[1] = (T)((double)c.iv0 - c.gv);
  r.x0[2] = (T)((double)c.ip0 - c.gw);
  r.idx = idx;
  cis_turns(vis_phase_turns(p, c), r.pc, r.ps);
  r.iu = (uint16_t)wrap(c.iu0, p.nu);
  r.iv = (uint16_t)wrap(c.iv0, p.nv);
  r.ip = (c.ip0 + REC_IP_BIAS) | (c.conj ? REC_CONJ_BIT : 0);
  recs[k] = r;
}

// ES tap for the run kernels: fp32 uses the SFU (sqrt.approx / ex2.approx); the absolute error
// stays ~1e-7 of the kernel peak, far below the fp32 accuracy floor (epsilon >= 3e-7).
__device__ __forceinline__ float es_fast(float x, float beta_log2e) {
  float a = fmaf(-x, x, 1.0f);
  float s, e;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(fmaxf(a, 0.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(beta_log2e * (s - 1.0f)));
  return a < 0.0f ? 0.0f : e;
}
__device__ __forceinline__ double es_fast(double x, double beta) { return es_eval(x, beta); }

// tap k (cell i0 + k) of a sample whose first cell sits at x0 = i0 - g in (-W/2, -W/2 + 1].
// (A piecewise-polynomial form of the fp64 taps, degree W+3 as in ducc0, was measured on B200 and is NOT faster
// than exp + sqrt: 10 16-byte coefficient loads + 19 dependent DFMAs per tap; it was dropped.)
__device__ __forceinline__ float tap_eval(const GParams& p, float x0, int k, float bscale, float xs) {
  return es_fast((x0 + (float)k) * xs, bscale);
}
__device__ __forceinline__ double tap_eval(const GParams& p, double x0, int k, double bscale, double xs) {
  return es_fast((x0 + (double)k) * xs, bscale);
}
__device__ __forceinline__ float es_scale(float beta) { return beta * 1.4426950408889634f; }
__device__ __forceinline__ double es_scale(double beta) { return beta; }

#define RUN_WARPS 8      /* warps per CTA, gridding */
#define DEG_WARPS 4      /* warps per CTA, degridding (48 KB static shared memory) */
#ifndef RUN_SLICE
#define RUN_SLICE 512
#endif
#ifndef RUN_SLICE_TAIL
#define RUN_SLICE_TAIL 64
#endif
#ifndef GRID_UNROLL
#define GRID_UNROLL 2
#endif
constexpr int kGridUnroll = GRID_UNROLL;
#ifndef DEG_UNROLL
#define DEG_UNROLL 2
#endif
constexpr int kDegUnroll = DEG_UNROLL;

template <typename T> struct RunCfg;
template <> struct RunCfg<float> { static constexpr int NB = 32; };
template <> struct RunCfg<double> { static constexpr int NB = 16; };

// evaluate the 24 taps of the nb staged samples: lane t < 24 owns tap t (axis = t/8, k = t%8)
// (fp64 path; the fp32 kernels evaluate all 24 taps of a sample in its own lane, see run_taps_lane)
template <typename T, int NB>
__device__ __forceinline__ void run_taps(const GParams& p, const T (*x0s)[4], T (*taps)[24], int nb, int lane,
                                         T bscale, T xs) {
  if (lane < 24) {
    const int axis = lane >> 3;
    const int kk = lane & 7;
    const bool flat_w = (axis == 2) && !p.do_wgridding;
#pragma unroll 4
    for (int v = 0; v < nb; ++v) {
      T val = tap_eval(p, x0s[v][axis], kk, bscale, xs);
      if (flat_w) val = (lane == 16) ? (T)1 : (T)0;
      taps[v][lane] = val;
    }
  }
}

// lane <-> sample: all 24 taps of this lane's sample, written as six 16-byte stores.  Every lane is
// busy and there is no loop over the batch, which halves the cost of the tap stage (ncu: the
// lane <-> tap version was 26 % of the gridding kernel's stall samples).
template <typename T>
__device__ __forceinline__ void run_taps_lane(const GParams& p, const T (&x0)[3], T* __restrict__ dst, T bscale, T xs) {
#pragma unroll
  for (int axis = 0; axis < 3; ++axis) {
    T t[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) t[k] = es_fast((x0[axis] + (T)k) * xs, bscale);
    if (axis == 2 && !p.do_wgridding) {
      t[0] = (T)1;
#pragma unroll
      for (int k = 1; k < 8; ++k) t[k] = (T)0;
    }
    if constexpr (sizeof(T) == 4) {
      float4* d4 = reinterpret_cast<float4*>(dst + axis * 8);
      d4[0] = make_float4(t[0], t[1], t[2], t[3]);
      d4[1] = make_float4(t[4], t[5], t[6], t[7]);
    } else {
      double2* d2 = reinterpret_cast<double2*>(dst + axis * 8);
#pragma unroll
      for (int k = 0; k < 4; ++k) d2[k] = make_double2(t[2 * k], t[2 * k + 1]);
    }
  }
}

// general flush (any W <= 8, footprints that wrap around the grid edge)
template <typename T>
__device__ __forceinline__ void run_flush(const GParams& p, typename cplx_of<T>::type* __restrict__ grid,
                                          typename cplx_of<T>::type (&acc)[8][2], uint64_t origin, int j, int q2) {
  const int W = p.W, npl = p.do_wgridding ? W : 1;
  int iv = (int)(origin & 0xffffu) + j;
  int iu0 = (int)((origin >> 16) & 0xffffu);
  int ip = origin_plane(origin);
  if (iv >= p.nv) iv -= p.nv;
  const int plane_sz = p.nu * p.nv;  // < 2^31 (nu, nv <= 32768 enforced by the host)
  const bool jok = j < W;
  if (W == 8 && npl == 8 && iu0 >= 1 && iu0 + 8 <= p.nu) {
    // common case: every lane owns live cells and the 8 rows do not wrap -> one pointer, constant stride.
    // Mirror planes (pl < 0) walk the mirrored rows of plane -pl-1 backwards, conjugated.
    const int mv = iv ? p.nv - iv : 0;
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
      const int pl = ip + q2 + 4 * qq;
      const bool mir = pl < 0;
      typename cplx_of<T>::type* gq = grid + (mir ? (int64_t)(-pl - 1) * plane_sz + (int64_t)(p.nu - iu0) * p.nv + mv
                                                  : (int64_t)pl * plane_sz + (int64_t)iu0 * p.nv + iv);
      const int step = mir ? -p.nv : p.nv;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        atomic_add_c(gq, acc[i][qq].x, mir ? -acc[i][qq].y : acc[i][qq].y);
        gq += step;
        acc[i][qq].x = 0;
        acc[i][qq].y = 0;
      }
    }
    return;
  }
#pragma unroll
  for (int qq = 0; qq < 2; ++qq) {
    int q = q2 + 4 * qq;
    bool ok = jok && q < npl;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (ok && i < W) {
        int iu = iu0 + i;
        if (iu >= p.nu) iu -= p.nu;
        bool cj;
        typename cplx_of<T>::type* g = grid + plane_cell(p, ip + q, iu, iv, cj);
        atomic_add_c(g, acc[i][qq].x, cj ? -acc[i][qq].y : acc[i][qq].y);
      }
      acc[i][qq].x = 0;
      acc[i][qq].y = 0;
    }
  }
}

// the run's footprint -> registers (degridding), same two paths
template <typename T>
__device__ __forceinline__ void run_fetch(const GParams& p, const typename cplx_of<T>::type* __restrict__ grid,
                                          typename cplx_of<T>::type (&gv)[8][2], uint64_t origin, int j, int q2) {
  using C = typename cplx_of<T>::type;
  const int W = p.W, npl = p.do_wgridding ? W : 1;
  int iv = (int)(origin & 0xffffu) + j;
  int iu0 = (int)((origin >> 16) & 0xffffu);
  int ip = origin_plane(origin);
  if (iv >= p.nv) iv -= p.nv;
  const int plane_sz = p.nu * p.nv;
  const bool jok = j < W;
  if (W == 8 && npl == 8 && iu0 >= 1 && iu0 + 8 <= p.nu) {
    const int mv = iv ? p.nv - iv : 0;
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
      const int pl = ip + q2 + 4 * qq;
      const bool mir = pl < 0;
      const C* gq = grid + (mir ? (int64_t)(-pl - 1) * plane_sz + (int64_t)(p.nu - iu0) * p.nv + mv
                                : (int64_t)pl * plane_sz + (int64_t)iu0 * p.nv + iv);
      const int step = mir ? -p.nv : p.nv;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        C val = *gq;
        if (mir) val.y = -val.y;
        gv[i][qq] = val;
        gq += step;
      }
    }
    return;
  }
#pragma unroll
  for (int qq = 0; qq < 2; ++qq) {
    int q = q2 + 4 * qq;
    bool ok = jok && q < npl;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      C val; val.x = 0; val.y = 0;
      if (ok && i < W) {
        int iu = iu0 + i;
        if (iu >= p.nu) iu -= p.nu;
        bool cj;
        val = grid[plane_cell(p, ip + q, iu, iv, cj)];
        if (cj) val.y = -val.y;
      }
      gv[i][qq] = val;
    }
  }
}

__device__ __forceinline__ uint64_t shfl_u64(uint64_t x, int src) {
  const uint32_t lo = __shfl_sync(0xffffffffu, (uint32_t)x, src), hi = __shfl_sync(0xffffffffu, (uint32_t)(x >> 32), src);
  return ((uint64_t)hi << 32) | lo;
}

// ---------------------------------------------------------------------------
// Cyclic column ownership (W = 8, full 8-plane support, rows that do not wrap).
// Consecutive runs of a (tile, plane) bucket come in the order (iu, iv): the next run usually starts ONE cell
// further along v, so 7 of its 8 footprint columns are the previous run's.  Lane (j, q2) therefore owns the
// absolute grid column c with c mod 8 == j instead of the column at offset j from the run origin: when the origin
// moves along v only the lanes whose column leaves the footprint flush (gridding) or fetch (degridding) — one
// lane group of eight instead of all of them, i.e. up to 8x fewer L2 atomics / gather loads at short run lengths
// (band 7 of C2: 6.7 samples per run, the L2 was at 60 % in k_grid_runs and the FMA pipe at 35 %).  The tap a
// lane applies is k = (j - iv0) mod 8.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool run_is_cyclic(const GParams& p, uint64_t origin) {
  const int iu0 = (int)((origin >> 16) & 0xffffu);
  return p.W == 8 && p.do_wgridding && iu0 >= 1 && iu0 + 8 <= p.nu;
}
__device__ __forceinline__ int run_column(const GParams& p, uint64_t origin, int j) {
  const int iv0 = (int)(origin & 0xffffu);
  int c = iv0 + ((j - iv0) & 7);
  if (c >= p.nv) c -= p.nv;  // nv is a multiple of 8: c mod 8 stays j
  return c;
}

// flush / fetch of ONE footprint column (absolute column iv) of the run at `origin`: 8 rows x this lane's 2 planes
template <typename T>
__device__ __forceinline__ void run_flush_col(const GParams& p, typename cplx_of<T>::type* __restrict__ grid,
                                              typename cplx_of<T>::type (&acc)[8][2], uint64_t origin, int iv, int q2) {
  const int iu0 = (int)((origin >> 16) & 0xffffu);
  const int ip = origin_plane(origin);
  const int plane_sz = p.nu * p.nv;
  const int mv = iv ? p.nv - iv : 0;
#pragma unroll
  for (int qq = 0; qq < 2; ++qq) {
    const int pl = ip + q2 + 4 * qq;
    const bool mir = pl < 0;
    typename cplx_of<T>::type* gq = grid + (mir ? (int64_t)(-pl - 1) * plane_sz + (int64_t)(p.nu - iu0) * p.nv + mv
                                                : (int64_t)pl * plane_sz + (int64_t)iu0 * p.nv + iv);
    const int step = mir ? -p.nv : p.nv;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      atomic_add_c(gq, acc[i][qq].x, mir ? -acc[i][qq].y : acc[i][qq].y);
      gq += step;
      acc[i][qq].x = 0;
      acc[i][qq].y = 0;
    }
  }
}
template <typename T>
__device__ __forceinline__ void run_fetch_col(const GParams& p, const typename cplx_of<T>::type* __restrict__ grid,
                                              typename cplx_of<T>::type (&gv)[8][2], uint64_t origin, int iv, int q2) {
  using C = typename cplx_of<T>::type;
  const int iu0 = (int)((origin >> 16) & 0xffffu);
  const int ip = origin_plane(origin);
  const int plane_sz = p.nu * p.nv;
  const int mv = iv ? p.nv - iv : 0;
#pragma unroll
  for (int qq = 0; qq < 2; ++qq) {
    const int pl = ip + q2 + 4 * qq;
    const bool mir = pl < 0;
    const C* gq = grid + (mir ? (int64_t)(-pl - 1) * plane_sz + (int64_t)(p.nu - iu0) * p.nv + mv
                              : (int64_t)pl * plane_sz + (int64_t)iu0 * p.nv + iv);
    const int step = mir ? -p.nv : p.nv;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      C val = *gq;
      if (mir) val.y = -val.y;
      gv[i][qq] = val;
      gq += step;
    }
  }
}

// the next slice [kbeg, kend) of the sorted samples for this warp (lane 0 draws it from the launch's counter).
// The first 7/8 of the samples go out in slices of `big` (RUN_SLICE when there is enough work for every warp, see
// run_slice() on the host), the rest in slices of RUN_SLICE_TAIL, so the warps finish within a short slice of each
// other while most runs are not cut by a slice boundary.
__device__ __forceinline__ bool next_slice(unsigned long long* queue, int lane, int64_t nact, int big, int64_t& kbeg,
                                           int64_t& kend) {
  unsigned long long t = 0;
  if (lane == 0) t = atomicAdd(queue, 1ull);
  const int64_t sl = (int64_t)shfl_u64(t, 0);
  const int64_t nbig = (nact - (nact >> 3)) / big;
  kbeg = sl < nbig ? sl * big : nbig * big + (sl - nbig) * RUN_SLICE_TAIL;
  kend = min(nact, kbeg + (sl < nbig ? big : RUN_SLICE_TAIL));
  return kbeg < nact;
}

// run boundaries of a staged batch as a bit mask: bit v set <=> sample v starts a new run
__device__ __forceinline__ uint32_t run_starts(uint64_t org, uint64_t cur, int lane, int nb) {
  uint64_t prev = shfl_u64(org, lane > 0 ? lane - 1 : 0);
  if (lane == 0) prev = cur;
  return __ballot_sync(0xffffffffu, lane < nb && org != prev);
}

// ---------------------------------------------------------------------------
// kernel 2: gridding by runs
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(RUN_WARPS * 32, (sizeof(T) == 4 ? 3 : 1))  // fp32: <= 80 registers, 3 CTAs / SM
k_grid_runs(GParams p, const VisRec<T>* __restrict__ recs, int64_t nact,
            const typename cplx_of<T>::type* __restrict__ vis, int64_t vis_rs, int64_t vis_cs,
            const T* __restrict__ wgt, typename cplx_of<T>::type* __restrict__ grid, int vis_sorted,
            int apply_phase, unsigned long long* __restrict__ queue, int slice) {
  using C = typename cplx_of<T>::type;
  constexpr int NB = RunCfg<T>::NB;
  __shared__ __align__(16) T taps[RUN_WARPS][NB][24];
  __shared__ __align__(16) T x0s[RUN_WARPS][sizeof(T) == 8 ? NB : 1][4];  // fp64 keeps the lane <-> tap stage
  __shared__ C amp[RUN_WARPS][NB];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = lane & 7, q2 = lane >> 3;
  const T bscale = es_scale((T)p.beta), xs = (T)(2.0 / p.W);
  C acc[8][2];  // (re, im) pairs: one packed FMA per cell and sample
#pragma unroll
  for (int i = 0; i < 8; ++i) { acc[i][0].x = acc[i][0].y = 0; acc[i][1].x = acc[i][1].y = 0; }
  uint64_t cur = ~0ull;
  bool cyc = false;  // the current run uses cyclic column ownership
  int myc = 0;       // ... and this lane holds absolute column myc
  int kj = j;        // v-tap this lane applies
  // slices are handed out in sort order from a device counter: their cost varies with the run length (the dense
  // core against the outer uv plane), and a fixed stride left the last warps running alone for ~5 % of the kernel
  for (;;) {
    int64_t kbeg, kend;
    if (!next_slice(queue, lane, nact, slice, kbeg, kend)) break;
    // records are fetched one batch ahead (their latency hides behind the FMA stage)
    VisRec<T> rnext;
    if (kbeg + lane < kend && lane < NB) rnext = recs[kbeg + lane];
    for (int64_t k0 = kbeg; k0 < kend; k0 += NB) {
      const int nb = (int)min((int64_t)NB, kend - k0);
      const VisRec<T> r = rnext;
      uint64_t org = ~0ull;
      if (lane < nb) {  // (a) lane <-> sample
        const int64_t k = k0 + lane;
        C a;
        if (vis_sorted) a = vis[k];
        else {
          int64_t row = r.idx / p.nchan;
          int chan = (int)(r.idx - row * p.nchan);
          a = vis[row * vis_rs + chan * vis_cs];
        }
        const T w = wgt ? wgt[r.idx] : (T)1;
        if (k + NB < kend) rnext = recs[k + NB];
        if constexpr (sizeof(T) == 4) {
          const T x0[3] = {r.x0[0], r.x0[1], r.x0[2]};
          run_taps_lane<T>(p, x0, &taps[warp][lane][0], bscale, xs);  // independent of the loads above
        } else {
          x0s[warp][lane][0] = r.x0[0]; x0s[warp][lane][1] = r.x0[1]; x0s[warp][lane][2] = r.x0[2];
        }
        T pc = apply_phase ? r.pc : (T)1, ps = apply_phase ? r.ps : (T)0;
        if (apply_phase && (r.ip & REC_CONJ_BIT)) a.y = -a.y;  // folded sample (the Hessian path stays folded)
        C sa;
        sa.x = (a.x * pc - a.y * ps) * w;
        sa.y = (a.x * ps + a.y * pc) * w;
        amp[warp][lane] = sa;
        org = pack_origin(r.iu, r.iv, r.ip);
      }
      const uint32_t starts = run_starts(org, cur, lane, nb);
      __syncwarp();
      if constexpr (sizeof(T) == 8) {
        run_taps<T, NB>(p, x0s[warp], taps[warp], nb, lane, bscale, xs);
        __syncwarp();
      }
      int v = 0;
      while (v < nb) {  // (c) lane <-> footprint cell, one run segment at a time
        if ((starts >> v) & 1u) {
          const uint64_t nxt = shfl_u64(org, v);
          const bool ncyc = run_is_cyclic(p, nxt);
          if (cur != ~0ull) {
            if (cyc && ncyc && (cur >> 16) == (nxt >> 16)) {
              // same rows and planes, origin moved along v: only the lanes whose column leaves the footprint flush
              const int c = run_column(p, nxt, j);
              if (c != myc) run_flush_col<T>(p, grid, acc, cur, myc, q2);
            } else if (cyc) run_flush_col<T>(p, grid, acc, cur, myc, q2);
            else run_flush<T>(p, grid, acc, cur, j, q2);
          }
          cur = nxt;
          cyc = ncyc;
          myc = run_column(p, nxt, j);
          kj = ncyc ? ((j - (int)(nxt & 0xffffu)) & 7) : j;
        }
        const uint32_t rest = v < 31 ? (starts & (0xffffffffu << (v + 1))) : 0u;
        const int vend = rest ? min(__ffs(rest) - 1, nb) : nb;
#pragma unroll kGridUnroll
        for (; v < vend; ++v) {
          const T* tp = taps[warp][v];
          const T tv = tp[8 + kj];
          const T c0 = tv * tp[16 + q2], c1 = tv * tp[20 + q2];
          const C a = amp[warp][v];
          const C a0 = cmul_s(a, c0), a1 = cmul_s(a, c1);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const T u = tp[i];
            acc[i][0] = cfma_s(a0, u, acc[i][0]);
            acc[i][1] = cfma_s(a1, u, acc[i][1]);
          }
        }
      }
      __syncwarp();
    }
  }
  if (cur != ~0ull) {
    if (cyc) run_flush_col<T>(p, grid, acc, cur, myc, q2);
    else run_flush<T>(p, grid, acc, cur, j, q2);
  }
}

// ---------------------------------------------------------------------------
// kernel 3: degridding by runs
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(DEG_WARPS * 32)
k_degrid_runs(GParams p, const VisRec<T>* __restrict__ recs, int64_t nact,
              const typename cplx_of<T>::type* __restrict__ grid, const T* __restrict__ wgt,
              typename cplx_of<T>::type* __restrict__ vis_out,
              typename cplx_of<T>::type* __restrict__ out_sorted, int apply_phase,
              unsigned long long* __restrict__ queue, int slice) {
  using C = typename cplx_of<T>::type;
  constexpr int NB = RunCfg<T>::NB;
  __shared__ __align__(16) T taps[DEG_WARPS][NB][24];
  __shared__ __align__(16) T x0s[DEG_WARPS][sizeof(T) == 8 ? NB : 1][4];
  __shared__ C part[DEG_WARPS][NB][32];  // per-sample partial sums of the 32 lanes
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = lane & 7, q2 = lane >> 3;
  const T bscale = es_scale((T)p.beta), xs = (T)(2.0 / p.W);
  C gv[8][2];  // the run's footprint as (re, im) pairs
#pragma unroll
  for (int i = 0; i < 8; ++i) { gv[i][0].x = gv[i][0].y = 0; gv[i][1].x = gv[i][1].y = 0; }
  uint64_t cur = ~0ull;
  bool cyc = false;  // cyclic column ownership, see run_is_cyclic
  int myc = 0, kj = j;
  for (;;) {  // slices from the device counter, see k_grid_runs
    int64_t kbeg, kend;
    if (!next_slice(queue, lane, nact, slice, kbeg, kend)) break;
    VisRec<T> rnext;
    if (kbeg + lane < kend && lane < NB) rnext = recs[kbeg + lane];
    for (int64_t k0 = kbeg; k0 < kend; k0 += NB) {
      const int nb = (int)min((int64_t)NB, kend - k0);
      const VisRec<T> r = rnext;
      uint64_t org = ~0ull;
      T w = (T)1;
      if (lane < nb) {
        if (wgt) w = wgt[r.idx];  // consumed after the gather stage
        if (k0 + lane + NB < kend) rnext = recs[k0 + lane + NB];
        if constexpr (sizeof(T) == 4) {
          const T x0[3] = {r.x0[0], r.x0[1], r.x0[2]};
          run_taps_lane<T>(p, x0, &taps[warp][lane][0], bscale, xs);
        } else {
          x0s[warp][lane][0] = r.x0[0]; x0s[warp][lane][1] = r.x0[1]; x0s[warp][lane][2] = r.x0[2];
        }
        org = pack_origin(r.iu, r.iv, r.ip);
      }
      const uint32_t starts = run_starts(org, cur, lane, nb);
      __syncwarp();
      if constexpr (sizeof(T) == 8) {
        run_taps<T, NB>(p, x0s[warp], taps[warp], nb, lane, bscale, xs);
        __syncwarp();
      }
      int v = 0;
      while (v < nb) {
        if ((starts >> v) & 1u) {  // new run: fetch its footprint once (only the columns that are new to it)
          const uint64_t nxt = shfl_u64(org, v);
          const bool ncyc = run_is_cyclic(p, nxt);
          const int c = run_column(p, nxt, j);
          const bool keep = cyc && ncyc && cur != ~0ull && (cur >> 16) == (nxt >> 16) && c == myc;
          cur = nxt;
          cyc = ncyc;
          if (ncyc) {
            if (!keep) run_fetch_col<T>(p, grid, gv, cur, c, q2);
            myc = c;
            kj = (j - (int)(nxt & 0xffffu)) & 7;
          } else {
            run_fetch<T>(p, grid, gv, cur, j, q2);
            kj = j;
          }
        }
        const uint32_t rest = v < 31 ? (starts & (0xffffffffu << (v + 1))) : 0u;
        const int vend = rest ? min(__ffs(rest) - 1, nb) : nb;
#pragma unroll kDegUnroll
        for (; v < vend; ++v) {
          const T* tp = taps[warp][v];
          C a0 = cmul_s(gv[0][0], tp[0]), a1 = cmul_s(gv[0][1], tp[0]);
#pragma unroll
          for (int i = 1; i < 8; ++i) {
            const T u = tp[i];
            a0 = cfma_s(gv[i][0], u, a0);
            a1 = cfma_s(gv[i][1], u, a1);
          }
          const T tv = tp[8 + kj];
          const T c0 = tv * tp[16 + q2], c1 = tv * tp[20 + q2];
          part[warp][v][lane] = cfma_s(a1, c1, cmul_s(a0, c0));
        }
      }
      __syncwarp();
      if (lane < nb) {  // lane <-> sample again: skewed (conflict-free) sum over the 32 partials
        C sum; sum.x = 0; sum.y = 0;
#pragma unroll 8
        for (int l = 0; l < 32; ++l) sum = cfma_s(part[warp][lane][(lane + l) & 31], (T)1, sum);
        T re = sum.x, im = sum.y;
        if (apply_phase) {  // multiply by e^{-i t}
          re = sum.x * r.pc + sum.y * r.ps;
          im = sum.y * r.pc - sum.x * r.ps;
        }
        if (apply_phase && (r.ip & REC_CONJ_BIT)) im = -im;
        re *= w; im *= w;
        C o; o.x = re; o.y = im;
        if (out_sorted) out_sorted[k0 + lane] = o; else vis_out[r.idx] = o;
      }
      __syncwarp();
    }
  }
}

// ===========================================================================
// Wide-support run kernels (fp64, 13 <= W <= 16; fp64 at 9 <= W <= 12 runs on the DMMA kernels of runs_mma.cuh,
// and fp32 stops at W = 8).
//
// The footprint no longer fits one warp's registers, so a TEAM of WIDE_R warps shares every run: warp r of
// the team owns the u-rows  i = r*WIDE_RPW .. r*WIDE_RPW+WIDE_RPW-1.  Lane = (j, q2) with j = v-offset (0..15) and
// q2 = plane slot (0..1); a lane holds WIDE_RPW rows x WIDE_NQ planes (q = q2 + 2*qq), so a team covers the
// 16 x 16 x 16 footprint.
// The team works on one batch of samples at a time: warp 0 stages weight * phase * vis, ALL WIDE_R warps
// evaluate the 3 W taps of the batch together (each tap once per team: in fp64 the tap evaluation costs
// more than the FMAs, and evaluating it per warp made it 8 times redundant), then every warp runs the
// FMA stage for its rows.  Named barriers (one id per team) separate the stages.
// ===========================================================================
#define WIDE_WARPS 8
#define WIDE_R 8     // warps per team
#define WIDE_RPW 2   // u-rows per warp
#define WIDE_NQ 8    // planes per lane
#define WIDE_SLICE 256  /* samples per (statically strided) slice of a team */
#define WIDE_NB 16   // samples staged per batch
#define WIDE_NT 48   // tap slots per sample: 16 u, 16 v, 16 w (the first W of each are live)

__device__ __forceinline__ void team_sync(int team, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(nthreads) : "memory");
}

// all threads of the team: tap t = axis * W + k of sample v
__device__ __forceinline__ void wide_taps(const GParams& p, const double (*x0s)[4], double (*taps)[WIDE_NT], int nb,
                                          int ttid, int tthreads, double bscale, double xs) {
  const int W = p.W, nt = 3 * W;
  for (int idx = ttid; idx < nt * nb; idx += tthreads) {
    const int v = idx / nt, t = idx - v * nt;
    const int axis = t / W, k = t - axis * W;
    double val = tap_eval(p, x0s[v][axis], k, bscale, xs);
    if (axis == 2 && !p.do_wgridding) val = (k == 0) ? 1.0 : 0.0;
    taps[v][axis * 16 + k] = val;
  }
  if (W < 16) {  // slots beyond the support are read (times zero grid values / never flushed): keep them zero
    const int nz = 3 * (16 - W);
    for (int idx = ttid; idx < nz * nb; idx += tthreads) {
      const int v = idx / nz, t = idx - v * nz;
      const int axis = t / (16 - W), k = W + (t - axis * (16 - W));
      taps[v][axis * 16 + k] = 0.0;
    }
  }
}

__device__ __forceinline__ void wide_flush(const GParams& p, double2* __restrict__ grid,
                                           double (&accr)[WIDE_RPW][WIDE_NQ], double (&acci)[WIDE_RPW][WIDE_NQ],
                                           uint64_t origin, int j, int q2, int row0) {
  const int W = p.W, npl = p.do_wgridding ? W : 1;
  int iv = (int)(origin & 0xffffu) + j;
  int iu0 = (int)((origin >> 16) & 0xffffu);
  int ip = origin_plane(origin);
  if (iv >= p.nv) iv -= p.nv;
  const bool jok = j < W;
#pragma unroll
  for (int qq = 0; qq < WIDE_NQ; ++qq) {
    const int q = q2 + 2 * qq;
    const bool ok = jok && q < npl;
#pragma unroll
    for (int ii = 0; ii < WIDE_RPW; ++ii) {
      const int i = row0 + ii;
      if (ok && i < W) {
        int iu = iu0 + i;
        if (iu >= p.nu) iu -= p.nu;
        bool cj;
        double2* g = grid + plane_cell(p, ip + q, iu, iv, cj);
        atomic_add_c(g, accr[ii][qq], cj ? -acci[ii][qq] : acci[ii][qq]);
      }
      accr[ii][qq] = 0;
      acci[ii][qq] = 0;
    }
  }
}

__global__ void __launch_bounds__(WIDE_WARPS * 32)
k_grid_runs_wide(GParams p, const VisRec<double>* __restrict__ recs, int64_t nact, const double2* __restrict__ vis,
                 int64_t vis_rs, int64_t vis_cs, const double* __restrict__ wgt, double2* __restrict__ grid,
                 int vis_sorted, int apply_phase, unsigned long long* __restrict__ queue) {
  constexpr int NB = WIDE_NB, NTEAM = WIDE_WARPS / WIDE_R;
  __shared__ double taps[NTEAM][NB][WIDE_NT];
  __shared__ __align__(16) double x0s[NTEAM][NB][4];
  __shared__ double2 amp[NTEAM][NB];
  __shared__ unsigned long long team_slice[NTEAM];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = warp / WIDE_R, r = warp - team * WIDE_R;
  const int ttid = r * 32 + lane;
  const int j = lane & 15, q2 = lane >> 4;
  const int row0 = r * WIDE_RPW;
  const double bscale = es_scale(p.beta), xs = 2.0 / p.W;
  double accr[WIDE_RPW][WIDE_NQ], acci[WIDE_RPW][WIDE_NQ];
#pragma unroll
  for (int ii = 0; ii < WIDE_RPW; ++ii)
#pragma unroll
    for (int qq = 0; qq < WIDE_NQ; ++qq) { accr[ii][qq] = 0; acci[ii][qq] = 0; }
  uint64_t cur = ~0ull;
  const int64_t nslice = (nact + WIDE_SLICE - 1) / WIDE_SLICE;
  for (;;) {
    // the team's next slice, drawn by its first thread from the launch's counter (see k_grid_runs)
    if (ttid == 0) team_slice[team] = atomicAdd(queue, 1ull);
    team_sync(team, 32 * WIDE_R);
    const int64_t sl = (int64_t)team_slice[team];
    team_sync(team, 32 * WIDE_R);  // everybody has read it before the next draw overwrites it
    if (sl >= nslice) break;
    const int64_t kend = min(nact, (sl + 1) * WIDE_SLICE);
    for (int64_t k0 = sl * WIDE_SLICE; k0 < kend; k0 += NB) {
      const int nb = (int)min((int64_t)NB, kend - k0);
      uint64_t org = ~0ull;
      if (lane < nb) {  // every warp reads the records (it needs the run origins); warp 0 stages the rest
        const int64_t k = k0 + lane;
        const VisRec<double> rec = recs[k];
        org = pack_origin(rec.iu, rec.iv, rec.ip);
        if (r == 0) {
          double2 a;
          if (vis_sorted) a = vis[k];
          else {
            int64_t row = rec.idx / p.nchan;
            int chan = (int)(rec.idx - row * p.nchan);
            a = vis[row * vis_rs + chan * vis_cs];
          }
          double w = wgt ? wgt[rec.idx] : 1.0;
          double pc = apply_phase ? rec.pc : 1.0, ps = apply_phase ? rec.ps : 0.0;
          if (apply_phase && (rec.ip & REC_CONJ_BIT)) a.y = -a.y;  // folded sample (the Hessian path stays folded)
          double2 sa;
          sa.x = (a.x * pc - a.y * ps) * w;
          sa.y = (a.x * ps + a.y * pc) * w;
          amp[team][lane] = sa;
          x0s[team][lane][0] = rec.x0[0]; x0s[team][lane][1] = rec.x0[1]; x0s[team][lane][2] = rec.x0[2];
        }
      }
      const uint32_t starts = run_starts(org, cur, lane, nb);
      team_sync(team, 32 * WIDE_R);
      wide_taps(p, x0s[team], taps[team], nb, ttid, 32 * WIDE_R, bscale, xs);
      team_sync(team, 32 * WIDE_R);
      for (int v = 0; v < nb; ++v) {
        if ((starts >> v) & 1u) {
          if (cur != ~0ull) wide_flush(p, grid, accr, acci, cur, j, q2, row0);
          cur = shfl_u64(org, v);
        }
        const double* tp = taps[team][v];
        const double tv = tp[16 + j];
        const double2 a = amp[team][v];
        const double ar = a.x * tv, ai = a.y * tv;
        double ur[WIDE_RPW], ui[WIDE_RPW];
#pragma unroll
        for (int ii = 0; ii < WIDE_RPW; ++ii) { ur[ii] = ar * tp[row0 + ii]; ui[ii] = ai * tp[row0 + ii]; }
#pragma unroll
        for (int qq = 0; qq < WIDE_NQ; ++qq) {
          const double wq = tp[32 + q2 + 2 * qq];
#pragma unroll
          for (int ii = 0; ii < WIDE_RPW; ++ii) {
            accr[ii][qq] += ur[ii] * wq;
            acci[ii][qq] += ui[ii] * wq;
          }
        }
      }
      team_sync(team, 32 * WIDE_R);  // the next batch overwrites the staging buffers
    }
  }
  if (cur != ~0ull) wide_flush(p, grid, accr, acci, cur, j, q2, row0);
}

// Degridding keeps INDEPENDENT warps (measured on B200, C2 band in fp64 at epsilon 1e-7: the cooperative
// variant with team barriers was 17 % slower here, because every new run starts with a footprint fetch whose
// latency the barriers then serialise across the team; for gridding, whose flushes are fire-and-forget, the
// cooperative form above is 19 % faster).  Each warp stages the records and evaluates the taps it needs itself.
__device__ __forceinline__ void wide_taps_warp(const GParams& p, const double (*x0s)[4], double (*taps)[WIDE_RPW + 32],
                                               int nb, int lane, int row0, double bscale, double xs) {
  constexpr int NT = WIDE_RPW + 32;
  for (int idx = lane; idx < NT * nb; idx += 32) {
    const int v = idx / NT, t = idx - v * NT;
    int axis, k;
    if (t < WIDE_RPW) { axis = 0; k = row0 + t; }
    else if (t < WIDE_RPW + 16) { axis = 1; k = t - WIDE_RPW; }
    else { axis = 2; k = t - WIDE_RPW - 16; }
    double val = es_fast((x0s[v][axis] + (double)k) * xs, bscale);
    if (axis == 2 && !p.do_wgridding) val = (k == 0) ? 1.0 : 0.0;
    taps[v][t] = val;
  }
}

// degridding: each warp of the team produces the partial sum over its rows; partials of the WIDE_R
// warps are combined with one atomicAdd per sample and warp into a zero-initialised output.
__global__ void __launch_bounds__(WIDE_WARPS * 32)
k_degrid_runs_wide(GParams p, const VisRec<double>* __restrict__ recs, int64_t nact, const double2* __restrict__ grid,
                   const double* __restrict__ wgt, double2* __restrict__ vis_out, double2* __restrict__ out_sorted,
                   int apply_phase, unsigned long long* __restrict__ queue) {
  constexpr int NB = WIDE_NB, NT = WIDE_RPW + 32;  // taps per sample and warp: WIDE_RPW u, 16 v, 16 w
  __shared__ double taps[WIDE_WARPS][NB][NT];
  __shared__ __align__(16) double x0s[WIDE_WARPS][NB][4];
  __shared__ uint64_t orgs[WIDE_WARPS][NB];
  // per-sample partial sums of the 32 lanes: summed lane <-> sample after the batch (skewed, conflict-free) instead
  // of a 5-level shuffle reduction per sample, whose dependent latency dominated this kernel (ncu: "wait" stalls)
  extern __shared__ __align__(16) unsigned char wide_part_raw[];  // WIDE_WARPS * NB * 32 complex (dynamic: > 48 KB in fp64)
  double2 (*part)[NB][32] = reinterpret_cast<double2 (*)[NB][32]>(wide_part_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = lane & 15, q2 = lane >> 4;
  const int64_t gwarp = (int64_t)blockIdx.x * WIDE_WARPS + warp;
  const int row0 = (int)(gwarp % WIDE_R) * WIDE_RPW;
  const int W = p.W, npl = p.do_wgridding ? W : 1;
  const double bscale = es_scale(p.beta), xs = 2.0 / p.W;
  const int plane_sz = p.nu * p.nv;
  double gr[WIDE_RPW][WIDE_NQ], gi[WIDE_RPW][WIDE_NQ];
#pragma unroll
  for (int ii = 0; ii < WIDE_RPW; ++ii)
#pragma unroll
    for (int qq = 0; qq < WIDE_NQ; ++qq) { gr[ii][qq] = 0; gi[ii][qq] = 0; }
  uint64_t cur = ~0ull;
  const int64_t nslice = (nact + WIDE_SLICE - 1) / WIDE_SLICE;
  // the warps are independent: every (slice, row group) pair is drawn exactly once from the row group's own counter
  unsigned long long* myq = queue + (gwarp % WIDE_R);
  for (;;) {
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(myq, 1ull);
    const int64_t sl = (int64_t)shfl_u64(t, 0);
    if (sl >= nslice) break;
    const int64_t kend = min(nact, (sl + 1) * WIDE_SLICE);
    for (int64_t k0 = sl * WIDE_SLICE; k0 < kend; k0 += NB) {
      const int nb = (int)min((int64_t)NB, kend - k0);
      VisRec<double> r;
      if (lane < nb) {
        r = recs[k0 + lane];
        x0s[warp][lane][0] = r.x0[0]; x0s[warp][lane][1] = r.x0[1]; x0s[warp][lane][2] = r.x0[2];
        orgs[warp][lane] = pack_origin(r.iu, r.iv, r.ip);
      }
      __syncwarp();
      wide_taps_warp(p, x0s[warp], taps[warp], nb, lane, row0, bscale, xs);
      __syncwarp();
      for (int v = 0; v < nb; ++v) {
        const uint64_t org = orgs[warp][v];
        if (org != cur) {
          cur = org;
          int iv = (int)(org & 0xffffu) + j;
          int iu0 = (int)((org >> 16) & 0xffffu);
          int ip = origin_plane(org);
          if (iv >= p.nv) iv -= p.nv;
          const bool jok = j < W;
          if (iu0 >= 1 && iu0 + W <= p.nu) {  // rows do not wrap: constant stride (see wide_flush)
            const int mv = iv ? p.nv - iv : 0;
#pragma unroll
            for (int qq = 0; qq < WIDE_NQ; ++qq) {
              const int q = q2 + 2 * qq, pl = ip + q;
              const bool ok = jok && q < npl, mir = pl < 0;
              const double2* g = grid + (mir ? (int64_t)(-pl - 1) * plane_sz + (int64_t)(p.nu - iu0 - row0) * p.nv + mv
                                             : (int64_t)pl * plane_sz + (int64_t)(iu0 + row0) * p.nv + iv);
              const int step = mir ? -p.nv : p.nv;
#pragma unroll
              for (int ii = 0; ii < WIDE_RPW; ++ii) {
                double2 val; val.x = 0; val.y = 0;
                if (ok && row0 + ii < W) {
                  val = g[ii * step];
                  if (mir) val.y = -val.y;
                }
                gr[ii][qq] = val.x; gi[ii][qq] = val.y;
              }
            }
          } else {
#pragma unroll
          for (int qq = 0; qq < WIDE_NQ; ++qq) {
            const int q = q2 + 2 * qq;
            const bool ok = jok && q < npl;
#pragma unroll
            for (int ii = 0; ii < WIDE_RPW; ++ii) {
              const int i = row0 + ii;
              double2 val; val.x = 0; val.y = 0;
              if (ok && i < W) {
                int iu = iu0 + i;
                if (iu >= p.nu) iu -= p.nu;
                bool cj;
                val = grid[plane_cell(p, ip + q, iu, iv, cj)];
                if (cj) val.y = -val.y;
              }
              gr[ii][qq] = val.x; gi[ii][qq] = val.y;
            }
          }
          }
        }
        const double* tp = taps[warp][v];
        double sr = 0, si = 0;
#pragma unroll
        for (int qq = 0; qq < WIDE_NQ; ++qq) {
          double pr = 0, pi = 0;
#pragma unroll
          for (int ii = 0; ii < WIDE_RPW; ++ii) { pr += gr[ii][qq] * tp[ii]; pi += gi[ii][qq] * tp[ii]; }
          const double wq = tp[WIDE_RPW + 16 + q2 + 2 * qq];
          sr += pr * wq; si += pi * wq;
        }
        const double tv = tp[WIDE_RPW + j];
        double2 pv; pv.x = sr * tv; pv.y = si * tv;
        part[warp][v][lane] = pv;
      }
      __syncwarp();
      if (lane < nb) {
        double myr = 0, myi = 0;
#pragma unroll 8
        for (int l = 0; l < 32; ++l) {
          const double2 pv = part[warp][lane][(lane + l) & 31];
          myr += pv.x; myi += pv.y;
        }
        double re = myr, im = myi;
        if (apply_phase) {
          re = myr * r.pc + myi * r.ps;
          im = myi * r.pc - myr * r.ps;
        }
        if (apply_phase && (r.ip & REC_CONJ_BIT)) im = -im;
        if (wgt) { double w = wgt[r.idx]; re *= w; im *= w; }
        double2* dst = out_sorted ? (out_sorted + k0 + lane) : (vis_out + r.idx);
        atomicAdd(&dst->x, re);
        atomicAdd(&dst->y, im);
      }
      __syncwarp();
    }
  }
}
