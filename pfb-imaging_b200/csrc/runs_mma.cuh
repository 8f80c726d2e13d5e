// fp64 run kernels for 9 <= W <= 12 on the FP64 tensor-core path (DMMA m8n8k4), the production setting of pfb's own
// entry points (precision="double", epsilon 1e-7: W = 12).
//
// A run (all samples whose 12 x 12 x 12 footprint starts at the same grid cell, see runs.cuh) is a small dense
// contraction once the taps are known:
//
//   gridding    C[(i,j), (q,c)] += sum_s  (ku_s[i] kv_s[j]) * (amp_s^c kw_s[q])      M = 144, N = 24, K = samples
//   degridding  D[s, (q,c)]      = sum_(i,j) (ku_s[i] kv_s[j]) * G[(i,j), (q,c)]     M = samples, N = 24, K = 144
//               vis_s            = sum_q kw_s[q] (D[s,(q,0)] + i D[s,(q,1)])
//
// with c = real / imaginary part.  On B200 DMMA runs at the DFMA flop rate (measured: 37 against 34 TFLOP/s), but one
// DMMA replaces 8 DFMA warp instructions, and scalar team kernels (k_*_runs_wide, which serve 13 <= W <= 16) are ISSUE
// bound: ncu on the C2 band at epsilon 1e-7 shows 680 / 980 warp instructions per sample (gridding / degridding)
// against ~200 that are DFMAs, the fp64 pipe ~25 % busy.  Here a sample costs 13.5 DMMAs per direction for the whole
// team and every tap is evaluated once per team.
//
// Team = 3 warps; warp r owns the u-rows 4r .. 4r+3 (48 of the 144 (i,j) cells).
//   gridding:   6 M-tiles (2 rows x 4 columns each) x 3 N-tiles per warp = 36 accumulator doubles per lane; the C
//               fragment of a lane is (re, im) of one cell, so the flush is one complex RED pair per tile.
//   degridding: the warp's 48 cells are 12 k-steps; the B fragments (the run's footprint, 36 doubles per lane) are
//               fetched once per run; 8 samples per MMA step; the three row partials meet in the zero-initialised
//               output through atomics like in k_degrid_runs_wide.
#pragma once
#include "runs.cuh"

#define MMA_R 3        /* warps per team */
#define MMA_TEAMS 1    /* teams per CTA */
#define MMA_NB 32      /* samples staged per batch */
#define MMA_TS 44      /* doubles per staged sample: 12 u-, 12 v-, 12 w-taps, amplitude / phase (3); 44 = 12 mod 16 keeps the
                          4 rows x 4 consecutive slots of a half-warp operand load on distinct 8-byte banks */
#define MMA_ROWS (MMA_NB + 8)  /* MMA steps may read (never use) up to 7 rows past the batch */
#define MMA_SLICE 256
#ifndef MMA_MINB
#define MMA_MINB 5  /* resident 96-thread CTAs per SM the register budget is set for */
#endif

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// ES tap in fp64 without the library's special-case handling: a * rsqrt(a) from the MUFU seed and one third-order
// Newton step instead of the correctly rounded sqrt, e^y (y in [-beta, 0]) by Cody-Waite reduction and a degree-13
// Taylor polynomial on |r| <= ln2 / 2 (coefficients in constant memory: an fp64 immediate costs two extra moves).
// Relative error ~1e-15 beta (tests/test_gpu_mma.py compares the kernels built on it with the exp / sqrt ones);
// ~40 instead of ~73 instructions per tap.
__constant__ double kExpC[12] = {1.6059043836821613e-10, 2.08767569878681e-09,   2.505210838544172e-08,
                                 2.755731922398589e-07,  2.7557319223985893e-06, 2.48015873015873e-05,
                                 1.984126984126984e-04,  1.388888888888889e-03,  8.333333333333333e-03,
                                 4.1666666666666664e-02, 1.6666666666666666e-01, 0.5};  // 1/13! .. 1/2!
__device__ __forceinline__ double exp_neg_fast(double y) {
  const double t = fma(y, 1.4426950408889634, 6755399441055744.0);  // round to nearest through 1.5 * 2^52
  const int n = __double2loint(t);
  const double fn = t - 6755399441055744.0;
  double r = fma(fn, -6.93147180369123816490e-01, y);
  r = fma(fn, -1.90821492927058770002e-10, r);
  double q = kExpC[0];
#pragma unroll
  for (int i = 1; i < 12; ++i) q = fma(q, r, kExpC[i]);
  q = fma(q, r, 1.0);
  q = fma(q, r, 1.0);
  return __hiloint2double(__double2hiint(q) + (n << 20), __double2loint(q));  // * 2^n (q in [0.7, 1.42], n >= -60)
}
// x in [-1, 1] (the taps of a sample never leave the support; |a| absorbs an x that exceeds 1 by a rounding error)
__device__ __forceinline__ double es_fast64(double x, double beta) {
  const double a = fabs(fma(-x, x, 1.0));
  double y0;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(a + 1e-300));  // a == 0 (x == 1): s = 0 * 1e150 = 0
  const double e = fma(a * y0, -y0, 1.0);
  const double y1 = fma(fma(e, 0.375, 0.5), y0 * e, y0);  // 1/sqrt(a) to ~1 ulp
  return exp_neg_fast(beta * fma(a, y1, -1.0));
}

// warp r of the team evaluates the 12 taps of axis r for the sample of its lane (lane <-> sample, no index
// arithmetic, 12 independent evaluations in flight) and writes them as six 16-byte stores
__device__ __forceinline__ void mma_taps_axis(int W, bool flat, double x0, double* __restrict__ dst, double bscale, double xs) {
#pragma unroll
  for (int k = 0; k < 12; k += 2) {
    double t0 = k < W ? es_fast64((x0 + (double)k) * xs, bscale) : 0.0;
    double t1 = k + 1 < W ? es_fast64((x0 + (double)(k + 1)) * xs, bscale) : 0.0;
    if (flat) { t0 = k == 0 ? 1.0 : 0.0; t1 = 0.0; }
    *reinterpret_cast<double2*>(dst + k) = make_double2(t0, t1);
  }
}

// record fields every warp of the team needs: run origin (+ flat index) from the 16-byte tail, tap origin of one axis
__device__ __forceinline__ uint64_t mma_rec(const VisRec<double>* __restrict__ recs, int64_t k, int axis, uint32_t& idx,
                                            int32_t& ipraw, double& x0) {
  const char* b = reinterpret_cast<const char*>(recs + k);
  const uint2 t0 = *reinterpret_cast<const uint2*>(b + 40), t1 = *reinterpret_cast<const uint2*>(b + 48);
  x0 = *reinterpret_cast<const double*>(b + 8 * axis);
  idx = t0.x;
  ipraw = (int32_t)t1.x;
  return pack_origin(t0.y & 0xffffu, t0.y >> 16, ipraw);
}

__device__ __forceinline__ int seg_end(uint32_t starts, int a, int nb) {  // first run start after sample a, or nb
  const uint32_t m = a >= 31 ? 0u : (starts & ~((2u << a) - 1u));
  return m ? __ffs(m) - 1 : nb;
}

// Cyclic column ownership (as in k_grid_runs, here for 12 columns): consecutive runs of a (tile, plane) bucket come
// in the order (iu, iv), so the next run usually starts a few cells further along v and most of its 12 footprint
// columns are the previous run's.  A lane therefore owns the absolute grid column col with col mod 12 == c (c = its
// column class) inside [iv0, iv0 + 12) instead of the column at a fixed offset from the origin; when the origin moves
// by delta < 12 along v, only the delta classes whose column left the footprint are flushed (gridding) / fetched
// (degridding).  The tap a class multiplies is joff = col - iv0 = (c - iv0) mod 12.  Requires a footprint that does not
// wrap and stays off row / column 0 (mirror planes address nu - iu, nv - iv): "fast" runs; others take the general path.
struct RunPos {
  int iu0, iv0, ip, m0;
  bool fast;
};
__device__ __forceinline__ RunPos run_pos(const GParams& p, uint64_t org) {
  RunPos o;
  o.iv0 = (int)(org & 0xffffu);
  o.iu0 = (int)((org >> 16) & 0xffffu);
  o.ip = origin_plane(org);
  o.fast = o.iu0 >= 1 && o.iu0 + 12 <= p.nu && o.iv0 >= 1 && o.iv0 + 12 <= p.nv;
  o.m0 = o.iv0 % 12;
  return o;
}
__device__ __forceinline__ int col_off(int c, int m0) {  // (c - iv0) mod 12
  const int j = c - m0;
  return j < 0 ? j + 12 : j;
}
// columns shared by two fast runs: same rows and planes, origin moved forward along v -> number of columns that left
__device__ __forceinline__ int run_shift(const RunPos& o, const RunPos& n) {
  if (!(o.fast && n.fast) || o.iu0 != n.iu0 || o.ip != n.ip || n.iv0 <= o.iv0) return 12;
  const int d = n.iv0 - o.iv0;
  return d < 12 ? d : 12;
}

__global__ void __launch_bounds__(MMA_R* MMA_TEAMS * 32, MMA_MINB)
k_grid_runs_mma(GParams p, const VisRec<double>* __restrict__ recs, int64_t nact, const double2* __restrict__ vis,
                int64_t vis_rs, int64_t vis_cs, const double* __restrict__ wgt, double2* __restrict__ grid,
                int vis_sorted, int apply_phase, unsigned long long* __restrict__ queue) {
  // staged samples, double buffered: batch b + 1 is written while slower warps of the team still read batch b
  __shared__ __align__(16) double stb[MMA_TEAMS][2][MMA_ROWS][MMA_TS];
  __shared__ unsigned long long team_slice[MMA_TEAMS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = warp / MMA_R, r = warp - team * MMA_R;
  const int ttid = r * 32 + lane;
  const int g = lane >> 2, l3 = lane & 3;
  const int W = p.W, npl = p.do_wgridding ? W : 1;
  const double bscale = p.beta, xs = 2.0 / p.W;
  const bool flat = r == 2 && !p.do_wgridding;
  const int64_t plane_sz = (int64_t)p.nu * p.nv;
  int buf = 0;
  // operand slots of this lane inside a staged sample (see the tile layout above)
  const int rowl = 4 * r + (g >> 2);      // + 2 * rp : footprint row of the A / C elements
  const int cl = g & 3;                   // + 4 * jg : column class of the A / C elements
  const int bw = 24 + (lane >> 3);        // + 4 * nt : w-tap of the B element
  const int bc = 36 + (g & 1);            // amplitude component of the B element
  double acc[6][3][2];
#pragma unroll
  for (int t = 0; t < 6; ++t)
#pragma unroll
    for (int n = 0; n < 3; ++n) { acc[t][n][0] = 0; acc[t][n][1] = 0; }
  for (int v = ttid; v < 2 * (MMA_ROWS - MMA_NB); v += 32 * MMA_R)  // rows past the batch are read by masked steps: keep them finite
    for (int t = 0; t < MMA_TS; ++t) stb[team][v & 1][MMA_NB + (v >> 1)][t] = 0.0;
  uint64_t cur = ~0ull;
  RunPos cp;
  cp.fast = false; cp.iu0 = cp.iv0 = cp.ip = cp.m0 = 0;
  int kvi[3] = {12 + cl, 16 + cl, 20 + cl};  // v-tap slots of the three column classes for the current run

  // general flush: column at offset j = class from the origin, wrap-around and row / column 0 handled by plane_cell
  auto flush_general = [&]() {
#pragma unroll
    for (int t = 0; t < 6; ++t) {
      const int i = rowl + 2 * (t / 3), j = 4 * (t % 3) + cl;
      int iu = cp.iu0 + i, iv = cp.iv0 + j;
      if (iu >= p.nu) iu -= p.nu;
      if (iv >= p.nv) iv -= p.nv;
      const bool ok = i < W && j < W;
#pragma unroll
      for (int n = 0; n < 3; ++n) {
        const int q = 4 * n + l3;
        if (ok && q < npl) {
          bool cj;
          double2* dst = grid + plane_cell(p, cp.ip + q, iu, iv, cj);
          atomic_add_c(dst, acc[t][n][0], cj ? -acc[t][n][1] : acc[t][n][1]);
        }
        acc[t][n][0] = 0;
        acc[t][n][1] = 0;
      }
    }
  };
  // fast flush of the column classes whose column lies in the first `delta` columns of the current footprint
  auto flush_cols = [&](int delta) {
    const int64_t prow = (int64_t)(cp.iu0 + rowl) * p.nv, mrow = (int64_t)(p.nu - cp.iu0 - rowl) * p.nv;
#pragma unroll
    for (int jg = 0; jg < 3; ++jg) {
      const int joff = col_off(4 * jg + cl, cp.m0);
      const bool fl = joff < delta;
      if (__any_sync(0xffffffffu, fl)) {
        if (fl) {
          const int col = cp.iv0 + joff;
#pragma unroll
          for (int n = 0; n < 3; ++n) {
            const int q = 4 * n + l3, pl = cp.ip + q;
            if (q < npl) {
              const bool mir = pl < 0;
              double2* base = grid + (mir ? (int64_t)(-pl - 1) * plane_sz + mrow + (p.nv - col) : (int64_t)pl * plane_sz + prow + col);
              const int64_t step = mir ? -2 * (int64_t)p.nv : 2 * (int64_t)p.nv;
#pragma unroll
              for (int rp = 0; rp < 2; ++rp)
                if (rowl + 2 * rp < W)
                  atomic_add_c(base + rp * step, acc[rp * 3 + jg][n][0], mir ? -acc[rp * 3 + jg][n][1] : acc[rp * 3 + jg][n][1]);
            }
#pragma unroll
            for (int rp = 0; rp < 2; ++rp) { acc[rp * 3 + jg][n][0] = 0; acc[rp * 3 + jg][n][1] = 0; }
          }
        }
      }
    }
  };

  const int64_t nslice = (nact + MMA_SLICE - 1) / MMA_SLICE;
  for (;;) {
    if (ttid == 0) team_slice[team] = atomicAdd(queue, 1ull);
    team_sync(team, 32 * MMA_R);
    const int64_t sl = (int64_t)team_slice[team];
    team_sync(team, 32 * MMA_R);
    if (sl >= nslice) break;
    const int64_t kend = min(nact, (sl + 1) * MMA_SLICE);
    for (int64_t k0 = sl * MMA_SLICE; k0 < kend; k0 += MMA_NB) {
      const int nb = (int)min((int64_t)MMA_NB, kend - k0);
      // lane <-> sample: run origin, the 12 taps of axis r; warp 0 also stages weight * phase * visibility
      double (*st)[MMA_TS] = stb[team][buf];
      buf ^= 1;
      uint64_t org = ~0ull;
      double x0 = 0.5 - 0.5 * W;  // lanes past the batch: any position inside the support keeps their rows finite
      double2 sa = make_double2(0.0, 0.0);
      if (lane < nb) {
        const int64_t k = k0 + lane;
        uint32_t idx;
        int32_t ipraw;
        org = mma_rec(recs, k, r, idx, ipraw, x0);
        if (r == 0) {
          double2 a;
          if (vis_sorted) a = vis[k];
          else {
            const int64_t row = idx / p.nchan;
            const int chan = (int)(idx - row * p.nchan);
            a = vis[row * vis_rs + chan * vis_cs];
          }
          const double w = wgt ? wgt[idx] : 1.0;
          double pc = 1.0, ps = 0.0;
          if (apply_phase) {
            pc = recs[k].pc; ps = recs[k].ps;
            if (ipraw & REC_CONJ_BIT) a.y = -a.y;  // folded sample (the Hessian path stays folded)
          }
          sa.x = (a.x * pc - a.y * ps) * w;
          sa.y = (a.x * ps + a.y * pc) * w;
        }
      }
      mma_taps_axis(W, flat, x0, &st[lane][12 * r], bscale, xs);
      if (r == 0) *reinterpret_cast<double2*>(&st[lane][36]) = sa;
      const uint32_t starts = run_starts(org, cur, lane, nb);
      team_sync(team, 32 * MMA_R);
      int a = 0;
      while (a < nb) {
        if ((starts >> a) & 1u) {
          const uint64_t nxt = shfl_u64(org, a);
          const RunPos np_ = run_pos(p, nxt);
          if (cur != ~0ull) {
            if (cp.fast) flush_cols(run_shift(cp, np_));
            else flush_general();
          }
          cur = nxt;
          cp = np_;
#pragma unroll
          for (int jg = 0; jg < 3; ++jg) kvi[jg] = 12 + (cp.fast ? col_off(4 * jg + cl, cp.m0) : 4 * jg + cl);
        }
        const int b = seg_end(starts, a, nb);
        for (int v = a; v < b; v += 4) {
          const double* tp = st[v + l3];
          const bool valid = v + l3 < b;
          const double am = tp[bc];
          double B[3], A[6];
#pragma unroll
          for (int n = 0; n < 3; ++n) B[n] = valid ? am * tp[bw + 4 * n] : 0.0;
          double ku[2], kv[3];
          ku[0] = tp[rowl]; ku[1] = tp[rowl + 2];
#pragma unroll
          for (int jg = 0; jg < 3; ++jg) kv[jg] = tp[kvi[jg]];
#pragma unroll
          for (int t = 0; t < 6; ++t) A[t] = ku[t / 3] * kv[t % 3];
#pragma unroll
          for (int t = 0; t < 6; ++t)
#pragma unroll
            for (int n = 0; n < 3; ++n) dmma884(acc[t][n][0], acc[t][n][1], A[t], B[n]);
        }
        a = b;
      }
    }
  }
  if (cur != ~0ull) {
    if (cp.fast) flush_cols(12);
    else flush_general();
  }
}

// Degridding.  Taps are shared by the team (named barriers); the footprint of a run lives in the B fragments and only
// the column classes that entered the footprint are fetched when the run origin moves along v.
__global__ void __launch_bounds__(MMA_R* MMA_TEAMS * 32, MMA_MINB)
k_degrid_runs_mma(GParams p, const VisRec<double>* __restrict__ recs, int64_t nact, const double2* __restrict__ grid,
                  const double* __restrict__ wgt, double2* __restrict__ vis_out, double2* __restrict__ out_sorted,
                  int apply_phase, unsigned long long* __restrict__ queue) {
  __shared__ __align__(16) double stb[MMA_TEAMS][2][MMA_ROWS][MMA_TS];
  __shared__ uint32_t sidxb[MMA_TEAMS][2][MMA_NB];
  __shared__ unsigned long long team_slice[MMA_TEAMS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = warp / MMA_R, r = warp - team * MMA_R;
  const int ttid = r * 32 + lane;
  const int g = lane >> 2, l3 = lane & 3;
  const int W = p.W, npl = p.do_wgridding ? W : 1;
  const double bscale = p.beta, xs = 2.0 / p.W;
  const int64_t plane_sz = (int64_t)p.nu * p.nv;
  const double* gd = reinterpret_cast<const double*>(grid);
  const int cpart = g & 1;
  const bool flat = r == 2 && !p.do_wgridding;
  int buf = 0;
  // B fragments: cell (row 4r + ks/3, column class 4 (ks%3) + l3), plane q = 4 nt + (lane >> 3), part c = g & 1
  double gb[12][3];
#pragma unroll
  for (int ks = 0; ks < 12; ++ks)
#pragma unroll
    for (int n = 0; n < 3; ++n) gb[ks][n] = 0.0;
  for (int v = ttid; v < 2 * (MMA_ROWS - MMA_NB); v += 32 * MMA_R)
    for (int t = 0; t < MMA_TS; ++t) stb[team][v & 1][MMA_NB + (v >> 1)][t] = 0.0;
  uint64_t cur = ~0ull;
  RunPos cp;
  cp.fast = false; cp.iu0 = cp.iv0 = cp.ip = cp.m0 = 0;
  int kvi[3] = {12 + l3, 16 + l3, 20 + l3};

  auto fetch_general = [&]() {
#pragma unroll
    for (int ks = 0; ks < 12; ++ks) {
      const int i = 4 * r + ks / 3, j = 4 * (ks % 3) + l3;
      int iu = cp.iu0 + i, iv = cp.iv0 + j;
      if (iu >= p.nu) iu -= p.nu;
      if (iv >= p.nv) iv -= p.nv;
      const bool ok = i < W && j < W;
#pragma unroll
      for (int n = 0; n < 3; ++n) {
        const int q = 4 * n + (lane >> 3);
        double val = 0.0;
        if (ok && q < npl) {
          bool cj;
          val = gd[2 * plane_cell(p, cp.ip + q, iu, iv, cj) + cpart];
          if (cj && cpart) val = -val;
        }
        gb[ks][n] = val;
      }
    }
  };
  // fast fetch of the column classes whose column lies in the last `delta` columns of the current footprint
  auto fetch_cols = [&](int delta) {
    const int64_t prow = (int64_t)(cp.iu0 + 4 * r) * p.nv, mrow = (int64_t)(p.nu - cp.iu0 - 4 * r) * p.nv;
#pragma unroll
    for (int jg = 0; jg < 3; ++jg) {
      const int joff = col_off(4 * jg + l3, cp.m0);
      const bool ld = joff >= 12 - delta;
      if (__any_sync(0xffffffffu, ld)) {
        if (ld) {
          const int col = cp.iv0 + joff;
#pragma unroll
          for (int n = 0; n < 3; ++n) {
            const int q = 4 * n + (lane >> 3), pl = cp.ip + q;
            const bool mir = pl < 0;
            const double* base = gd + 2 * (mir ? (int64_t)(-pl - 1) * plane_sz + mrow + (p.nv - col) : (int64_t)pl * plane_sz + prow + col) + cpart;
            const int64_t step = mir ? -2 * (int64_t)p.nv : 2 * (int64_t)p.nv;
            const bool okq = q < npl;
#pragma unroll
            for (int ii = 0; ii < 4; ++ii) {
              double val = 0.0;
              if (okq && 4 * r + ii < W) val = base[ii * step];
              gb[3 * ii + jg][n] = (mir && cpart) ? -val : val;
            }
          }
        }
      }
    }
  };

  const int64_t nslice = (nact + MMA_SLICE - 1) / MMA_SLICE;
  for (;;) {
    if (ttid == 0) team_slice[team] = atomicAdd(queue, 1ull);
    team_sync(team, 32 * MMA_R);
    const int64_t sl = (int64_t)team_slice[team];
    team_sync(team, 32 * MMA_R);
    if (sl >= nslice) break;
    const int64_t kend = min(nact, (sl + 1) * MMA_SLICE);
    for (int64_t k0 = sl * MMA_SLICE; k0 < kend; k0 += MMA_NB) {
      const int nb = (int)min((int64_t)MMA_NB, kend - k0);
      // lane <-> sample: run origin, the 12 taps of axis r; warp 0 also stages phase, weight and the output slot
      double (*st)[MMA_TS] = stb[team][buf];
      uint32_t* sidx = sidxb[team][buf];
      buf ^= 1;
      uint64_t org = ~0ull;
      double x0 = 0.5 - 0.5 * W, pcw = 0.0, psw = 0.0, sg = 1.0;  // lanes past the batch: finite rows
      uint32_t idx = 0;
      if (lane < nb) {
        int32_t ipraw;
        org = mma_rec(recs, k0 + lane, r, idx, ipraw, x0);
        if (r == 0) {
          // out = w e^{-it} sum, conjugated for folded samples:
          //   re = w (sr pc + si ps), im = +-w (si pc - sr ps); slot 38 holds the sign
          const double w = wgt ? wgt[idx] : 1.0;
          pcw = w;
          if (apply_phase) {
            pcw = recs[k0 + lane].pc * w; psw = recs[k0 + lane].ps * w;
            if (ipraw & REC_CONJ_BIT) sg = -1.0;
          }
        }
      }
      mma_taps_axis(W, flat, x0, &st[lane][12 * r], bscale, xs);
      if (r == 0) {
        *reinterpret_cast<double2*>(&st[lane][36]) = make_double2(pcw, psw);
        st[lane][38] = sg;
        sidx[lane] = idx;
      }
      const uint32_t starts = run_starts(org, cur, lane, nb);
      team_sync(team, 32 * MMA_R);
      int a = 0;
      while (a < nb) {
        if ((starts >> a) & 1u) {
          const uint64_t nxt = shfl_u64(org, a);
          const RunPos np_ = run_pos(p, nxt);
          const int delta = cur != ~0ull ? run_shift(cp, np_) : 12;
          cur = nxt;
          cp = np_;
          if (cp.fast) fetch_cols(delta);
          else fetch_general();
#pragma unroll
          for (int jg = 0; jg < 3; ++jg) kvi[jg] = 12 + (cp.fast ? col_off(4 * jg + l3, cp.m0) : 4 * jg + l3);
        }
        const int b = seg_end(starts, a, nb);
        for (int v = a; v < b; v += 8) {
          const int s = v + g;  // this lane's sample in the A / D fragments
          const double* tp = st[s];
          double ku[4], kv[3];
#pragma unroll
          for (int ii = 0; ii < 4; ++ii) ku[ii] = tp[4 * r + ii];
#pragma unroll
          for (int jg = 0; jg < 3; ++jg) kv[jg] = tp[kvi[jg]];
          double d[2][3][2];
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int n = 0; n < 3; ++n) { d[h][n][0] = 0; d[h][n][1] = 0; }
#pragma unroll
          for (int ks = 0; ks < 12; ++ks) {
            const double A = ku[ks / 3] * kv[ks % 3];
#pragma unroll
            for (int n = 0; n < 3; ++n) dmma884(d[ks & 1][n][0], d[ks & 1][n][1], A, gb[ks][n]);
          }
          // D fragment: sample s, plane q = 4 n + l3, (re, im)
          double sr = 0, si = 0;
#pragma unroll
          for (int n = 0; n < 3; ++n) {
            const double kw = tp[24 + 4 * n + l3];
            sr += (d[0][n][0] + d[1][n][0]) * kw;
            si += (d[0][n][1] + d[1][n][1]) * kw;
          }
          sr += __shfl_xor_sync(0xffffffffu, sr, 1); si += __shfl_xor_sync(0xffffffffu, si, 1);
          sr += __shfl_xor_sync(0xffffffffu, sr, 2); si += __shfl_xor_sync(0xffffffffu, si, 2);
          if (s < b && l3 < 2) {
            const double pcw = tp[36], psw = tp[37];
            // l3 == 0 adds the real part, l3 == 1 the imaginary part
            const double val = l3 == 0 ? sr * pcw + si * psw : (si * pcw - sr * psw) * tp[38];
            double2* dst = out_sorted ? (out_sorted + k0 + s) : (vis_out + sidx[s]);
            atomicAdd(reinterpret_cast<double*>(dst) + l3, val);
          }
        }
        a = b;
      }
    }
  }
}
