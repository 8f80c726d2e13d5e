// fp32 "pair" FFT engine: two interleaved transforms (two neighbouring grid columns, or two image rows) are
// carried through every butterfly as ONE packed value, so the whole transform runs on the two-wide fp32
// pipe of sm_100 (FADD2 / FMUL2 / FFMA2, scalar twiddles broadcast by the instruction): half the math
// instructions per transform of fft.cuh's scalar engine, 16-byte shared-memory accesses.
//
// Shared-memory element n (a "pair element") is 16 bytes {re0, re1, im0, im1} — the real parts of transform
// 0 and 1 in one 64-bit register pair, the imaginary parts in the other.  Element e lives in the 16-byte
// chunk  sw2(e) = e ^ ((e >> 3) & 7) (chunk index bits 0-2 ^= bits 3-5: the 128-byte XOR swizzle): no padding and
// no bank conflicts in the late stages (a lane's 8 consecutive rows share one 128-byte line; the XOR spreads the
// lanes of a warp over the 8 chunks).
//
// NP interleaved pair elements per transform index (NP = 1, 2, 4): element (n, p) has index n * NP + p
// (several column pairs per CTA for short transforms).
//
// Forward transform only (e^{-2 pi i nk/N}), decimation in frequency: natural-order input, output in the
// mixed-radix digit-reversed order of fft.cuh (pos -> k = rev[pos]).  The inverse is swap-in / swap-out:
// IDFT(x) = swap(DFT(swap(x))) with swap(a + ib) = b + ia, which costs nothing in this layout.
// The first stage can read its input in the dense array-of-structures order global memory (and the TMA unit)
// delivers, {re0, im0, re1, im1} at chunk e, and writes swizzled pair elements (see p2_stage, DENSE).
#pragma once
#include "fft.cuh"

typedef unsigned long long u64;
struct pc2 { u64 r, i; };  // two complex numbers: r = (re0, re1), i = (im0, im1)

__device__ __forceinline__ u64 f2add(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 f2sub(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 f2mul(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 f2fma(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 f2bc(float f) { u64 d; asm("mov.b64 %0, {%1, %1};" : "=l"(d) : "f"(f)); return d; }  // (f, f): a broadcast operand in SASS
__device__ __forceinline__ u64 f2pack(float a, float b) { u64 d; asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(a), "f"(b)); return d; }
__device__ __forceinline__ void f2unpack(u64 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }

__device__ __forceinline__ pc2 padd(pc2 a, pc2 b) { return {f2add(a.r, b.r), f2add(a.i, b.i)}; }
__device__ __forceinline__ pc2 psub(pc2 a, pc2 b) { return {f2sub(a.r, b.r), f2sub(a.i, b.i)}; }
// a + (-i) b  and  a - (-i) b   ((-i) b = (b.i, -b.r))
__device__ __forceinline__ pc2 padd_mi(pc2 a, pc2 b) { return {f2add(a.r, b.i), f2sub(a.i, b.r)}; }
__device__ __forceinline__ pc2 psub_mi(pc2 a, pc2 b) { return {f2sub(a.r, b.i), f2add(a.i, b.r)}; }
// x * (c + i s), scalar twiddle shared by both transforms: 4 packed instructions for two complex products
__device__ __forceinline__ pc2 pmulw(pc2 x, float c, float s) {
  const u64 t = f2mul(x.r, f2bc(c)), u = f2mul(x.r, f2bc(s));
  return {f2fma(x.i, f2bc(-s), t), f2fma(x.i, f2bc(c), u)};
}
__device__ __forceinline__ float2 cmulf(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

__device__ __forceinline__ int sw2(int e) { return e ^ ((e >> 3) & 7); }

// Twiddles from SHARED memory: e^{-2 pi i t/N} = coarse[t >> 6] * fine[t & 63] (N/64 + 64 table entries instead of N;
// a global-memory table costs an L2 round trip per butterfly — with one or two butterflies per thread and stage
// nothing hides it: ncu showed a quarter of the column kernel's stall samples on the first use of the twiddle).
struct P2Tw {
  const float2* coarse;  // [ceil(N/64)]: e^{-2 pi i 64 j/N}
  const float2* fine;    // [64]:         e^{-2 pi i f/N}
};
__device__ __forceinline__ int p2_tw_entries(int N) { return (N + 63) / 64 + 64; }
// fill the two tables (at `dst`, p2_tw_entries(N) float2) from the full global table tw[t] = e^{-2 pi i t/N}
__device__ __forceinline__ P2Tw p2_tw_fill(float2* dst, const float2* __restrict__ tw, int N, int tid, int nthr) {
  const int nc = (N + 63) / 64;
  for (int j = tid; j < nc; j += nthr) dst[j] = tw[64 * j];
  for (int f = tid; f < 64; f += nthr) dst[nc + f] = f < N ? tw[f] : make_float2(1.f, 0.f);
  return {dst, dst + nc};
}
__device__ __forceinline__ float2 p2_tw_get(const P2Tw& tw, int t) {
  const float2 a = tw.coarse[t >> 6], b = tw.fine[t & 63];
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

__device__ __forceinline__ void pbf4(pc2& a, pc2& b, pc2& c, pc2& d) {
  const pc2 t0 = padd(a, c), t1 = psub(a, c), t2 = padd(b, d), bd = psub(b, d);
  a = padd(t0, t2);
  c = psub(t0, t2);
  b = padd_mi(t1, bd);
  d = psub_mi(t1, bd);
}

template <int R> struct PDft;
template <> struct PDft<2> {
  __device__ static __forceinline__ void run(pc2* x) {
    const pc2 t = psub(x[0], x[1]);
    x[0] = padd(x[0], x[1]);
    x[1] = t;
  }
};
template <> struct PDft<4> {
  __device__ static __forceinline__ void run(pc2* x) { pbf4(x[0], x[1], x[2], x[3]); }
};
template <> struct PDft<8> {
  __device__ static __forceinline__ void run(pc2* x) {
    pc2 e0 = x[0], e1 = x[2], e2 = x[4], e3 = x[6];
    pc2 o0 = x[1], o1 = x[3], o2 = x[5], o3 = x[7];
    pbf4(e0, e1, e2, e3);
    pbf4(o0, o1, o2, o3);
    const u64 h = f2bc(0.70710678118654752440f);
    // o1 * (1 - i)/sqrt2 = ((r + i) h, (i - r) h);   o3 * (-1 - i)/sqrt2 = ((i - r) h, -(r + i) h)
    const pc2 p1 = {f2mul(f2add(o1.r, o1.i), h), f2mul(f2sub(o1.i, o1.r), h)};
    const u64 p3 = f2mul(f2sub(o3.i, o3.r), h), q3 = f2mul(f2add(o3.r, o3.i), h);
    x[0] = padd(e0, o0); x[4] = psub(e0, o0);
    x[1] = padd(e1, p1); x[5] = psub(e1, p1);
    x[2] = padd_mi(e2, o2); x[6] = psub_mi(e2, o2);
    x[3] = {f2add(e3.r, p3), f2sub(e3.i, q3)};
    x[7] = {f2sub(e3.r, p3), f2add(e3.i, q3)};
  }
};
template <> struct PDft<16> {
  __device__ static __forceinline__ void run(pc2* x) {
    // n = 4 n1 + n2, k = k1 + 4 k2: A[n2][k1] = DFT4_{n1} x[4 n1 + n2]; A *= W16^{n2 k1}; X[k1 + 4 k2] = DFT4_{n2} A
    pc2 a[4][4];
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) {
      a[n2][0] = x[n2]; a[n2][1] = x[4 + n2]; a[n2][2] = x[8 + n2]; a[n2][3] = x[12 + n2];
      pbf4(a[n2][0], a[n2][1], a[n2][2], a[n2][3]);
    }
    const float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f, h = 0.70710678118654752440f;
    // W16^m = cos(pi m/8) - i sin(pi m/8)
    a[1][1] = pmulw(a[1][1], c1, -s1); a[1][2] = pmulw(a[1][2], h, -h);  a[1][3] = pmulw(a[1][3], s1, -c1);
    a[2][1] = pmulw(a[2][1], h, -h);   a[2][2] = {a[2][2].i, f2sub(0ull, a[2][2].r)}; a[2][3] = pmulw(a[2][3], -h, -h);
    a[3][1] = pmulw(a[3][1], s1, -c1); a[3][2] = pmulw(a[3][2], -h, -h); a[3][3] = pmulw(a[3][3], -c1, s1);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) {
      pbf4(a[0][k1], a[1][k1], a[2][k1], a[3][k1]);
      x[k1] = a[0][k1]; x[k1 + 4] = a[1][k1]; x[k1 + 8] = a[2][k1]; x[k1 + 12] = a[3][k1];
    }
  }
};
template <> struct PDft<3> {
  __device__ static __forceinline__ void run(pc2* x) {
    const float s = 0.86602540378443864676f;
    const pc2 t = padd(x[1], x[2]), d = psub(x[1], x[2]);
    const pc2 m = {f2fma(t.r, f2bc(-0.5f), x[0].r), f2fma(t.i, f2bc(-0.5f), x[0].i)};
    x[0] = padd(x[0], t);
    // m -+ i s d
    x[1] = {f2fma(d.i, f2bc(s), m.r), f2fma(d.r, f2bc(-s), m.i)};
    x[2] = {f2fma(d.i, f2bc(-s), m.r), f2fma(d.r, f2bc(s), m.i)};
  }
};
template <int R> __device__ __forceinline__ void pdft_direct(pc2* x) {
  pc2 y[R];
#pragma unroll
  for (int k = 0; k < R; ++k) {
    pc2 acc = x[0];
#pragma unroll
    for (int n = 1; n < R; ++n) {
      double c, s;
      root_of_unity<R>((n * k) % R, c, s);  // e^{-2 pi i nk/R} = c - i s
      const float cc = (float)c, ss = (float)s;
      acc.r = f2fma(x[n].r, f2bc(cc), acc.r);
      acc.r = f2fma(x[n].i, f2bc(ss), acc.r);
      acc.i = f2fma(x[n].i, f2bc(cc), acc.i);
      acc.i = f2fma(x[n].r, f2bc(-ss), acc.i);
    }
    y[k] = acc;
  }
#pragma unroll
  for (int k = 0; k < R; ++k) x[k] = y[k];
}
template <> struct PDft<5> { __device__ static __forceinline__ void run(pc2* x) { pdft_direct<5>(x); } };
template <> struct PDft<7> { __device__ static __forceinline__ void run(pc2* x) { pdft_direct<7>(x); } };
template <> struct PDft<11> { __device__ static __forceinline__ void run(pc2* x) { pdft_direct<11>(x); } };

// x[m] *= w^m, m = 1..R-1, the powers composed from one table value by scalar products of depth <= 3
// (R = 16: w^(4a+b) = w^(4a) w^b, 14 products; shared by the two transforms of the pair)
template <int R>
__device__ __forceinline__ void ptwiddle(pc2* x, float2 w1) {
  x[1] = pmulw(x[1], w1.x, w1.y);
  if constexpr (R == 2) return;
  const float2 w2 = cmulf(w1, w1);
  x[2] = pmulw(x[2], w2.x, w2.y);
  if constexpr (R == 3) return;
  const float2 w3 = cmulf(w2, w1);
  x[3] = pmulw(x[3], w3.x, w3.y);
  if constexpr (R == 4) return;
  if constexpr (R == 8 || R == 16) {
    const float2 w4 = cmulf(w2, w2);
    x[4] = pmulw(x[4], w4.x, w4.y);
    float2 t;
    t = cmulf(w4, w1); x[5] = pmulw(x[5], t.x, t.y);
    t = cmulf(w4, w2); x[6] = pmulw(x[6], t.x, t.y);
    t = cmulf(w4, w3); x[7] = pmulw(x[7], t.x, t.y);
    if constexpr (R == 16) {
      const float2 w8 = cmulf(w4, w4);
      x[8] = pmulw(x[8], w8.x, w8.y);
      t = cmulf(w8, w1); x[9] = pmulw(x[9], t.x, t.y);
      t = cmulf(w8, w2); x[10] = pmulw(x[10], t.x, t.y);
      t = cmulf(w8, w3); x[11] = pmulw(x[11], t.x, t.y);
      const float2 w12 = cmulf(w8, w4);
      x[12] = pmulw(x[12], w12.x, w12.y);
      t = cmulf(w12, w1); x[13] = pmulw(x[13], t.x, t.y);
      t = cmulf(w12, w2); x[14] = pmulw(x[14], t.x, t.y);
      t = cmulf(w12, w3); x[15] = pmulw(x[15], t.x, t.y);
    }
  } else {
    float2 wm = w3;
#pragma unroll
    for (int m = 4; m < R; ++m) {
      wm = cmulf(wm, w1);
      x[m] = pmulw(x[m], wm.x, wm.y);
    }
  }
}

// input of the first stage: pair elements (swizzled), or dense array-of-structures, optionally re <-> im swapped
enum { P2_IN_PAIR = 0, P2_IN_AOS = 1, P2_IN_AOS_SWAP = 2 };

__device__ __forceinline__ pc2 p2_load(const float4* __restrict__ s, int chunk) {
  const ulonglong2 t = reinterpret_cast<const ulonglong2*>(s)[chunk];
  return {t.x, t.y};
}
__device__ __forceinline__ void p2_store(float4* __restrict__ s, int chunk, pc2 v) {
  reinterpret_cast<ulonglong2*>(s)[chunk] = make_ulonglong2(v.r, v.i);
}

// One DIF stage over the whole array.  L: current block length, M = L / R the butterfly stride.
//   MODE 0: any stride, the swizzle is evaluated per access
//   MODE 1: M * NP is a multiple of 64: the XOR term is the same for all R elements (one swizzled base + m * stride)
//   MODE 2: M * NP == 8 and R * 8 is a multiple of 64 (R = 8, 16): chunk = base + 8 m + (k ^ (m & 7))
//   MODE 3: M == 1, NP == 1, R == 8: one 128-byte line per butterfly, chunk = base + (m ^ (g & 7))
// DENSE (first stage only): the input is array-of-structures {re0, im0, re1, im1} at the UNswizzled chunk e — what
// cp.async.bulk.tensor (no hardware swizzle) or a plain row copy delivers.  The stage writes swizzled pair
// elements in place: the 8 chunks of a 128-byte line trade places, and with M * NP a multiple of 8 those are 8
// consecutive work items, i.e. lanes of ONE warp — a __syncwarp() between its loads and stores is all the ordering
// needed (every warp iterates the same number of times; `nthr` is a multiple of 32).
// VAR: 0 = DIF stage (butterfly, then output m *= W_L^{k m}), 1 = DIF stage with DENSE input, 2 = DIT stage (input m
// *= W_L^{k m}, then butterfly)
enum { P2_DIF = 0, P2_DIF_DENSE = 1, P2_DIT = 2 };
template <int R, int NP, int MODE, int VAR>
__device__ __forceinline__ void p2_stage(float4* __restrict__ s, const P2Tw& tw, int N, int L, int swap,
                                         int tid, int nthr) {
  constexpr bool DENSE = VAR == P2_DIF_DENSE, DIT = VAR == P2_DIT;
  constexpr int LGNP = NP == 1 ? 0 : (NP == 2 ? 1 : 2);
  const int M = L / R, MC = M * NP;
  const int tstride = N / L;
  const int nitems = (N / R) * NP;
  const bool pow2 = (M & (M - 1)) == 0;
  const int lgM = 31 - __clz(M);
  const int wend = DENSE ? ((nitems + 31) & ~31) : nitems;
  for (int w_ = tid; w_ < wend; w_ += nthr) {
    const bool act = !DENSE || w_ < nitems;
    const int w = act ? w_ : nitems - 1;  // idle lanes of the last warp load a valid item too (and store nothing)
    const int p = w & (NP - 1), bk = w >> LGNP;
    const int g = pow2 ? (bk >> lgM) : (bk / M);
    const int k = bk - g * M;
    float2 w1 = make_float2(1.f, 0.f);
    if (M > 1) w1 = (tstride & 63) ? p2_tw_get(tw, k * tstride) : tw.coarse[(k * tstride) >> 6];
    const int e0 = ((g * L + k) << LGNP) + p;
    pc2 x[R];
    int base = 0, kx = 0;
    if constexpr (MODE == 1) base = sw2(e0);
    else if constexpr (MODE == 2) { base = e0 & ~7; kx = e0 & 7; }
    else if constexpr (MODE == 3) { base = e0; kx = g & 7; }
    if constexpr (DENSE) {
#pragma unroll
      for (int m = 0; m < R; ++m) {
        const float4 t = s[e0 + m * MC];  // {re0, im0, re1, im1}
        const u64 re = f2pack(t.x, t.z), im = f2pack(t.y, t.w);
        x[m].r = swap ? im : re;
        x[m].i = swap ? re : im;
      }
      __syncwarp();
    } else if constexpr (MODE == 1) {
#pragma unroll
      for (int m = 0; m < R; ++m) x[m] = p2_load(s, base + m * MC);
    } else if constexpr (MODE == 2) {
#pragma unroll
      for (int m = 0; m < R; ++m) x[m] = p2_load(s, base + 8 * m + (kx ^ (m & 7)));
    } else if constexpr (MODE == 3) {
#pragma unroll
      for (int m = 0; m < R; ++m) x[m] = p2_load(s, base + (m ^ kx));
    } else {
#pragma unroll
      for (int m = 0; m < R; ++m) x[m] = p2_load(s, sw2(e0 + m * MC));
    }
    if (!act) continue;
    if (DIT && M > 1) ptwiddle<R>(x, w1);
    PDft<R>::run(x);
    if (!DIT && M > 1) ptwiddle<R>(x, w1);
    if constexpr (MODE == 1) {
#pragma unroll
      for (int m = 0; m < R; ++m) p2_store(s, base + m * MC, x[m]);
    } else if constexpr (MODE == 2) {
#pragma unroll
      for (int m = 0; m < R; ++m) p2_store(s, base + 8 * m + (kx ^ (m & 7)), x[m]);
    } else if constexpr (MODE == 3) {
#pragma unroll
      for (int m = 0; m < R; ++m) p2_store(s, base + (m ^ kx), x[m]);
    } else {
#pragma unroll
      for (int m = 0; m < R; ++m) p2_store(s, sw2(e0 + m * MC), x[m]);
    }
  }
}

template <int R, int NP, int VAR>
__device__ __forceinline__ void p2_stage_pick(float4* s, const P2Tw& tw, int N, int L, int swap, int tid, int nthr) {
  const int MC = (L / R) * NP;
  if ((MC & 63) == 0) { p2_stage<R, NP, 1, VAR>(s, tw, N, L, swap, tid, nthr); return; }
  if constexpr (R == 8 || R == 16) {
    if (MC == 8) { p2_stage<R, NP, 2, VAR>(s, tw, N, L, swap, tid, nthr); return; }
  }
  if constexpr (R == 8 && NP == 1 && VAR != P2_DIF_DENSE) {
    if (MC == 1) { p2_stage<R, NP, 3, VAR>(s, tw, N, L, swap, tid, nthr); return; }
  }
  p2_stage<R, NP, 0, VAR>(s, tw, N, L, swap, tid, nthr);
}

template <int NP, int VAR>
__device__ __forceinline__ void p2_stage_dispatch(int r, float4* s, const P2Tw& tw, int N, int L, int swap, int tid,
                                                  int nthr) {
  if (r == 16) { p2_stage_pick<16, NP, VAR>(s, tw, N, L, swap, tid, nthr); return; }
  switch (r) {
    case 8: p2_stage_pick<8, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
    case 4: p2_stage_pick<4, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
    case 2: p2_stage_pick<2, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
    case 3: p2_stage_pick<3, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
    case 5: p2_stage_pick<5, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
    case 7: p2_stage_pick<7, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
    default: p2_stage_pick<11, NP, VAR>(s, tw, N, L, swap, tid, nthr); break;
  }
}

// dense first-stage input is in-place safe when the stride of the first stage is a multiple of 8 chunks
__host__ __device__ inline bool p2_dense_ok(const FftDesc& d, int np) { return (((d.n / d.radix[0]) * np) & 7) == 0; }

// barrier among the `nthr` transform threads of a CTA (named barrier 1: the CTA may hold other warps)
__device__ __forceinline__ void p2_sync(int nthr) { asm volatile("bar.sync 1, %0;" ::"r"(nthr) : "memory"); }

// Forward DIF transform of the NP * 2 interleaved length-N arrays.  The caller makes the input visible to the
// `nthr` transform threads first; on return every stage is complete and synchronised among them.
template <int NP>
__device__ __forceinline__ void p2_fft_dif(float4* s, const P2Tw& tw, const FftDesc& d, int inmode, int tid, int nthr) {
  int L = d.n;
  for (int st = 0; st < d.nstage; ++st) {
    if (st == 0 && inmode != P2_IN_PAIR)
      p2_stage_dispatch<NP, P2_DIF_DENSE>(d.radix[0], s, tw, d.n, L, inmode == P2_IN_AOS_SWAP, tid, nthr);
    else
      p2_stage_dispatch<NP, P2_DIF>(d.radix[st], s, tw, d.n, L, 0, tid, nthr);
    L /= d.radix[st];
    p2_sync(nthr);
  }
}

// Forward DIT transform: the input element n sits at (swizzled) position posmap[n] (digit-reversed), the output is
// in natural order.
template <int NP>
__device__ __forceinline__ void p2_fft_dit(float4* s, const P2Tw& tw, const FftDesc& d, int tid, int nthr) {
  int L = 1;
  for (int st = d.nstage - 1; st >= 0; --st) {
    L *= d.radix[st];
    p2_stage_dispatch<NP, P2_DIT>(d.radix[st], s, tw, d.n, L, 0, tid, nthr);
    p2_sync(nthr);
  }
}
