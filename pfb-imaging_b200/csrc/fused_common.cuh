// Tables and vector access helpers shared by the fused plane-transform kernels (fused_fft.cuh, rows2.cuh).
#pragma once
#include "common.cuh"
#include "fft.cuh"

struct FusedTabs {
  FftDesc du, dv;            // transforms along u (length nu) and v (length nv)
  const void* tw_u;          // cx2<T>[nu]
  const void* tw_v;
  const int* rev_u;          // pos -> k
  const int* rev_v;
  const int* pos_v;          // k -> pos (DIT input scatter)
  const int* pos_u;          // k -> pos along u (drain loops of the column kernels walk k)
  const double* nutab;       // (nx,ny) fp64: n - 1 + nshift per pixel (w-screen phase = w_p * nutab, up to 1e3 turns)
  // cells any bound sample can touch: rows [a_lo, a_lo+a_len) and columns [b_lo, b_lo+b_len), circular
  int a_lo, a_len, b_lo, b_len;
  // plane subset of a launch: CTA plane index + q0 is the logical plane (w_q = w0 + q dw).  Launches over a subset
  // (band split across GPUs: the owner transforms planes [0, P - nq), a helper GPU the last nq) pass plane-stack
  // pointers biased so that logical plane q sits at `grid + q * nu * nv` whatever slot it is stored in.
  int q0;
  // batched snapshots: w of every plane and the image it belongs to (null: w0 + q dw, image 0)
  const double* plane_w;
  const int* plane_img;
};

__device__ __forceinline__ bool in_window(int n, int lo, int len, int size) {
  int rel = n - lo;
  if (rel < 0) rel += size;
  return rel < len;
}

#define ROWS_MAX_THREADS 256
#define ROWS_BIG_THREADS_F32 768  /* one CTA per SM: 85 registers */
#define ROWS_BIG_THREADS_F64 512  /* 128 registers */
#define ROWS_BIG_SMEM (113 * 1024)  /* beyond this only one row CTA fits an SM */
#ifndef PFBG_ROWS_INV_INFLIGHT
#define PFBG_ROWS_INV_INFLIGHT 3
#endif

// ---- vector access helpers: the load / store loops of these kernels are latency-bound (ncu: 40-55 % of
// the stall samples were long-scoreboard waits in the fill / drain loops), so every global access moves
// 16 bytes and several independent accesses are in flight per thread -------------------------------
__device__ __forceinline__ void load4(const float* __restrict__ p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void load4(const double* __restrict__ p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void load4(const int* __restrict__ p, int (&v)[4]) {
  const int4 t = *reinterpret_cast<const int4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
// two consecutive complex values (16-byte aligned pair)
__device__ __forceinline__ void load_pair(const cx2<float>* __restrict__ p, cx2<float>& a, cx2<float>& b) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  a = {t.x, t.y}; b = {t.z, t.w};
}
__device__ __forceinline__ void load_pair(const cx2<double>* __restrict__ p, cx2<double>& a, cx2<double>& b) {
  const double2 t = *reinterpret_cast<const double2*>(p), u = *reinterpret_cast<const double2*>(p + 1);
  a = {t.x, t.y}; b = {u.x, u.y};
}
__device__ __forceinline__ void store_pair(cx2<float>* __restrict__ p, const cx2<float>& a, const cx2<float>& b) {
  *reinterpret_cast<float4*>(p) = make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void store_pair(cx2<double>* __restrict__ p, const cx2<double>& a, const cx2<double>& b) {
  *reinterpret_cast<double2*>(p) = make_double2(a.x, a.y);
  *reinterpret_cast<double2*>(p + 1) = make_double2(b.x, b.y);
}
// one row of a column block: C complex values = 32 bytes (8 / 16 bytes for the narrow blocks)
template <typename T, int C>
__device__ __forceinline__ void load_row(const cx2<T>* __restrict__ p, cx2<T> (&v)[C]) {
  if constexpr (C >= 2) {
#pragma unroll
    for (int c = 0; c < C; c += 2) load_pair(p + c, v[c], v[c + 1]);
  } else {
    v[0] = p[0];
  }
}
template <typename T, int C>
__device__ __forceinline__ void store_row(cx2<T>* __restrict__ p, const cx2<T> (&v)[C]) {
  if constexpr (C >= 2) {
#pragma unroll
    for (int c = 0; c < C; c += 2) store_pair(p + c, v[c], v[c + 1]);
  } else {
    p[0] = v[0];
  }
}

