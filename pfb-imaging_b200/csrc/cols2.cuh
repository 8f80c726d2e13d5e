// Column passes of the fused plane transforms on the pair engine (fft2.cuh), fed by the TMA unit.
//
// A work item is one block of FOUR neighbouring grid columns (two column pairs, one 32-byte sector per grid row) of
// one plane.  A CTA is persistent (one per SM); items are dealt round-robin.  Per item:
//   * one thread arms an mbarrier with the byte count and issues the cp.async.bulk.tensor loads of the rows that
//     hold data (boxes of 32 bytes x 256 / 32 rows, dense in shared memory), all threads zero the other rows;
//   * the first FFT stage reads the dense array-of-structures rows and writes the engine's swizzled pair layout;
//     the remaining stages run in place on packed two-wide butterflies (both column pairs at once, NP = 2);
//   * the rows that are needed are written back, one full 32-byte sector per row.
// Against the single-buffer kernels of fused_fft.cuh (k_cols_fwd / k_cols_inv): the global -> shared fill is done
// by the copy engine instead of a latency-bound LDG / STS loop (a third of those kernels' time), the butterflies
// issue half the instructions, twiddles and the digit-reversal table come from shared memory.
//
// (A double-buffered variant with 16-byte-wide boxes — one column pair per buffer, the next pair's load running
// under the butterflies — was built first and measured: every 16-byte row costs a 64-byte DRAM access and the L2
// does not keep the neighbours for the next item, 1.8 GB instead of 0.45 GB per band and pass; no faster than the
// old kernels.  Two full-sector buffers do not fit the 227 KB of shared memory at nu = 6144.)
//
//   forward (degrid direction): loads the nx image rows (two segments around the zero padding), writes the rows of
//                               the active uv window
//   inverse (grid direction)  : loads the active rows (circular window), writes the nx image rows; conj-in/conj-out
//                               of the old kernels becomes swap-in / swap-out, free in the pair layout
#pragma once
#include <cuda.h>
#include "fft2.cuh"
#include "cols2_api.h"

#define COLS2_THREADS 384      // radix-16 stages, 128 registers per thread
#define COLS2_BOX_BIG 256
#define COLS2_BOX_SMALL 32


__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one 2-D box: coordinates (c0 = float index along a grid row, c1 = row of the plane stack)
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}

// rows [r0, r1) of the four columns starting at column `col` of stack row block `rowbase` -> buffer rows [r0, r1)
__device__ __forceinline__ void cols2_load_rows(float4* buf, const CUtensorMap* mbig, const CUtensorMap* msmall, int col,
                                                int rowbase, int r0, int r1, uint64_t* bar) {
  int r = r0;
  for (; r + COLS2_BOX_BIG <= r1; r += COLS2_BOX_BIG) tma_load_2d(buf + 2 * r, mbig, 2 * col, rowbase + r, bar);
  for (; r < r1; r += COLS2_BOX_SMALL) tma_load_2d(buf + 2 * r, msmall, 2 * col, rowbase + r, bar);
}

__global__ void __launch_bounds__(COLS2_THREADS, 1)
k_cols2(const __grid_constant__ CUtensorMap mbig, const __grid_constant__ CUtensorMap msmall,
        const __grid_constant__ Cols2Args a, float2* __restrict__ out) {
  extern __shared__ __align__(1024) unsigned char smem_raw1k[];
  unsigned char* smem_raw = smem_raw1k;
  const int nu = a.nu, hx = a.nx / 2;
  float4* const s = reinterpret_cast<float4*>(smem_raw);  // nu rows x 2 chunks (column pairs) of 16 bytes
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + (size_t)nu * 32);
  float2* twtab = reinterpret_cast<float2*>(bar + 8);                                    // two-level twiddle table
  unsigned short* pos16 = reinterpret_cast<unsigned short*>(twtab + p2_tw_entries(nu));  // k -> position, nu entries
  constexpr int NTHR = COLS2_THREADS;
  const int tid = threadIdx.x;
  const P2Tw tw = p2_tw_fill(twtab, a.tw_u, nu, tid, NTHR);
  for (int k = tid; k < nu; k += NTHR) pos16[k] = (unsigned short)a.pos_u[k];
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_proxy_async();
  }
  __syncthreads();
  // work items: (plane, column block)
  const int nblk = a.b_len >> 2;
  const int64_t nitems = (int64_t)a.nq * nblk;
  // items are dealt round-robin: neighbouring column blocks (which share 64-byte DRAM atoms) are loaded by
  // neighbouring CTAs at about the same time, so one DRAM access serves both (contiguous ranges per CTA were
  // measured at 2.7x the DRAM reads: the L2 does not keep the neighbour for the next item)
  uint32_t phase = 0;
  // loaded row segments [s0a, s1a) and [s0b, s1b); everything else is zero
  int s0a, s1a, s0b, s1b;
  if (!a.inverse) {
    s0a = 0; s1a = hx; s0b = nu - hx; s1b = nu;
  } else {
    const int end = a.a_lo + a.a_len;
    if (end <= nu) { s0a = a.a_lo; s1a = end; s0b = 0; s1b = 0; }
    else { s0a = a.a_lo; s1a = nu; s0b = 0; s1b = end - nu; }
  }
  const uint32_t tx_bytes = (uint32_t)((s1a - s0a) + (s1b - s0b)) * 32u;
  const int inmode = a.inverse ? P2_IN_AOS_SWAP : P2_IN_AOS;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);

  for (int64_t it = blockIdx.x; it < nitems; it += gridDim.x) {
    const int q = (int)(it / nblk), j = (int)(it - (int64_t)q * nblk);
    int col = a.b_lo + 4 * j;
    if (col >= a.nv) col -= a.nv;
    // ---- fill: the copy engine brings the data rows, the threads zero the rest (disjoint rows)
    if (tid == 0) {
      const int rowbase = (a.q0 + q - a.slot0) * nu;
      mbar_expect_tx(bar, tx_bytes);
      cols2_load_rows(s, &mbig, &msmall, col, rowbase, s0a, s1a, bar);
      cols2_load_rows(s, &mbig, &msmall, col, rowbase, s0b, s1b, bar);
    }
    if (s1b > s0b) {  // two segments: the gap between them ([s1a, s0b) forward, [s1b, s0a) inverse)
      const int z0 = !a.inverse ? s1a : s1b, z1 = !a.inverse ? s0b : s0a;
      for (int e = 2 * z0 + tid; e < 2 * z1; e += NTHR) s[e] = z;
    } else {  // one segment [s0a, s1a): rows [0, s0a) and [s1a, nu)
      for (int e = tid; e < 2 * s0a; e += NTHR) s[e] = z;
      for (int e = 2 * s1a + tid; e < 2 * nu; e += NTHR) s[e] = z;
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    __syncthreads();  // everybody's zero rows are in place
    p2_fft_dif<2>(s, tw, a.du, inmode, tid, NTHR);
    // ---- write-back: one 32-byte sector per row
    float2* go = out + (int64_t)(a.q0 + q) * nu * a.nv + col;  // `out` is biased: logical plane q at out + q nu nv
    if (!a.inverse) {
#pragma unroll 4
      for (int t = tid; t < a.a_len; t += NTHR) {  // rows of the active window
        int k = a.a_lo + t;
        if (k >= nu) k -= nu;
        const int e = 2 * pos16[k];
        const float4 v0 = s[sw2(e)], v1 = s[sw2(e + 1)];  // {re0, re1, im0, im1} of column pairs 0 and 1
        float4* dst = reinterpret_cast<float4*>(go + (int64_t)k * a.nv);
        dst[0] = make_float4(v0.x, v0.z, v0.y, v0.w);
        dst[1] = make_float4(v1.x, v1.z, v1.y, v1.w);
      }
    } else {
#pragma unroll 4
      for (int t = tid; t < a.nx; t += NTHR) {  // the nx image rows; swap back: the transform ran on (im, re)
        const int k = t < hx ? t : t + (nu - a.nx);
        const int e = 2 * pos16[k];
        const float4 v0 = s[sw2(e)], v1 = s[sw2(e + 1)];  // {im0, im1, re0, re1}
        float4* dst = reinterpret_cast<float4*>(go + (int64_t)k * a.nv);
        dst[0] = make_float4(v0.z, v0.x, v0.w, v0.y);
        dst[1] = make_float4(v1.z, v1.x, v1.w, v1.y);
      }
    }
    fence_proxy_async();  // generic-proxy accesses of this item before the copy engine's writes of the next
    __syncthreads();
  }
}
