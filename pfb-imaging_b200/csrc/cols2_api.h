// Host interface of the TMA-fed column transforms (colsfft.cu), used by pfbgrid.cu.
#pragma once
#include <cuda_runtime.h>
#include "fused_common.cuh"

struct Cols2Args {
  FftDesc du;
  const float2* tw_u;
  const int* pos_u;          // k -> position of output k in the digit-reversed result
  int nu, nv, nx;
  int a_lo, a_len, b_lo, b_len;  // active window (multiples of 32), circular
  int q0, nq;                // logical planes [q0, q0 + nq)
  int slot0;                 // logical plane stored in slot 0 of the local stack (tensor-map row = (q - slot0) nu + a)
  int inverse;
};

// true when the pair-engine column kernels can serve this geometry (fp32 only): two nu x 16-byte buffers fit shared
// memory and the loaded row segments are made of 32-row boxes
bool cols2_supported(int nu, int nv, int nx, const FftDesc& du);
// one launch over planes [a.q0, a.q0 + a.nq): `stack` = the local plane stack (slot 0 = logical plane a.slot0,
// `stack_planes` planes: what the tensor maps describe and the loads read), `out` = where the result rows go,
// biased so that logical plane q sits at out + q nu nv (the local stack, or a peer-mapped one).
// Returns cudaSuccess or the failing error; *what names the failing step.
cudaError_t cols2_launch(const Cols2Args& a, const float2* stack, int stack_planes, float2* out, cudaStream_t s,
                         const char** what);

// Row passes on the pair engine (rows2.cuh, fp32): the same image row of two neighbouring planes per CTA.
// `stack_biased`: logical plane q at stack_biased + q nu nv.  Planes [ft.q0, ft.q0 + nq); nq must be even
// (cudaErrorInvalidValue otherwise).
bool rows2_supported(int nv);
cudaError_t rows2_fwd_launch(const GParams& g, const FusedTabs& ft, int nq, bool fast, const float* x, const float* beam,
                             const float* corr, float2* stack_biased, cudaStream_t s);
cudaError_t rows2_inv_launch(const GParams& g, const FusedTabs& ft, int nq, bool fast, const float2* stack_biased,
                             double* accimg, cudaStream_t s);
