// Host plumbing shared by the translation units of libpfbgrid.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <vector>

#include "../../include/pfbgrid.h"

// pfbgrid.cu: the message of pfbg_last_error (returns code), pfbg_launch_count, 256-byte device scratch blocks
int pfbg_fail(int code, const char* fmt, ...);
inline constexpr auto& fail = pfbg_fail;
void pfbg_count_launch();
void* pfbg_scratch_get(int device);
void pfbg_scratch_put(int device, void* p);
// psfconv.cu: what the batched solvers of pfbsara.cu check before borrowing a convolver, whether p is a device array
// on `device`, and pfbg_conv_apply_scaled without its argument checks
int pfbg_conv_props(const pfbg_conv* cv, int* precision, int* device, int* nx, int* ny, int* has_kernel);
bool pfbg_on_device(const void* p, int device);
int pfbg_conv_apply_dev(pfbg_conv* cv, const void* x, const void* beam, const void* xin, double eta, double scale,
                        void* out, void* stream);
// weighting.cu: counts of nsnap snapshots (row_snap: snapshot of each row, NULL for one; scale[f] / lightspeed = f/c),
// then the Briggs / uniform re-weighting of wgt in place, on stream s.  counts: nsnap * nx * ny reals, sums: 3 * nsnap doubles
int pfbg_counts_reweight(int precision, cudaStream_t s, int64_t nrow, int nchan, int nx, int ny, double cell_x,
                         double cell_y, double usign, double vsign, double lightspeed, const double* uvw,
                         const double* scale, const uint8_t* mask, const int* row_snap, int64_t nsnap, double robust,
                         void* counts, double* sums, void* wgt);

#define CK(call)                                                                           \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess)                                                                 \
      return pfbg_fail(PFBG_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                       __FILE__, __LINE__);                                                \
  } while (0)
#define CKRC(call)              \
  do {                          \
    int rc_ = (call);           \
    if (rc_ != PFBG_OK) return rc_; \
  } while (0)
#define LAUNCHED() pfbg_count_launch()

// Device buffers of one call, freed on return; host arguments are copied in (copy) or only allocated for.
struct TmpBufs {
  std::vector<void*> ptrs;
  ~TmpBufs() { for (void* p : ptrs) cudaFree(p); }
  int get(void** out, const void* src, size_t bytes, bool dev, bool copy, cudaStream_t s) {
    if (dev) { *out = (void*)src; return PFBG_OK; }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes ? bytes : 16);
    if (e != cudaSuccess) return fail(PFBG_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    ptrs.push_back(p);
    if (copy && bytes) {
      e = cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, s);
      if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "H2D copy failed: %s", cudaGetErrorString(e));
    }
    *out = p;
    return PFBG_OK;
  }
};
