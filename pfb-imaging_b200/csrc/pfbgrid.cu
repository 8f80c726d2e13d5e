// C-ABI implementation (include/pfbgrid.h): plan, binding/sort, cuFFT plumbing
// and launch sequencing of the sm_100a kernels in kernels.cuh / runs.cuh / fused_fft.cuh.
#include <cuda_runtime.h>
#include <cufft.h>
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <mutex>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pfbgrid.h"
#include "kernels.cuh"
#include "runs.cuh"
#include "runs_mma.cuh"
#include "fused_fft.cuh"
#include "cols2_api.h"
#include "fft_host.h"
#include "host.h"

// ---------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------
static thread_local std::string g_err;
static std::atomic<int64_t> g_launches{0};

int pfbg_fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
void pfbg_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// Small device scratch blocks (256 B) for the scalar reductions of every translation unit: a caller holds a block
// for the duration of its call, so two host threads (or two streams driven from different threads) on one device
// never share an accumulator; blocks are recycled, never freed while the process lives (no cudaMalloc / cudaFree
// inside solver loops).
static std::mutex g_scratch_mu;
static std::vector<void*> g_scratch_free[64];
void* pfbg_scratch_get(int device) {
  if (device < 0 || device >= 64) return nullptr;
  {
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    if (!g_scratch_free[device].empty()) {
      void* p = g_scratch_free[device].back();
      g_scratch_free[device].pop_back();
      return p;
    }
  }
  void* p = nullptr;
  if (cudaMalloc(&p, 256) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void pfbg_scratch_put(int device, void* p) {
  if (!p || device < 0 || device >= 64) return;
  std::lock_guard<std::mutex> lk(g_scratch_mu);
  g_scratch_free[device].push_back(p);
}

#define CKFFT(call)                                                                        \
  do {                                                                                     \
    cufftResult r_ = (call);                                                               \
    if (r_ != CUFFT_SUCCESS)                                                               \
      return fail(PFBG_ERR_CUFFT, "%s failed: cufft status %d (%s:%d)", #call, (int)r_,    \
                  __FILE__, __LINE__);                                                     \
  } while (0)

extern "C" const char* pfbg_last_error(void) { return g_err.c_str(); }
extern "C" int pfbg_version(void) { return 100; }
extern "C" int64_t pfbg_launch_count(void) { return g_launches.load(); }
extern "C" int pfbg_device_count(int32_t* count) {
  int n = 0;
  CK(cudaGetDeviceCount(&n));
  *count = n;
  return PFBG_OK;
}

// ---------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

struct pfbg_plan {
  int precision = 0, device = 0;
  GParams gp{};
  int n_gl = 0;
  // device state
  DevBuf corr;                 // (nx,ny) T
  DevBuf grid;                 // (nplanes,nu,nv) C
  bool grid_external = false;  // the stack is lent by the caller (pfbg_plan_set_stack): never allocated / freed here
  bool grid_lazy = false;      // PFBG_PLAN_EXTERNAL_STACK: no stack until one is lent
  DevBuf uvw, fscale, mask;    // bound geometry
  DevBuf wgt;                  // bound weights (nrow,nchan) T
  DevBuf wcounts;              // pfbg_bind_weights_robust: (nbatch,nx_pad,ny_pad) T counts + 3 sums per snapshot
  DevBuf sorted_idx;           // (nactive) u32
  DevBuf recs;                 // (nactive) VisRec<T>, bucket order (run kernels, W <= 8)
  bool use_runs = false;
  DevBuf mvis;                 // (nactive) C, Hessian model vis in bucket order
  DevBuf img_in, img_out, img_beam;  // staging for host-pointer calls
  DevBuf vis_stage, wgt_stage;
  DevBuf flag;
  DevBuf srt_ka, srt_kb, srt_va, srt_vb, srt_tmp;  // sort scratch, kept between bindings when small (snapshot imaging)
  // pinned host staging for host-pointer calls (pageable user arrays are copied through these by
  // several threads, chunk by chunk, overlapped with the DMA)
  void* h_in = nullptr;
  size_t h_in_bytes = 0;
  void* h_out = nullptr;
  size_t h_out_bytes = 0;
  cudaEvent_t stage_ev[16]{};
  bool stage_ev_ok = false;
  // fused FFT path (fused_fft.cuh)
  DevBuf tw_u, tw_v, rev_u, rev_v, pos_v, pos_u, cellflags, accimg, nutab;
  FusedTabs ftabs{};
  bool fused = false;          // tables built and sizes fit shared memory
  int col_c = 4;               // columns per CTA in the column passes
  bool cols2 = false;          // fp32: TMA-fed pair-engine column kernels (cols2.cuh) serve this geometry
  bool rows2 = false;          // fp32: pair-engine row kernels (rows2.cuh), two planes per CTA
  cufftHandle fft = 0;
  int fft_batch = 1;           // planes per cuFFT execution (a divisor of nplanes; bounds the work area)
  bool fft_ok = false;
  size_t fft_work = 0;
  int64_t nrow = 0, nvis = 0, nactive = 0;
  bool bound = false, has_mask = false, has_wgt = false;
  bool beam_on_device = false;  // img_beam holds the beam of the last host-pointer Hessian call
  size_t total_bytes = 0;
  // batched snapshots (pfbg_plan_set_batch): nbatch images of one geometry share the plane stack
  int nbatch = 1;
  DevBuf row_snap, snap_w0, snap_pbase, snap_np, plane_w, plane_img;
  // band split across two GPUs (pfbg_split_*): the plane transforms of the last split_nq planes run on a helper
  int split_role = 0;             // 0 none, 1 owner, 2 helper
  int split_nq = 0;
  int stack_planes = 0;           // planes the local stack holds (helper: split_nq)
  DevBuf xshare, partial, mailbox, x_local;  // owner: xshare / partial / mailbox are exported; helper: mailbox, x_local
  void* peer_grid = nullptr;      // helper: the owner's plane stack (peer-mapped)
  void* peer_xshare = nullptr;    // helper: the owner's x [* beam]
  void* peer_partial = nullptr;   // helper: the owner's fp64 partial image
  unsigned long long* peer_mailbox = nullptr;  // the other side's flags
  unsigned long long split_step = 0;
  // profiling
  bool profiling = false;
  cudaEvent_t ev[8]{};
  bool ev_ok = false;
  int n_ev = 0;
};

static int dev_alloc(pfbg_plan* pl, DevBuf& b, size_t bytes);
// (re)size the plane stack: a lent stack is never reallocated, it must be large enough
static int stack_alloc(pfbg_plan* pl, size_t bytes) {
  if (pl->grid_external) {
    if (pl->grid.bytes < bytes) return fail(PFBG_ERR_NOMEM, "the lent plane stack holds %zu bytes, %zu are needed", pl->grid.bytes, bytes);
    return PFBG_OK;
  }
  if (pl->grid_lazy) return PFBG_OK;  // sized when a stack is lent
  return dev_alloc(pl, pl->grid, bytes);
}
static int dev_alloc(pfbg_plan* pl, DevBuf& b, size_t bytes) {
  if (b.bytes >= bytes && b.p) return PFBG_OK;
  if (b.p) {
    cudaFree(b.p);
    pl->total_bytes -= b.bytes;
    b.p = nullptr;
    b.bytes = 0;
  }
  if (bytes == 0) return PFBG_OK;
  cudaError_t e = cudaMalloc(&b.p, bytes);
  if (e != cudaSuccess) {
    b.p = nullptr;
    cudaGetLastError();
    return fail(PFBG_ERR_NOMEM, "cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
  }
  b.bytes = bytes;
  pl->total_bytes += bytes;
  return PFBG_OK;
}
static void dev_free(pfbg_plan* pl, DevBuf& b) {
  if (b.p) {
    cudaFree(b.p);
    pl->total_bytes -= b.bytes;
  }
  b.p = nullptr;
  b.bytes = 0;
}

static inline size_t real_bytes(const pfbg_plan* pl) { return pl->precision == PFBG_F32 ? 4 : 8; }
// pixels of the image argument of grid / degrid / hessian: nbatch images for a batched plan
static inline size_t img_elems(const pfbg_plan* pl) { return (size_t)pl->nbatch * pl->gp.nx * pl->gp.ny; }

extern "C" int pfbg_plan_destroy(pfbg_plan* pl) {
  if (!pl) return PFBG_OK;
  cudaSetDevice(pl->device);
  if (pl->fft_ok) cufftDestroy(pl->fft);
  if (pl->grid_external) { pl->grid.p = nullptr; pl->grid.bytes = 0; }
  DevBuf* all[] = {&pl->corr, &pl->grid, &pl->uvw, &pl->fscale, &pl->mask, &pl->wgt, &pl->wcounts, &pl->sorted_idx, &pl->srt_ka, &pl->srt_kb, &pl->srt_va, &pl->srt_vb, &pl->srt_tmp,
                   &pl->xshare, &pl->partial, &pl->mailbox, &pl->x_local,
                   &pl->row_snap, &pl->snap_w0, &pl->snap_pbase, &pl->snap_np, &pl->plane_w, &pl->plane_img,
                   &pl->recs, &pl->mvis, &pl->tw_u, &pl->tw_v, &pl->rev_u, &pl->rev_v, &pl->pos_v, &pl->pos_u, &pl->cellflags, &pl->accimg, &pl->nutab, &pl->img_in, &pl->img_out, &pl->img_beam, &pl->vis_stage, &pl->wgt_stage,
                   &pl->flag};
  for (DevBuf* b : all) dev_free(pl, *b);
  if (pl->ev_ok)
    for (auto& e : pl->ev) cudaEventDestroy(e);
  if (pl->stage_ev_ok)
    for (auto& e : pl->stage_ev) cudaEventDestroy(e);
  if (pl->h_in) cudaFreeHost(pl->h_in);
  if (pl->h_out) cudaFreeHost(pl->h_out);
  delete pl;
  return PFBG_OK;
}

// Lend the plan a plane stack owned by the caller (device memory of the plan's device).  The stack is scratch
// between calls — every grid / degrid / Hessian call rebuilds it — so the plans of the bands of one GPU can take
// turns on ONE stack per compute stream instead of holding nplanes * nu * nv cells each (C4: 62 GB per band).
// dev_ptr == NULL takes the loan back (a plan created without PFBG_PLAN_EXTERNAL_STACK allocates its own again).
extern "C" int pfbg_plan_set_stack(pfbg_plan* pl, void* dev_ptr, uint64_t bytes) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  if (pl->split_role != 0) return fail(PFBG_ERR_STATE, "the stack of a split band is exported to its helper and cannot be replaced");
  CK(cudaSetDevice(pl->device));
  const size_t need = (size_t)pl->stack_planes * pl->gp.nu * pl->gp.nv * 2 * real_bytes(pl);
  if (!dev_ptr) {
    if (pl->grid_external) { pl->grid.p = nullptr; pl->grid.bytes = 0; pl->grid_external = false; }
    if (!pl->grid_lazy) CKRC(dev_alloc(pl, pl->grid, need));
    return PFBG_OK;
  }
  if (bytes < need) return fail(PFBG_ERR_ARG, "the lent stack holds %llu bytes, the plan needs %zu", (unsigned long long)bytes, need);
  if (((uintptr_t)dev_ptr & 255) != 0) return fail(PFBG_ERR_ARG, "the lent stack must be 256-byte aligned");
  cudaPointerAttributes at;
  CK(cudaPointerGetAttributes(&at, dev_ptr));
  if (at.type != cudaMemoryTypeDevice || at.device != pl->device) return fail(PFBG_ERR_ARG, "the lent stack is not device memory of device %d", pl->device);
  if (!pl->grid_external) dev_free(pl, pl->grid);
  pl->grid.p = dev_ptr;
  pl->grid.bytes = (size_t)bytes;
  pl->grid_external = true;
  return PFBG_OK;
}

template <typename T> static int fused_setup_t(pfbg_plan* pl);
static int cufft_setup(pfbg_plan* pl);

static int plan_create_impl(const pfbg_plan_desc* d, int stack_planes, pfbg_plan** out);
extern "C" int pfbg_plan_create(const pfbg_plan_desc* d, pfbg_plan** out) {
  return plan_create_impl(d, d ? d->nplanes : 0, out);
}

// stack_planes < nplanes: a transform helper of a split band, which only stores the planes it transforms
static int plan_create_impl(const pfbg_plan_desc* d, int stack_planes, pfbg_plan** out) {
  if (!d || !out) return fail(PFBG_ERR_ARG, "null argument");
  *out = nullptr;
  if (d->precision != PFBG_F32 && d->precision != PFBG_F64) return fail(PFBG_ERR_ARG, "bad precision");
  if (d->nx <= 0 || d->ny <= 0 || (d->nx & 1) || (d->ny & 1)) return fail(PFBG_ERR_ARG, "nx, ny must be positive and even");
  if (d->W < 4 || d->W > PFBG_MAXW) return fail(PFBG_ERR_ARG, "kernel support W=%d outside [4,%d]", d->W, PFBG_MAXW);
  if (d->nu % (2 * PFBG_TILE) || d->nv % (2 * PFBG_TILE)) return fail(PFBG_ERR_ARG, "nu, nv must be multiples of %d", 2 * PFBG_TILE);
  if (d->nu < d->nx + d->W || d->nv < d->ny + d->W) return fail(PFBG_ERR_ARG, "grid smaller than image + support");
  if (d->nplanes < 1 || (d->do_wgridding && d->nplanes < d->W)) return fail(PFBG_ERR_ARG, "nplanes=%d too small for W=%d", d->nplanes, d->W);
  if (!d->do_wgridding && d->nplanes != 1) return fail(PFBG_ERR_ARG, "nplanes must be 1 without w-gridding");
  if (d->pmirror < 0 || d->pmirror > 32 || (d->pmirror > 0 && (d->nplanes < d->pmirror || d->w0 != 0.5 * d->dw)))
    return fail(PFBG_ERR_ARG, "mirror planes need 0 <= pmirror <= min(32, nplanes) and w0 == dw/2");
  if (!d->corr_u || !d->corr_v) return fail(PFBG_ERR_ARG, "missing correction vectors");
  if (d->do_wgridding && (!d->gl_x || !d->gl_w || d->n_gl <= 0 || !(d->dw > 0))) return fail(PFBG_ERR_ARG, "missing quadrature / dw for w-gridding");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (d->device < 0 || d->device >= ndev) return fail(PFBG_ERR_ARG, "device %d out of range (%d visible)", d->device, ndev);
  CK(cudaSetDevice(d->device));
  {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, d->device));
    if (prop.major != 10) return fail(PFBG_ERR_STATE, "device %d is sm_%d%d; this library is built for sm_100a only", d->device, prop.major, prop.minor);
  }

  pfbg_plan* pl = new pfbg_plan();
  pl->precision = d->precision;
  pl->device = d->device;
  GParams& g = pl->gp;
  g.nx = d->nx; g.ny = d->ny; g.nu = d->nu; g.nv = d->nv; g.W = d->W; g.nplanes = d->nplanes;
  g.nchan = 0;
  g.nbatch = 1;
  g.row_snap = nullptr; g.snap_w0 = nullptr; g.snap_pbase = nullptr; g.snap_np = nullptr;
  g.do_wgridding = d->do_wgridding; g.divide_by_n = d->divide_by_n;
  g.beta = d->beta; g.pixsize_x = d->pixsize_x; g.pixsize_y = d->pixsize_y;
  g.center_x = d->center_x; g.center_y = d->center_y;
  g.usign = d->usign; g.vsign = d->vsign; g.wsign = d->wsign;
  g.w0 = d->w0; g.dw = d->dw; g.nshift = d->nshift;
  g.pmirror = d->do_wgridding ? d->pmirror : 0;
  g.fast_screen = (d->precision == PFBG_F32 && d->fast_screen) ? 1 : 0;
  g.ntile_u = d->nu / PFBG_TILE; g.ntile_v = d->nv / PFBG_TILE;
  pl->n_gl = d->n_gl;

  auto bail = [&](int rc) { pfbg_plan_destroy(pl); return rc; };
  const size_t rb = real_bytes(pl);
  int rc;
  if ((rc = dev_alloc(pl, pl->corr, (size_t)g.nx * g.ny * rb))) return bail(rc);
  pl->stack_planes = stack_planes;
  pl->grid_lazy = (d->flags & PFBG_PLAN_EXTERNAL_STACK) != 0;
  if (!pl->grid_lazy && (rc = dev_alloc(pl, pl->grid, (size_t)stack_planes * g.nu * g.nv * 2 * rb))) return bail(rc);
  if ((rc = dev_alloc(pl, pl->flag, 128))) return bail(rc);

  // correction image
  {
    DevBuf cu, cv, gx, gw;
    std::vector<double> glw;
    auto cleanup = [&]() { dev_free(pl, cu); dev_free(pl, cv); dev_free(pl, gx); dev_free(pl, gw); };
    if ((rc = dev_alloc(pl, cu, g.nx * sizeof(double))) || (rc = dev_alloc(pl, cv, g.ny * sizeof(double)))) { cleanup(); return bail(rc); }
    cudaMemcpy(cu.p, d->corr_u, g.nx * sizeof(double), cudaMemcpyHostToDevice);
    cudaMemcpy(cv.p, d->corr_v, g.ny * sizeof(double), cudaMemcpyHostToDevice);
    int ngl = 0;
    if (g.do_wgridding) {
      ngl = d->n_gl;
      glw.resize(ngl);
      // psihat(xi) = (W/2) int_{-1}^{1} phi cos = W * sum_k w_k phi(x_k) cos(pi W xi x_k) over the half interval
      for (int k = 0; k < ngl; ++k) {
        double x = d->gl_x[k];
        glw[k] = (double)g.W * d->gl_w[k] * exp(g.beta * (sqrt((1.0 - x) * (1.0 + x)) - 1.0));
      }
      if ((rc = dev_alloc(pl, gx, ngl * sizeof(double))) || (rc = dev_alloc(pl, gw, ngl * sizeof(double)))) { cleanup(); return bail(rc); }
      cudaMemcpy(gx.p, d->gl_x, ngl * sizeof(double), cudaMemcpyHostToDevice);
      cudaMemcpy(gw.p, glw.data(), ngl * sizeof(double), cudaMemcpyHostToDevice);
    }
    dim3 blk(128), grd((g.ny + 127) / 128, g.nx);
    if (pl->precision == PFBG_F32)
      k_corr_init<float><<<grd, blk>>>(g, (const double*)cu.p, (const double*)cv.p, (const double*)gx.p, (const double*)gw.p, ngl, (float*)pl->corr.p);
    else
      k_corr_init<double><<<grd, blk>>>(g, (const double*)cu.p, (const double*)cv.p, (const double*)gx.p, (const double*)gw.p, ngl, (double*)pl->corr.p);
    LAUNCHED();
    cudaError_t e = cudaDeviceSynchronize();
    cleanup();
    if (e != cudaSuccess) { fail(PFBG_ERR_CUDA, "correction kernel failed: %s", cudaGetErrorString(e)); return bail(PFBG_ERR_CUDA); }
  }

  // plane transforms: fused in-shared-memory FFT when the sizes fit, cuFFT otherwise
  {
    int rc2 = pl->precision == PFBG_F32 ? fused_setup_t<float>(pl) : fused_setup_t<double>(pl);
    if (rc2) return bail(rc2);
    if (!pl->fused && (rc2 = cufft_setup(pl))) return bail(rc2);
  }
  *out = pl;
  return PFBG_OK;
}

// ---------------------------------------------------------------------------
// fused FFT tables
// ---------------------------------------------------------------------------
template <typename T>
static int upload_twiddles(pfbg_plan* pl, DevBuf& buf, int n) {
  const std::vector<cx2<T>> tw = twiddles<T>(n);
  CKRC(dev_alloc(pl, buf, (size_t)n * sizeof(cx2<T>)));
  CK(cudaMemcpy(buf.p, tw.data(), (size_t)n * sizeof(cx2<T>), cudaMemcpyHostToDevice));
  return PFBG_OK;
}

template <typename T>
static int fused_setup_t(pfbg_plan* pl) {
  using C = typename cplx_of<T>::type;
  const GParams& g = pl->gp;
  pl->fused = false;
  const char* env = getenv("PFBG_FFT");
  if (env && strcmp(env, "cufft") == 0) return PFBG_OK;
  // columns per CTA in the column passes: a full 32-byte sector per row if that fits shared memory,
  // otherwise narrower blocks (half / quarter sectors; L2 merges the neighbours) for large grids
  pl->col_c = (int)(32 / sizeof(C));
  const int full_c = pl->col_c;
  if (const char* cc = getenv("PFBG_COLC")) {  // tuning hook: narrower blocks -> more resident CTAs per SM
    const int v = atoi(cc);
    if (v == 1 || v == 2 || v == 4) pl->col_c = v < full_c ? v : full_c;
  }
  while (pl->col_c > 1 && fft_smem_bytes<T>(g.nu * pl->col_c) > kMaxSmem) pl->col_c /= 2;
  // Narrower column blocks stay fused, measured on B200: half-sector blocks win at 8640^2 (the PSF grid of a 4096^2
  // field, 12 planes: 20.6 ms per Hessian apply against cuFFT's 25.9 ms in fp32, 34.6 vs 48.1 ms in fp64, and no work
  // area) and quarter-sector blocks (fp32 grids up to ~27k) are on par (15360^2 x 33 planes: 312 ms vs 339 ms).
  // cuFFT takes what the shared-memory engine cannot: rows or one-column blocks beyond shared memory, other primes.
  if (fft_smem_bytes<T>(g.nv) > kMaxSmem) return PFBG_OK;
  if (fft_smem_bytes<T>(g.nu * pl->col_c) > kMaxSmem) return PFBG_OK;
  FftDesc du, dv;
  const int maxr = sizeof(T) == 4 ? 16 : 8;
  if (!factorize(g.nu, du, maxr) || !factorize(g.nv, dv, maxr)) return PFBG_OK;
  std::vector<int> rev, pos;
  CKRC(upload_twiddles<T>(pl, pl->tw_u, g.nu));
  CKRC(upload_twiddles<T>(pl, pl->tw_v, g.nv));
  digit_tables(du, rev, pos);
  CKRC(dev_alloc(pl, pl->rev_u, (size_t)g.nu * 4));
  CK(cudaMemcpy(pl->rev_u.p, rev.data(), (size_t)g.nu * 4, cudaMemcpyHostToDevice));
  CKRC(dev_alloc(pl, pl->pos_u, (size_t)g.nu * 4));
  CK(cudaMemcpy(pl->pos_u.p, pos.data(), (size_t)g.nu * 4, cudaMemcpyHostToDevice));
  digit_tables(dv, rev, pos);
  CKRC(dev_alloc(pl, pl->rev_v, (size_t)g.nv * 4));
  CKRC(dev_alloc(pl, pl->pos_v, (size_t)g.nv * 4));
  CK(cudaMemcpy(pl->rev_v.p, rev.data(), (size_t)g.nv * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->pos_v.p, pos.data(), (size_t)g.nv * 4, cudaMemcpyHostToDevice));
  FusedTabs& ft = pl->ftabs;
  ft.du = du; ft.dv = dv;
  ft.tw_u = pl->tw_u.p; ft.tw_v = pl->tw_v.p;
  ft.rev_u = (const int*)pl->rev_u.p; ft.rev_v = (const int*)pl->rev_v.p; ft.pos_v = (const int*)pl->pos_v.p; ft.pos_u = (const int*)pl->pos_u.p;
  ft.a_lo = 0; ft.a_len = g.nu; ft.b_lo = 0; ft.b_len = g.nv;
  ft.q0 = 0;
  // opt in to large dynamic shared memory
  CK(cudaFuncSetAttribute(k_rows_fwd<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_rows_inv<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_rows_inv<T>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  CK(cudaFuncSetAttribute(k_rows_fwd<T>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  CK(cudaFuncSetAttribute(k_rows_fwd<T, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_rows_inv<T, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  if constexpr (sizeof(T) == 4) {
    CK(cudaFuncSetAttribute(k_rows_fwd<T, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CK(cudaFuncSetAttribute(k_rows_inv<T, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CK(cudaFuncSetAttribute(k_rows_fwd<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CK(cudaFuncSetAttribute(k_rows_inv<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CK(cudaFuncSetAttribute(k_rows_inv<T, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CK(cudaFuncSetAttribute(k_rows_fwd<T, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  }
  CKRC(dev_alloc(pl, pl->accimg, (size_t)g.nx * g.ny * sizeof(double)));
  CKRC(dev_alloc(pl, pl->nutab, (size_t)g.nx * g.ny * sizeof(double)));
  k_nu_table<<<dim3((g.ny + 127) / 128, g.nx), 128>>>(g, (double*)pl->nutab.p);
  LAUNCHED();
  CK(cudaDeviceSynchronize());
  ft.nutab = (const double*)pl->nutab.p;
  CK(cudaFuncSetAttribute(k_cols_fwd<T, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_cols_inv<T, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_cols_fwd<T, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_cols_inv<T, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_cols_fwd<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  CK(cudaFuncSetAttribute(k_cols_inv<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  pl->cols2 = false;
  if constexpr (sizeof(T) == 4) {
    const char* ce = getenv("PFBG_COLS");  // PFBG_COLS=old: the single-buffer column kernels of fused_fft.cuh
    pl->cols2 = !(ce && strcmp(ce, "old") == 0) && pl->col_c == full_c && cols2_supported(g.nu, g.nv, g.nx, du);
    const char* re = getenv("PFBG_ROWS");  // PFBG_ROWS=old: one plane per CTA (k_rows_fwd / k_rows_inv)
    pl->rows2 = !(re && strcmp(re, "old") == 0) && rows2_supported(g.nv);
  }
  pl->fused = true;
  return PFBG_OK;
}

static int cufft_setup(pfbg_plan* pl) {
  if (pl->fft_ok) return PFBG_OK;
  const GParams& g = pl->gp;
  CKFFT(cufftCreate(&pl->fft));
  pl->fft_ok = true;
  long long n[2] = {g.nu, g.nv};
  size_t ws = 0;
  // cuFFT's work area is about one batch of planes: keep a batch below ~8 GB so that very large
  // stacks (e.g. 15360^2 x 64 planes = 121 GB) still fit the 180 GB of HBM
  const size_t plane_bytes = (size_t)g.nu * g.nv * 2 * real_bytes(pl);
  int batch = g.nplanes;
  while (batch > 1 && ((size_t)batch * plane_bytes > ((size_t)8 << 30) || g.nplanes % batch)) --batch;
  pl->fft_batch = batch;
  cufftResult r = cufftMakePlanMany64(pl->fft, 2, n, nullptr, 1, 0, nullptr, 1, 0,
                                      pl->precision == PFBG_F32 ? CUFFT_C2C : CUFFT_Z2Z, batch, &ws);
  if (r != CUFFT_SUCCESS)
    return fail(PFBG_ERR_CUFFT, "cufftMakePlanMany64(%d x %d, batch %d) failed (%d)", g.nu, g.nv, batch, (int)r);
  pl->fft_work = ws;
  pl->total_bytes += ws;
  return PFBG_OK;
}

// circular window covering every flagged 32-cell group: complement of the longest run of clear groups
static void window_from_flags(const std::vector<int>& f, int size, int& lo, int& len) {
  const int ng = (int)f.size();
  int best_len = 0, best_start = 0, any = 0;
  for (int v : f) any |= v;
  if (!any) { lo = 0; len = 32 <= size ? 32 : size; return; }
  // scan twice around the circle for the longest clear run
  int run = 0;
  for (int i = 0; i < 2 * ng; ++i) {
    if (!f[i % ng]) {
      ++run;
      if (run > best_len && run <= ng) { best_len = run; best_start = i - run + 1; }
    } else run = 0;
  }
  if (best_len >= ng) { lo = 0; len = size; return; }
  int first = (best_start + best_len) % ng;  // first flagged group after the gap
  lo = first * 32;
  len = (ng - best_len) * 32;
  if (len > size) len = size;
}

// Re-target a plan to another w-range (same image geometry, sigma, W: corr / dw / nshift unchanged).
// Lets one plan object serve many snapshots (pfb hci): no reallocation unless the stack must grow.
extern "C" int pfbg_plan_set_wrange(pfbg_plan* pl, double w0, int32_t nplanes, int32_t pmirror) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  GParams& g = pl->gp;
  if (!g.do_wgridding) {
    if (nplanes != 1) return fail(PFBG_ERR_ARG, "nplanes must be 1 without w-gridding");
    return PFBG_OK;
  }
  if (nplanes < g.W) return fail(PFBG_ERR_ARG, "nplanes=%d too small for W=%d", nplanes, g.W);
  if (pmirror < 0 || pmirror > 32 || (pmirror > 0 && (nplanes < pmirror || w0 != 0.5 * g.dw)))
    return fail(PFBG_ERR_ARG, "mirror planes need 0 <= pmirror <= min(32, nplanes) and w0 == dw/2");
  CK(cudaSetDevice(pl->device));
  if (pl->split_role) return fail(PFBG_ERR_STATE, "plan is part of a band split");
  if (pl->nbatch > 1) return fail(PFBG_ERR_STATE, "plan is batched (pfbg_plan_set_batch)");
  const size_t need = (size_t)nplanes * g.nu * g.nv * 2 * real_bytes(pl);
  pl->stack_planes = nplanes;
  if (need > pl->grid.bytes) {
    CK(cudaDeviceSynchronize());
    CKRC(stack_alloc(pl, need));
  }
  if (nplanes != g.nplanes && pl->fft_ok) {  // the cuFFT batch depends on the plane count: rebuild lazily
    cufftDestroy(pl->fft);
    pl->fft_ok = false;
    pl->total_bytes -= pl->fft_work;
    pl->fft_work = 0;
  }
  g.w0 = w0;
  g.nplanes = nplanes;
  g.pmirror = pmirror;
  pl->bound = false;
  return PFBG_OK;
}


// ---------------------------------------------------------------------------
// Batched snapshots: nbatch small images of ONE geometry in one launch sequence (pfb hci makes thousands of
// 512^2 vis2dirty calls, utils/stokes2im.py:635-683; a launch sequence per snapshot is launch-latency bound).
// The snapshots share sigma, W, dw, nshift, the correction image and the transform tables; each owns a block of
// planes of one stack and an image slot.  Afterwards pfbg_bind_vis_batch / pfbg_grid / pfbg_degrid / pfbg_hessian take
// and return nbatch images (nbatch, nx, ny) and the rows of all snapshots concatenated.
// ---------------------------------------------------------------------------
extern "C" int pfbg_plan_set_batch(pfbg_plan* pl, int32_t nbatch, const double* snap_w0, const int32_t* snap_np) {
  if (!pl || !snap_w0 || !snap_np) return fail(PFBG_ERR_ARG, "null argument");
  if (nbatch < 1) return fail(PFBG_ERR_ARG, "nbatch must be positive");
  if (!pl->fused) return fail(PFBG_ERR_STATE, "batched plans need the fused plane transforms (grid too large for shared memory?)");
  if (pl->split_role) return fail(PFBG_ERR_STATE, "plan is part of a band split");
  GParams& g = pl->gp;
  if (g.pmirror) return fail(PFBG_ERR_ARG, "batched plans do not use mirror planes (make the plan with pmirror = 0)");
  CK(cudaSetDevice(pl->device));
  CK(cudaDeviceSynchronize());
  std::vector<int> pbase(nbatch), pimg;
  std::vector<double> pw;
  int64_t total = 0;
  for (int s = 0; s < nbatch; ++s) {
    const int np_ = snap_np[s];
    if (np_ < (g.do_wgridding ? g.W : 1) || (!g.do_wgridding && np_ != 1))
      return fail(PFBG_ERR_ARG, "snapshot %d: %d planes for W=%d", s, np_, g.W);
    pbase[s] = (int)total;
    for (int q = 0; q < np_; ++q) { pw.push_back(snap_w0[s] + q * g.dw); pimg.push_back(s); }
    total += np_;
  }
  if (total > (1 << 20)) return fail(PFBG_ERR_ARG, "too many planes in one batch");
  const size_t rb = real_bytes(pl);
  CKRC(stack_alloc(pl, (size_t)total * g.nu * g.nv * 2 * rb));
  CKRC(dev_alloc(pl, pl->snap_w0, (size_t)nbatch * 8));
  CKRC(dev_alloc(pl, pl->snap_pbase, (size_t)nbatch * 4));
  CKRC(dev_alloc(pl, pl->snap_np, (size_t)nbatch * 4));
  CKRC(dev_alloc(pl, pl->plane_w, (size_t)total * 8));
  CKRC(dev_alloc(pl, pl->plane_img, (size_t)total * 4));
  CKRC(dev_alloc(pl, pl->accimg, (size_t)nbatch * g.nx * g.ny * sizeof(double)));
  CK(cudaMemcpy(pl->snap_w0.p, snap_w0, (size_t)nbatch * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->snap_pbase.p, pbase.data(), (size_t)nbatch * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->snap_np.p, snap_np, (size_t)nbatch * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->plane_w.p, pw.data(), (size_t)total * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(pl->plane_img.p, pimg.data(), (size_t)total * 4, cudaMemcpyHostToDevice));
  pl->nbatch = nbatch;
  pl->stack_planes = (int)total;
  g.nplanes = (int)total;
  g.nbatch = nbatch;
  g.snap_w0 = (const double*)pl->snap_w0.p;
  g.snap_pbase = (const int*)pl->snap_pbase.p;
  g.snap_np = (const int*)pl->snap_np.p;
  g.row_snap = nullptr;  // set by pfbg_bind_vis_batch
  pl->ftabs.plane_w = (const double*)pl->plane_w.p;
  pl->ftabs.plane_img = (const int*)pl->plane_img.p;
  pl->bound = false;
  return PFBG_OK;
}

// rows [row_offsets[s], row_offsets[s+1]) of uvw / mask (and later vis / wgt) belong to snapshot s
extern "C" int pfbg_bind_vis_batch(pfbg_plan* pl, const double* uvw, const double* fscale, const uint8_t* mask,
                                   int64_t nrow, int32_t nchan, const int64_t* row_offsets, uint32_t flags, void* stream) {
  if (!pl || !row_offsets) return fail(PFBG_ERR_ARG, "null argument");
  if (pl->nbatch < 1 || !pl->gp.snap_w0) return fail(PFBG_ERR_STATE, "pfbg_plan_set_batch first");
  if (flags & PFBG_DEVICE_PTRS) return fail(PFBG_ERR_ARG, "pfbg_bind_vis_batch takes host pointers");
  if (row_offsets[0] != 0 || row_offsets[pl->nbatch] != nrow) return fail(PFBG_ERR_ARG, "row_offsets must run from 0 to nrow");
  CK(cudaSetDevice(pl->device));
  std::vector<int> rs((size_t)(nrow > 0 ? nrow : 1));
  for (int s = 0; s < pl->nbatch; ++s) {
    if (row_offsets[s + 1] < row_offsets[s]) return fail(PFBG_ERR_ARG, "row_offsets must not decrease");
    for (int64_t r = row_offsets[s]; r < row_offsets[s + 1]; ++r) rs[(size_t)r] = s;
  }
  CKRC(dev_alloc(pl, pl->row_snap, rs.size() * 4));
  CK(cudaMemcpy(pl->row_snap.p, rs.data(), rs.size() * 4, cudaMemcpyHostToDevice));
  pl->gp.row_snap = (const int*)pl->row_snap.p;
  return pfbg_bind_vis(pl, uvw, fscale, mask, nrow, nchan, flags, stream);
}

extern "C" int pfbg_plan_get_info(const pfbg_plan* pl, pfbg_plan_info* info) {
  if (!pl || !info) return fail(PFBG_ERR_ARG, "null argument");
  memset(info, 0, sizeof *info);
  info->nrow = pl->nrow; info->nvis = pl->nvis; info->nactive = pl->nactive;
  // bytes of plane stack this plan needs (== what it holds when it owns its stack; a lent stack may be larger)
  info->grid_bytes = (int64_t)((size_t)pl->stack_planes * pl->gp.nu * pl->gp.nv * 2 * real_bytes(pl));
  info->total_bytes = (int64_t)pl->total_bytes;
  info->nchan = pl->gp.nchan; info->nplanes = pl->gp.nplanes;
  info->nu = pl->gp.nu; info->nv = pl->gp.nv; info->W = pl->gp.W;
  info->n_work_items = 0;
  return PFBG_OK;
}

extern "C" int pfbg_plan_get_window(const pfbg_plan* pl, int32_t* w) {
  if (!pl || !w) return fail(PFBG_ERR_ARG, "null argument");
  w[0] = pl->ftabs.a_lo; w[1] = pl->ftabs.a_len; w[2] = pl->ftabs.b_lo; w[3] = pl->ftabs.b_len;
  return PFBG_OK;
}

extern "C" int pfbg_set_profiling(pfbg_plan* pl, int32_t on) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  CK(cudaSetDevice(pl->device));
  if (on && !pl->ev_ok) {
    for (auto& e : pl->ev) CK(cudaEventCreate(&e));
    pl->ev_ok = true;
  }
  pl->profiling = on != 0;
  pl->n_ev = 0;
  return PFBG_OK;
}
static inline void mark(pfbg_plan* pl, cudaStream_t s) {
  if (pl->profiling && pl->n_ev < 8) cudaEventRecord(pl->ev[pl->n_ev++], s);
}
extern "C" int pfbg_get_timings(pfbg_plan* pl, float* ms, int32_t n, int32_t* n_written) {
  if (!pl || !ms || !n_written) return fail(PFBG_ERR_ARG, "null argument");
  *n_written = 0;
  if (!pl->profiling || pl->n_ev < 2) return PFBG_OK;
  CK(cudaSetDevice(pl->device));
  CK(cudaEventSynchronize(pl->ev[pl->n_ev - 1]));
  for (int i = 0; i + 1 < pl->n_ev && i < n; ++i) {
    CK(cudaEventElapsedTime(&ms[i], pl->ev[i], pl->ev[i + 1]));
    *n_written = i + 1;
  }
  return PFBG_OK;
}

// ---------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------
static int host_threads() {
  static int n = [] {
    const char* e = getenv("PFBG_COPY_THREADS");
    int v = e ? atoi(e) : 0;
    if (v <= 0) {
      v = (int)std::thread::hardware_concurrency() / 2;
      if (v > 8) v = 8;
    }
    return v < 1 ? 1 : v;
  }();
  return n;
}

static void par_memcpy(void* dst, const void* src, size_t n) {
  const int nt = host_threads();
  if (nt == 1 || n < (size_t)(1 << 20)) { memcpy(dst, src, n); return; }
  std::vector<std::thread> th;
  // ceil(n / nt) rounded up to 64 bytes: the nt chunks cover all n bytes (floor(n / nt) would drop the last n % nt
  // when it is a multiple of 64)
  const size_t per = ((n + nt - 1) / nt + 63) & ~(size_t)63;
  for (int t = 0; t < nt; ++t) {
    size_t off = (size_t)t * per;
    if (off >= n) break;
    size_t len = off + per > n ? n - off : per;
    th.emplace_back([=] { memcpy((char*)dst + off, (const char*)src + off, len); });
  }
  for (auto& t : th) t.join();
}

// 64-bit content hash of a host range on several threads (memory-bandwidth bound: ~150 MB in a few ms).  The
// operator-level plan cache keys a bound band on the CONTENT of the caller's uvw / mask / weight / beam arrays
// with it: a single flipped flag or re-weighted sample changes the hash (a sampled checksum would miss it).
static inline uint64_t mix64(uint64_t h, uint64_t w) {
  h ^= w;
  h *= 0x9E3779B97F4A7C15ull;
  return h ^ (h >> 29);
}
static uint64_t hash_range(const unsigned char* p, size_t n, uint64_t seed) {
  uint64_t h[4] = {seed ^ 0x243F6A8885A308D3ull, seed ^ 0x13198A2E03707344ull, seed ^ 0xA4093822299F31D0ull, seed ^ 0x082EFA98EC4E6C89ull};
  size_t i = 0;
  for (; i + 32 <= n; i += 32) {  // four independent lanes: the multiplies overlap
    uint64_t w[4];
    memcpy(w, p + i, 32);
    h[0] = mix64(h[0], w[0]); h[1] = mix64(h[1], w[1]); h[2] = mix64(h[2], w[2]); h[3] = mix64(h[3], w[3]);
  }
  uint64_t tail = 0;
  if (i < n) memcpy(&tail, p + i, n - i > 8 ? 8 : n - i);
  for (size_t k = i + 8; k < n; ++k) tail = mix64(tail, p[k]);
  uint64_t r = mix64(mix64(mix64(mix64(h[0], h[1]), h[2]), h[3]), tail);
  return mix64(r, (uint64_t)n);
}
extern "C" int pfbg_host_hash64(const void* ptr, uint64_t bytes, uint64_t* out) {
  if (!out || (!ptr && bytes)) return fail(PFBG_ERR_ARG, "null argument");
  const unsigned char* p = (const unsigned char*)ptr;
  const size_t n = (size_t)bytes;
  const int nt = n < ((size_t)4 << 20) ? 1 : host_threads();
  if (nt == 1) { *out = hash_range(p, n, 0); return PFBG_OK; }
  std::vector<uint64_t> part(nt, 0);
  std::vector<std::thread> th;
  const size_t per = ((n + nt - 1) / nt + 63) & ~(size_t)63;  // covers all n bytes (see par_memcpy)
  for (int t = 0; t < nt; ++t) {
    const size_t off = (size_t)t * per;
    if (off >= n) break;
    const size_t len = off + per > n ? n - off : per;
    th.emplace_back([=, &part] { part[t] = hash_range(p + off, len, (uint64_t)t + 1); });
  }
  for (auto& t : th) t.join();
  uint64_t r = 0x6A09E667F3BCC908ull;
  for (int t = 0; t < nt; ++t) r = mix64(r, part[t]);
  *out = r;
  return PFBG_OK;
}

static int pinned(void*& p, size_t& have, size_t need) {
  if (have >= need) return PFBG_OK;
  if (p) {
    cudaDeviceSynchronize();  // earlier async copies may still read the old buffer
    cudaFreeHost(p);
  }
  p = nullptr; have = 0;
  cudaError_t e = cudaHostAlloc(&p, need, cudaHostAllocDefault);
  if (e != cudaSuccess) { p = nullptr; return fail(PFBG_ERR_NOMEM, "cudaHostAlloc of %zu bytes failed: %s", need, cudaGetErrorString(e)); }
  have = need;
  return PFBG_OK;
}

static const size_t kChunk = (size_t)32 << 20;  // per-chunk thread spawn amortised; copy of chunk c+1 overlaps the DMA of chunk c

// host -> device through the pinned buffer: CPU copy of chunk c+1 overlaps the DMA of chunk c
static int h2d_staged(pfbg_plan* pl, void* dst, const void* src, size_t bytes, cudaStream_t s, size_t pin_off = 0) {
  if (bytes == 0) return PFBG_OK;
  CKRC(pinned(pl->h_in, pl->h_in_bytes, pin_off + bytes));
  // the pinned buffer may still feed an earlier async copy on this stream
  if (pin_off == 0) CK(cudaStreamSynchronize(s));
  for (size_t off = 0; off < bytes; off += kChunk) {
    size_t len = off + kChunk > bytes ? bytes - off : kChunk;
    par_memcpy((char*)pl->h_in + pin_off + off, (const char*)src + off, len);
    CK(cudaMemcpyAsync((char*)dst + off, (char*)pl->h_in + pin_off + off, len, cudaMemcpyHostToDevice, s));
  }
  return PFBG_OK;
}

// device -> host: DMA every chunk into the pinned buffer, copy chunk c out while c+1 is in flight
static int d2h_staged(pfbg_plan* pl, void* dst, const void* src, size_t bytes, cudaStream_t s) {
  if (bytes == 0) return PFBG_OK;
  CKRC(pinned(pl->h_out, pl->h_out_bytes, bytes));
  if (!pl->stage_ev_ok) {
    for (auto& e : pl->stage_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    pl->stage_ev_ok = true;
  }
  const size_t nchunk = (bytes + kChunk - 1) / kChunk;
  for (size_t base = 0; base < nchunk; base += 16) {
    const size_t nb = nchunk - base < 16 ? nchunk - base : 16;
    for (size_t c = 0; c < nb; ++c) {
      size_t off = (base + c) * kChunk, len = off + kChunk > bytes ? bytes - off : kChunk;
      CK(cudaMemcpyAsync((char*)pl->h_out + off, (const char*)src + off, len, cudaMemcpyDeviceToHost, s));
      CK(cudaEventRecord(pl->stage_ev[c], s));
    }
    for (size_t c = 0; c < nb; ++c) {
      size_t off = (base + c) * kChunk, len = off + kChunk > bytes ? bytes - off : kChunk;
      CK(cudaEventSynchronize(pl->stage_ev[c]));
      par_memcpy((char*)dst + off, (char*)pl->h_out + off, len);
    }
  }
  return PFBG_OK;
}

extern "C" int pfbg_host_register(void* ptr, uint64_t bytes) {
  if (!ptr || !bytes) return fail(PFBG_ERR_ARG, "null range");
  cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(PFBG_ERR_CUDA, "cudaHostRegister failed: %s", cudaGetErrorString(e)); }
  return PFBG_OK;
}
extern "C" int pfbg_host_unregister(void* ptr) {
  if (!ptr) return PFBG_OK;
  cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(PFBG_ERR_CUDA, "cudaHostUnregister failed: %s", cudaGetErrorString(e)); }
  return PFBG_OK;
}

static int fetch(pfbg_plan* pl, DevBuf& stage, const void* src, size_t bytes, bool dev, cudaStream_t s,
                 const void** out, size_t pin_off = 0, bool src_pinned = false) {
  // device pointers are used in place; host pointers are staged on the stream
  if (dev) { *out = src; return PFBG_OK; }
  CKRC(dev_alloc(pl, stage, bytes));
  if (src_pinned) {  // caller-registered memory: one DMA, no staging copy
    CK(cudaMemcpyAsync(stage.p, src, bytes, cudaMemcpyHostToDevice, s));
    *out = stage.p;
    return PFBG_OK;
  }
  CKRC(h2d_staged(pl, stage.p, src, bytes, s, pin_off));
  *out = stage.p;
  return PFBG_OK;
}

static int fft_exec(pfbg_plan* pl, cudaStream_t s, int dir) {
  CKFFT(cufftSetStream(pl->fft, s));
  const size_t plane = (size_t)pl->gp.nu * pl->gp.nv;
  for (int p0 = 0; p0 < pl->gp.nplanes; p0 += pl->fft_batch) {
    if (pl->precision == PFBG_F32) {
      cufftComplex* g = (cufftComplex*)pl->grid.p + (size_t)p0 * plane;
      CKFFT(cufftExecC2C(pl->fft, g, g, dir));
    } else {
      cufftDoubleComplex* g = (cufftDoubleComplex*)pl->grid.p + (size_t)p0 * plane;
      CKFFT(cufftExecZ2Z(pl->fft, g, g, dir));
    }
    LAUNCHED();
  }
  return PFBG_OK;
}

// slice length of the run kernels' work queue: RUN_SLICE when every resident warp gets at least four of them,
// shorter (a multiple of RUN_SLICE_TAIL) for small bindings so that all warps have work
static int run_slice(const pfbg_plan* pl, int64_t nact, int warps_per_cta, int ctas_per_sm) {
  int sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, pl->device);
  const int64_t per_warp = nact / ((int64_t)sm * ctas_per_sm * warps_per_cta * 4);
  int64_t sl = per_warp / RUN_SLICE_TAIL * RUN_SLICE_TAIL;
  return (int)(sl < RUN_SLICE_TAIL ? RUN_SLICE_TAIL : (sl > RUN_SLICE ? RUN_SLICE : sl));
}

static int run_blocks(const pfbg_plan* pl, int64_t nact, int warps_per_cta, int ctas_per_sm) {
  int sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, pl->device);
  int64_t nslice = (nact + RUN_SLICE_TAIL - 1) / RUN_SLICE_TAIL;
  int64_t want = (nslice + warps_per_cta - 1) / warps_per_cta;
  int64_t cap = (int64_t)sm * ctas_per_sm;  // a multiple of the SM count: one full wave of resident CTAs
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

static int wide_blocks(const pfbg_plan* pl, int64_t nact, int team) {
  int sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, pl->device);
  int64_t nslice = (nact + WIDE_SLICE - 1) / WIDE_SLICE;
  int64_t want = (nslice * team + WIDE_WARPS - 1) / WIDE_WARPS;
  int64_t cap = (int64_t)sm * 2;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

// kernel family of the spreading / gathering passes of a binding: direct (no per-sample records), the one-warp run
// kernels (W <= 8), the scalar team kernels wide<3, 6, 4> (W <= 12) and wide<2, 8, 8>, or in fp64 at 9 <= W <= 12 the
// DMMA run kernels (runs_mma.cuh) unless PFBG_WIDE_MMA=0 asks for the scalar team kernels
enum RunArm { ARM_DIRECT, ARM_RUNS, ARM_WIDE6, ARM_WIDE8, ARM_MMA };
static RunArm run_arm(const pfbg_plan* pl) {
  if (!pl->use_runs) return ARM_DIRECT;
  if (pl->gp.W <= 8) return ARM_RUNS;
  if (pl->precision == PFBG_F64 && pl->gp.W <= 12) {
    const char* e = getenv("PFBG_WIDE_MMA");
    if (!(e && e[0] == '0')) return ARM_MMA;
  }
  return pl->gp.W <= 12 ? ARM_WIDE6 : ARM_WIDE8;
}

static int mma_blocks(const pfbg_plan* pl, int64_t nact) {
  int sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, pl->device);
  int64_t nslice = (nact + MMA_SLICE - 1) / MMA_SLICE;
  int64_t want = (nslice + MMA_TEAMS - 1) / MMA_TEAMS;
  int64_t cap = (int64_t)sm * 5;  // 5 resident 96-thread CTAs per SM (128 registers)
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

static int grid_blocks(const pfbg_plan* pl, int64_t nact) {
  int sm = 148;
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, pl->device);
  int64_t want = (nact + 7) / 8;
  int64_t cap = (int64_t)sm * 8;  // 8 resident CTAs of 256 threads per SM
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

// ---------------------------------------------------------------------------
// kernel 1: bind + bin + sort
// ---------------------------------------------------------------------------
extern "C" int pfbg_bind_vis(pfbg_plan* pl, const double* uvw, const double* fscale, const uint8_t* mask,
                             int64_t nrow, int32_t nchan, uint32_t flags, void* stream) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  if (nrow < 0 || nchan <= 0) return fail(PFBG_ERR_ARG, "bad nrow/nchan");
  if ((!uvw && nrow > 0) || !fscale) return fail(PFBG_ERR_ARG, "null uvw/fscale");
  int64_t nvis = nrow * (int64_t)nchan;
  if (nvis >= (int64_t)UINT32_MAX) return fail(PFBG_ERR_ARG, "more than 2^32-1 samples in one binding");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const cudaMemcpyKind kind = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  pl->bound = false;
  pl->gp.nchan = nchan;
  pl->nrow = nrow; pl->nvis = nvis; pl->nactive = 0;
  pl->has_wgt = false;
  CKRC(dev_alloc(pl, pl->uvw, (size_t)(nrow > 0 ? nrow : 1) * 3 * sizeof(double)));
  CKRC(dev_alloc(pl, pl->fscale, (size_t)nchan * sizeof(double)));
  // host arrays go through the pinned staging pipeline (threaded copy overlapped with the DMA), not a pageable memcpy
  if (nrow > 0) {
    if (dev) CK(cudaMemcpyAsync(pl->uvw.p, uvw, (size_t)nrow * 3 * sizeof(double), kind, s));
    else CKRC(h2d_staged(pl, pl->uvw.p, uvw, (size_t)nrow * 3 * sizeof(double), s));
  }
  CK(cudaMemcpyAsync(pl->fscale.p, fscale, (size_t)nchan * sizeof(double), kind, s));
  pl->has_mask = mask != nullptr;
  if (mask && nvis > 0) {
    CKRC(dev_alloc(pl, pl->mask, (size_t)nvis));
    if (dev) CK(cudaMemcpyAsync(pl->mask.p, mask, (size_t)nvis, kind, s));
    else CKRC(h2d_staged(pl, pl->mask.p, mask, (size_t)nvis, s));
  }
  if (nvis == 0) {
    pl->bound = true;
    CK(cudaStreamSynchronize(s));
    return PFBG_OK;
  }
  const GParams& g = pl->gp;
  // key width
  uint64_t maxkey = (uint64_t)g.ntile_u * g.ntile_v * (uint64_t)(g.nplanes + g.pmirror) * (PFBG_TILE * PFBG_TILE);
  int bits = 1;
  while ((1ull << bits) <= maxkey) ++bits;  // inactive key = maxkey needs `bits` bits
  DevBuf &keys_a = pl->srt_ka, &keys_b = pl->srt_kb, &vals_a = pl->srt_va, &vals_b = pl->srt_vb, &tmp = pl->srt_tmp;
  // keep the sort scratch (28 B per sample) for the next binding of this plan: pooled plans of one-shot calls re-bind
  // all the time (pfb grid: dirty, PSF, residual per band) and cudaMalloc / cudaFree of ~1 GB cost more than the sort
  const bool keep_scratch = nvis <= (int64_t)(96 << 20);
  auto cleanup = [&]() {
    if (keep_scratch) return;
    dev_free(pl, keys_a); dev_free(pl, keys_b); dev_free(pl, vals_a); dev_free(pl, vals_b); dev_free(pl, tmp);
  };
  int rc;
  if ((rc = dev_alloc(pl, keys_a, nvis * 8)) || (rc = dev_alloc(pl, keys_b, nvis * 8)) ||
      (rc = dev_alloc(pl, vals_a, nvis * 4)) || (rc = dev_alloc(pl, vals_b, nvis * 4))) { cleanup(); return rc; }
  CK(cudaMemsetAsync(pl->flag.p, 0, 64, s));
  {
    int blk = 256;
    int64_t grd = (nvis + blk - 1) / blk;
    k_bin<<<(unsigned)grd, blk, 0, s>>>(g, (const double*)pl->uvw.p, (const double*)pl->fscale.p,
                                        pl->has_mask ? (const uint8_t*)pl->mask.p : nullptr, nvis, maxkey,
                                        (uint64_t*)keys_a.p, (uint32_t*)vals_a.p, (unsigned long long*)pl->flag.p);
    LAUNCHED();
  }
  size_t tmp_bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const uint64_t*)keys_a.p, (uint64_t*)keys_b.p,
                                                  (const uint32_t*)vals_a.p, (uint32_t*)vals_b.p, nvis, 0, bits, s);
  if (e != cudaSuccess) { cleanup(); return fail(PFBG_ERR_CUDA, "cub sort sizing failed: %s", cudaGetErrorString(e)); }
  if ((rc = dev_alloc(pl, tmp, tmp_bytes ? tmp_bytes : 16))) { cleanup(); return rc; }
  e = cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, (const uint64_t*)keys_a.p, (uint64_t*)keys_b.p,
                                      (const uint32_t*)vals_a.p, (uint32_t*)vals_b.p, nvis, 0, bits, s);
  LAUNCHED();
  if (e != cudaSuccess) { cleanup(); return fail(PFBG_ERR_CUDA, "cub sort failed: %s", cudaGetErrorString(e)); }
  unsigned long long nact = 0;
  e = cudaMemcpyAsync(&nact, pl->flag.p, sizeof nact, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) { cleanup(); return fail(PFBG_ERR_CUDA, "binning failed: %s", cudaGetErrorString(e)); }
  pl->nactive = (int64_t)nact;
  if ((rc = dev_alloc(pl, pl->sorted_idx, (size_t)(nact ? nact : 1) * 4))) { cleanup(); return rc; }
  if (nact) {
    e = cudaMemcpyAsync(pl->sorted_idx.p, vals_b.p, (size_t)nact * 4, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { cleanup(); return fail(PFBG_ERR_CUDA, "copy of sorted order failed: %s", cudaGetErrorString(e)); }
  }
  cleanup();
  // per-sample records for the run kernels
  pl->use_runs = false;
  {
    const char* fd = getenv("PFBG_FORCE_DIRECT");
    bool force_direct = fd && fd[0] == '1';
    if (!force_direct && g.W <= 16 && g.nu <= 32768 && g.nv <= 32768 && nact > 0) {
      size_t rsz = pl->precision == PFBG_F32 ? sizeof(VisRec<float>) : sizeof(VisRec<double>);
      CKRC(dev_alloc(pl, pl->recs, (size_t)nact * rsz));
      unsigned grd = (unsigned)((nact + 255) / 256);
      if (pl->precision == PFBG_F32)
        k_make_recs<float><<<grd, 256, 0, s>>>(g, (const double*)pl->uvw.p, (const double*)pl->fscale.p,
                                                (const uint32_t*)pl->sorted_idx.p, (int64_t)nact, (VisRec<float>*)pl->recs.p);
      else
        k_make_recs<double><<<grd, 256, 0, s>>>(g, (const double*)pl->uvw.p, (const double*)pl->fscale.p,
                                                 (const uint32_t*)pl->sorted_idx.p, (int64_t)nact, (VisRec<double>*)pl->recs.p);
      LAUNCHED();
      CK(cudaGetLastError());
      CK(cudaStreamSynchronize(s));
      pl->use_runs = true;
    }
  }
  // active cell windows for the pruned transforms
  if (pl->fused) {
    FusedTabs& ft = pl->ftabs;
    ft.a_lo = 0; ft.a_len = g.nu; ft.b_lo = 0; ft.b_len = g.nv;
    if (pl->use_runs) {
      const int ngu = g.nu / 32, ngv = g.nv / 32;
      CKRC(dev_alloc(pl, pl->cellflags, (size_t)(ngu + ngv) * 4));
      CK(cudaMemsetAsync(pl->cellflags.p, 0, (size_t)(ngu + ngv) * 4, s));
      unsigned grd = (unsigned)((nact + 255) / 256);
      int* uf = (int*)pl->cellflags.p;
      if (pl->precision == PFBG_F32)
        k_mark_cells<VisRec<float>><<<grd, 256, 0, s>>>((const VisRec<float>*)pl->recs.p, (int64_t)nact, g.W, g.nu, g.nv, uf, uf + ngu);
      else
        k_mark_cells<VisRec<double>><<<grd, 256, 0, s>>>((const VisRec<double>*)pl->recs.p, (int64_t)nact, g.W, g.nu, g.nv, uf, uf + ngu);
      LAUNCHED();
      std::vector<int> fl(ngu + ngv);
      CK(cudaMemcpyAsync(fl.data(), pl->cellflags.p, fl.size() * 4, cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
      std::vector<int> fu(fl.begin(), fl.begin() + ngu), fv(fl.begin() + ngu, fl.end());
      window_from_flags(fu, g.nu, ft.a_lo, ft.a_len);
      window_from_flags(fv, g.nv, ft.b_lo, ft.b_len);
    }
  }
  pl->bound = true;
  return PFBG_OK;
}

extern "C" int pfbg_bind_weights(pfbg_plan* pl, const void* wgt, uint32_t flags, void* stream) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  if (!pl->bound) return fail(PFBG_ERR_STATE, "bind_vis must be called before bind_weights");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (!wgt || pl->nvis == 0) { pl->has_wgt = false; return PFBG_OK; }
  size_t bytes = (size_t)pl->nvis * real_bytes(pl);
  CKRC(dev_alloc(pl, pl->wgt, bytes));
  CK(cudaMemcpyAsync(pl->wgt.p, wgt, bytes, (flags & PFBG_DEVICE_PTRS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));
  pl->has_wgt = true;
  return PFBG_OK;
}

extern "C" int pfbg_bind_weights_robust(pfbg_plan* pl, const void* wgt, int32_t nx_pad, int32_t ny_pad, double cell_x,
                                        double cell_y, double robust, double usign, double vsign, uint32_t flags,
                                        void* stream) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  if (!pl->gp.row_snap || !pl->bound) return fail(PFBG_ERR_STATE, "the plan holds no batch of snapshots: pfbg_plan_set_batch and pfbg_bind_vis_batch first");
  if (!wgt && pl->nvis > 0) return fail(PFBG_ERR_ARG, "null wgt");
  if (nx_pad <= 0 || ny_pad <= 0) return fail(PFBG_ERR_ARG, "pad sizes must be positive, got %d x %d", nx_pad, ny_pad);
  if (!std::isfinite(cell_x) || !std::isfinite(cell_y) || !(cell_x > 0) || !(cell_y > 0))
    return fail(PFBG_ERR_ARG, "cell sizes must be finite and positive");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  pl->has_wgt = false;
  if (pl->nvis == 0) return PFBG_OK;
  const size_t rb = real_bytes(pl);
  const size_t cbytes = (size_t)pl->nbatch * nx_pad * ny_pad * rb, coff = (cbytes + 255) & ~(size_t)255;
  CKRC(dev_alloc(pl, pl->wgt, (size_t)pl->nvis * rb));
  CKRC(dev_alloc(pl, pl->wcounts, coff + (size_t)pl->nbatch * 3 * sizeof(double)));
  CK(cudaMemcpyAsync(pl->wgt.p, wgt, (size_t)pl->nvis * rb, (flags & PFBG_DEVICE_PTRS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  // the bound fscale is fl(freq / c): a division by lightspeed = 1 reproduces pfbg_counts' cell exactly
  CKRC(pfbg_counts_reweight(pl->precision, s, pl->nrow, pl->gp.nchan, nx_pad, ny_pad, cell_x, cell_y, usign, vsign, 1.0,
                            (const double*)pl->uvw.p, (const double*)pl->fscale.p,
                            pl->has_mask ? (const uint8_t*)pl->mask.p : nullptr, pl->gp.row_snap, pl->nbatch, robust,
                            pl->wcounts.p, (double*)((char*)pl->wcounts.p + coff), pl->wgt.p));
  if (!(flags & PFBG_DEVICE_PTRS)) CK(cudaStreamSynchronize(s));  // the caller may free its host array on return
  pl->has_wgt = true;
  return PFBG_OK;
}

extern "C" int pfbg_bin_dump(pfbg_plan* pl, int32_t* iu0, int32_t* iv0, int32_t* ip0, uint64_t* key,
                             uint32_t* sorted_idx) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  if (!pl->bound) return fail(PFBG_ERR_STATE, "no visibilities bound");
  if (!pl->grid.p) return fail(PFBG_ERR_STATE, "the plan has no plane stack (created with PFBG_PLAN_EXTERNAL_STACK): lend one with pfbg_plan_set_stack");
  CK(cudaSetDevice(pl->device));
  int64_t n = pl->nvis;
  if (n > 0 && (iu0 || iv0 || ip0 || key)) {
    DevBuf a, b, c, k;
    auto cleanup = [&]() { dev_free(pl, a); dev_free(pl, b); dev_free(pl, c); dev_free(pl, k); };
    int rc;
    if ((rc = dev_alloc(pl, a, n * 4)) || (rc = dev_alloc(pl, b, n * 4)) || (rc = dev_alloc(pl, c, n * 4)) ||
        (rc = dev_alloc(pl, k, n * 8))) { cleanup(); return rc; }
    k_bin_dump<<<(unsigned)((n + 255) / 256), 256>>>(pl->gp, (const double*)pl->uvw.p, (const double*)pl->fscale.p, n,
                                                     (int32_t*)a.p, (int32_t*)b.p, (int32_t*)c.p, (uint64_t*)k.p);
    LAUNCHED();
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess && iu0) e = cudaMemcpy(iu0, a.p, n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && iv0) e = cudaMemcpy(iv0, b.p, n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && ip0) e = cudaMemcpy(ip0, c.p, n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && key) e = cudaMemcpy(key, k.p, n * 8, cudaMemcpyDeviceToHost);
    cleanup();
    if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "bin dump failed: %s", cudaGetErrorString(e));
  }
  if (sorted_idx && pl->nactive > 0)
    CK(cudaMemcpy(sorted_idx, pl->sorted_idx.p, (size_t)pl->nactive * 4, cudaMemcpyDeviceToHost));
  return PFBG_OK;
}

// ---------------------------------------------------------------------------
// direction drivers (templated on precision)
// ---------------------------------------------------------------------------
template <typename T>
static int run_spread(pfbg_plan* pl, cudaStream_t s, const void* vis, int64_t rs, int64_t cs, const void* wgt,
                      int vis_sorted, int apply_phase) {
  using C = typename cplx_of<T>::type;
  if (pl->nactive == 0) return PFBG_OK;
  const RunArm arm = run_arm(pl);
  const VisRec<T>* recs = (const VisRec<T>*)pl->recs.p;
  unsigned long long* queue = (unsigned long long*)((char*)pl->flag.p + 16);  // slice counter of this launch
  if (arm != ARM_DIRECT) CK(cudaMemsetAsync(queue, 0, 8, s));
  switch (arm) {
    case ARM_MMA:
      if constexpr (sizeof(T) == 8)
        k_grid_runs_mma<<<mma_blocks(pl, pl->nactive), MMA_R * MMA_TEAMS * 32, 0, s>>>(
            pl->gp, recs, pl->nactive, (const double2*)vis, rs, cs, (const double*)wgt, (double2*)pl->grid.p,
            vis_sorted, apply_phase, queue);
      break;
    case ARM_WIDE6:
      k_grid_runs_wide<T, 3, 6, 4><<<wide_blocks(pl, pl->nactive, 4), WIDE_WARPS * 32, 0, s>>>(
          pl->gp, recs, pl->nactive, (const C*)vis, rs, cs, (const T*)wgt, (C*)pl->grid.p, vis_sorted, apply_phase,
          queue);
      break;
    case ARM_WIDE8:
      k_grid_runs_wide<T, 2, 8, 8><<<wide_blocks(pl, pl->nactive, 8), WIDE_WARPS * 32, 0, s>>>(
          pl->gp, recs, pl->nactive, (const C*)vis, rs, cs, (const T*)wgt, (C*)pl->grid.p, vis_sorted, apply_phase,
          queue);
      break;
    case ARM_RUNS: {
      const int ctas = 3;  // resident CTAs per SM
      const int slice = run_slice(pl, pl->nactive, RUN_WARPS, ctas);
      k_grid_runs<T><<<run_blocks(pl, pl->nactive, RUN_WARPS, ctas), RUN_WARPS * 32, 0, s>>>(
          pl->gp, recs, pl->nactive, (const C*)vis, rs, cs, (const T*)wgt, (C*)pl->grid.p, vis_sorted, apply_phase,
          queue, slice);
      break;
    }
    case ARM_DIRECT:
      k_grid_direct<T><<<grid_blocks(pl, pl->nactive), 256, 0, s>>>(
          pl->gp, (const double*)pl->uvw.p, (const double*)pl->fscale.p, (const uint32_t*)pl->sorted_idx.p, pl->nactive,
          (const C*)vis, rs, cs, (const T*)wgt, (C*)pl->grid.p, vis_sorted, apply_phase);
      break;
  }
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int run_gather(pfbg_plan* pl, cudaStream_t s, const void* wgt, void* vis_out, void* out_sorted, int apply_phase,
                      int vis_zeroed = 0) {
  using C = typename cplx_of<T>::type;
  if (pl->nactive == 0) return PFBG_OK;
  const RunArm arm = run_arm(pl);
  const VisRec<T>* recs = (const VisRec<T>*)pl->recs.p;
  const bool team = arm == ARM_WIDE6 || arm == ARM_WIDE8 || arm == ARM_MMA;
  if (team) {
    // the R warps of a team add their row-partials atomically: start from zero
    if (out_sorted) CK(cudaMemsetAsync(out_sorted, 0, (size_t)pl->nactive * sizeof(C), s));
    else if (!pl->has_mask) CK(cudaMemsetAsync(vis_out, 0, (size_t)pl->nvis * sizeof(C), s));
    else if (vis_zeroed == 0) {  // PFBG_NO_MASK_ZERO: masked samples stay untouched, only the active ones start from zero
      k_zero_active<C><<<(unsigned)((pl->nactive + 255) / 256), 256, 0, s>>>((C*)vis_out, (const uint32_t*)pl->sorted_idx.p, pl->nactive);
      LAUNCHED();
    }
  }
  // slice counters of this launch: one per row group (<= 8) for the team kernels
  unsigned long long* queue = (unsigned long long*)((char*)pl->flag.p + (team ? 32 : 24));
  if (arm != ARM_DIRECT) CK(cudaMemsetAsync(queue, 0, team ? 64 : 8, s));
  // per-sample lane partials of the team kernels (see k_degrid_runs_wide); the attribute is per device and cheap: set
  // on every launch rather than cached per process
  const size_t psm = (size_t)WIDE_WARPS * 16 * 32 * sizeof(C);
  switch (arm) {
    case ARM_MMA:
      if constexpr (sizeof(T) == 8)
        k_degrid_runs_mma<<<mma_blocks(pl, pl->nactive), MMA_R * MMA_TEAMS * 32, 0, s>>>(
            pl->gp, recs, pl->nactive, (const double2*)pl->grid.p, (const double*)wgt, (double2*)vis_out,
            (double2*)out_sorted, apply_phase, queue);
      break;
    case ARM_WIDE6:
      CK(cudaFuncSetAttribute(k_degrid_runs_wide<T, 3, 6, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
      k_degrid_runs_wide<T, 3, 6, 4><<<wide_blocks(pl, pl->nactive, 4), WIDE_WARPS * 32, psm, s>>>(
          pl->gp, recs, pl->nactive, (const C*)pl->grid.p, (const T*)wgt, (C*)vis_out, (C*)out_sorted, apply_phase,
          queue);
      break;
    case ARM_WIDE8:
      CK(cudaFuncSetAttribute(k_degrid_runs_wide<T, 2, 8, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
      k_degrid_runs_wide<T, 2, 8, 8><<<wide_blocks(pl, pl->nactive, 8), WIDE_WARPS * 32, psm, s>>>(
          pl->gp, recs, pl->nactive, (const C*)pl->grid.p, (const T*)wgt, (C*)vis_out, (C*)out_sorted, apply_phase,
          queue);
      break;
    case ARM_RUNS: {
      const int ctas = 5;  // resident CTAs per SM
      const int slice = run_slice(pl, pl->nactive, DEG_WARPS, ctas);
      k_degrid_runs<T><<<run_blocks(pl, pl->nactive, DEG_WARPS, ctas), DEG_WARPS * 32, 0, s>>>(
          pl->gp, recs, pl->nactive, (const C*)pl->grid.p, (const T*)wgt, (C*)vis_out, (C*)out_sorted, apply_phase,
          queue, slice);
      break;
    }
    case ARM_DIRECT:
      k_degrid_direct<T><<<grid_blocks(pl, pl->nactive), 256, 0, s>>>(
          pl->gp, (const double*)pl->uvw.p, (const double*)pl->fscale.p, (const uint32_t*)pl->sorted_idx.p, pl->nactive,
          (const C*)pl->grid.p, (const T*)wgt, (C*)vis_out, (C*)out_sorted, apply_phase);
      break;
  }
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int run_img2grid(pfbg_plan* pl, cudaStream_t s, const void* x, const void* beam) {
  using C = typename cplx_of<T>::type;
  const GParams& g = pl->gp;
  dim3 blk(256), grd((g.nv + 255) / 256, g.nu);
  k_img2grid<T><<<grd, blk, 0, s>>>(g, (const T*)x, (const T*)beam, (const T*)pl->corr.p, (C*)pl->grid.p);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int run_grid2img(pfbg_plan* pl, cudaStream_t s, const void* beam, const void* xin, double inv_wsum, double eta,
                        void* out) {
  using C = typename cplx_of<T>::type;
  const GParams& g = pl->gp;
  dim3 blk(256), grd((g.ny + 255) / 256, g.nx);
  k_grid2img<T><<<grd, blk, 0, s>>>(g, (const C*)pl->grid.p, (const T*)pl->corr.p, (const T*)beam, (const T*)xin,
                                    inv_wsum, eta, (T*)out);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

// TMA-fed pair-engine column pass (cols2.cuh) over logical planes [ft.q0, ft.q0 + nq): loads come from the local
// stack (slot 0 = logical plane slot0), results go to `out_biased` (logical plane q at out_biased + q nu nv)
static int run_cols2(pfbg_plan* pl, cudaStream_t s, const FusedTabs& ft, int slot0, int nq, bool inverse,
                     float2* out_biased) {
  const GParams& g = pl->gp;
  Cols2Args a;
  a.du = ft.du;
  a.tw_u = (const float2*)ft.tw_u;
  a.pos_u = ft.pos_u;
  a.nu = g.nu; a.nv = g.nv; a.nx = g.nx;
  a.a_lo = ft.a_lo; a.a_len = ft.a_len; a.b_lo = ft.b_lo; a.b_len = ft.b_len;
  a.q0 = ft.q0; a.nq = nq; a.slot0 = slot0;
  a.inverse = inverse ? 1 : 0;
  const char* what = "";
  cudaError_t e = cols2_launch(a, (const float2*)pl->grid.p, pl->stack_planes, out_biased, s, &what);
  if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  LAUNCHED();
  return PFBG_OK;
}

// Row pass of planes [ft.q0, ft.q0 + nq): the first nq2 on the pair engine (fp32, two planes per CTA; a last odd plane
// would cost a whole pair slot there, the one-plane kernel does it for ~0.55 of one: C2 has 4 bands with an odd plane
// count), the rest on the one-plane kernel, whose BIG variant (480-768 threads) takes rows whose FFT leaves one CTA per
// SM unless PFBG_ROWS_SMALL asks for the small one
struct RowSplit { int nq2, threads; bool big; };
template <typename T>
static RowSplit row_split(const pfbg_plan* pl, int nq) {
  const bool big = fft_smem_bytes<T>(pl->gp.nv) > (size_t)ROWS_BIG_SMEM && !getenv("PFBG_ROWS_SMALL");
  const int cap = !big ? ROWS_MAX_THREADS : sizeof(T) == 4 ? ROWS_BIG_THREADS_F32 : ROWS_BIG_THREADS_F64;
  return {sizeof(T) == 4 && pl->rows2 ? nq & ~1 : 0, row_threads(pl->gp.nv, cap, sizeof(T) == 8 ? 8 : 16), big};
}

// forward row pass (pad + screen the image, FFT along v) of planes [ft.q0, ft.q0 + nq) into the biased stack
template <typename T>
static int run_rows_fwd(pfbg_plan* pl, cudaStream_t s, const FusedTabs& ft, int nq, const void* x, const void* beam,
                        typename cplx_of<T>::type* stack) {
  const GParams& g = pl->gp;
  const RowSplit r = row_split<T>(pl, nq);
  const int nq2 = r.nq2;
  if constexpr (sizeof(T) == 4) {
    if (nq2 > 0) {
      cudaError_t e = rows2_fwd_launch(g, ft, nq2, g.fast_screen != 0, (const float*)x, (const float*)beam,
                                       (const float*)pl->corr.p, (float2*)stack, s);
      if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "k_rows2_fwd launch: %s", cudaGetErrorString(e));
      LAUNCHED();
    }
  }
  if (nq2 < nq) {
    auto k_rows = r.big ? &k_rows_fwd<T, false, true> : &k_rows_fwd<T, false>;
    if constexpr (sizeof(T) == 4) {
      if (g.fast_screen) k_rows = r.big ? &k_rows_fwd<T, true, true> : &k_rows_fwd<T, true>;
    }
    FusedTabs ft1 = ft;
    ft1.q0 = ft.q0 + nq2;
    k_rows<<<dim3(nq - nq2, g.nx), r.threads, fft_smem_bytes<T>(g.nv), s>>>(g, ft1, (const T*)x, (const T*)beam,
                                                                        (const T*)pl->corr.p, stack);
    LAUNCHED();
  }
  CK(cudaGetLastError());
  return PFBG_OK;
}

// inverse row pass (FFT along v, screen + crop) of planes [ft.q0, ft.q0 + nq), accumulated into accimg
template <typename T>
static int run_rows_inv(pfbg_plan* pl, cudaStream_t s, const FusedTabs& ft, int nq,
                        const typename cplx_of<T>::type* stack) {
  const GParams& g = pl->gp;
  const RowSplit r = row_split<T>(pl, nq);
  const int nq2 = r.nq2;
  if constexpr (sizeof(T) == 4) {
    if (nq2 > 0) {
      cudaError_t e = rows2_inv_launch(g, ft, nq2, g.fast_screen != 0, (const float2*)stack, (double*)pl->accimg.p, s);
      if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "k_rows2_inv launch: %s", cudaGetErrorString(e));
      LAUNCHED();
    }
  }
  if (nq2 < nq) {
    auto k_rows = r.big ? &k_rows_inv<T, false, true> : &k_rows_inv<T, false>;
    if constexpr (sizeof(T) == 4) {
      if (g.fast_screen) k_rows = r.big ? &k_rows_inv<T, true, true> : &k_rows_inv<T, true>;
    }
    FusedTabs ft1 = ft;
    ft1.q0 = ft.q0 + nq2;
    k_rows<<<dim3(nq - nq2, g.nx), r.threads, fft_smem_bytes<T>(g.nv), s>>>(g, ft1, stack, (double*)pl->accimg.p);
    LAUNCHED();
  }
  CK(cudaGetLastError());
  return PFBG_OK;
}

// one-plane column pass (fused_fft.cuh) of planes [ft.q0, ft.q0 + nq) in blocks of pl->col_c columns, src -> dst
template <typename T>
static int run_cols(pfbg_plan* pl, cudaStream_t s, const FusedTabs& ft, int nq, bool inverse,
                    const typename cplx_of<T>::type* src, typename cplx_of<T>::type* dst) {
  const int cc = pl->col_c;
  const auto k_cols = inverse ? (cc == 4 ? &k_cols_inv<T, 4> : cc == 2 ? &k_cols_inv<T, 2> : &k_cols_inv<T, 1>)
                              : (cc == 4 ? &k_cols_fwd<T, 4> : cc == 2 ? &k_cols_fwd<T, 2> : &k_cols_fwd<T, 1>);
  k_cols<<<dim3(ft.b_len / cc, nq), 512, fft_smem_bytes<T>(pl->gp.nu * cc), s>>>(pl->gp, ft, src, dst);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

// Plane subset of the fused transforms: logical planes [q0, q0 + nq).  `stack` is the local plane stack biased so
// that logical plane q sits at stack + q * nu * nv (a helper of a split band stores plane q0 in slot 0); `remote`
// (optional) is the peer-mapped stack of the band's owner: the forward column pass then writes there and the
// inverse column pass reads from there — the transfer over NVLink is fused into the transform kernels.
template <typename T>
static int run_fused_fwd(pfbg_plan* pl, cudaStream_t s, const void* x, const void* beam, int q0 = 0, int nq = -1,
                         void* remote = nullptr) {
  using C = typename cplx_of<T>::type;
  const GParams& g = pl->gp;
  if (nq < 0) nq = g.nplanes - (pl->split_role == 1 ? pl->split_nq : 0);
  if (nq == 0) return PFBG_OK;
  FusedTabs ft = pl->ftabs;
  ft.q0 = q0;
  const int slot0 = pl->split_role == 2 ? g.nplanes - pl->split_nq : 0;  // logical plane held by slot 0
  C* stack = (C*)pl->grid.p - (int64_t)slot0 * g.nu * g.nv;
  CKRC(run_rows_fwd<T>(pl, s, ft, nq, x, beam, stack));
  C* dst = remote ? (C*)remote : stack;
  if (pl->cols2) return run_cols2(pl, s, ft, slot0, nq, false, (float2*)dst);
  return run_cols<T>(pl, s, ft, nq, false, stack, dst);
}

// inverse transforms of planes [q0, q0 + nq) accumulated into accimg (zeroed first)
template <typename T>
static int run_fused_inv_acc(pfbg_plan* pl, cudaStream_t s, int q0, int nq, const void* remote) {
  using C = typename cplx_of<T>::type;
  const GParams& g = pl->gp;
  FusedTabs ft = pl->ftabs;
  ft.q0 = q0;
  const int slot0 = pl->split_role == 2 ? g.nplanes - pl->split_nq : 0;
  C* stack = (C*)pl->grid.p - (int64_t)slot0 * g.nu * g.nv;
  const int64_t npix = (int64_t)img_elems(pl);
  CK(cudaMemsetAsync(pl->accimg.p, 0, (size_t)npix * sizeof(double), s));
  if (nq == 0) return PFBG_OK;
  // (a helper's loads from the owner's peer-mapped stack stay on the one-plane kernel)
  if (pl->cols2 && !remote) CKRC(run_cols2(pl, s, ft, slot0, nq, true, (float2*)stack));
  else CKRC(run_cols<T>(pl, s, ft, nq, true, remote ? (const C*)remote : stack, stack));
  return run_rows_inv<T>(pl, s, ft, nq, stack);
}

static int split_wait(pfbg_plan* pl, cudaStream_t s, int slot);
static int split_signal(pfbg_plan* pl, cudaStream_t s, int slot);

template <typename T>
static int run_fused_inv(pfbg_plan* pl, cudaStream_t s, const void* beam, const void* xin, double inv_wsum, double eta,
                         void* out) {
  const GParams& g = pl->gp;
  const bool owner = pl->split_role == 1;
  CKRC(run_fused_inv_acc<T>(pl, s, 0, g.nplanes - (owner ? pl->split_nq : 0), nullptr));
  const int64_t npix = (int64_t)img_elems(pl);
  if (owner) CKRC(split_wait(pl, s, 1));  // the helper's partial image (its planes) has arrived
  k_finish_image<T><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>(npix, (int64_t)g.nx * g.ny, (const double*)pl->accimg.p,
                                                                owner ? (const double*)pl->partial.p : nullptr,
                                                                (const T*)pl->corr.p, (const T*)beam, (const T*)xin,
                                                                inv_wsum, eta, (T*)out);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

template <typename T>
static int run_zero_window(pfbg_plan* pl, cudaStream_t s) {
  using C = typename cplx_of<T>::type;
  const GParams& g = pl->gp;
  const FusedTabs& ft = pl->ftabs;
  int bx = (ft.b_len + 1023) / 1024;
  k_zero_window<C><<<dim3(bx, ft.a_len, g.nplanes), 256, 0, s>>>((C*)pl->grid.p, g.nu, g.nv, ft.a_lo, ft.a_len, ft.b_lo, ft.b_len);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

#define DISPATCH(fn, ...) (pl->precision == PFBG_F32 ? fn<float>(__VA_ARGS__) : fn<double>(__VA_ARGS__))

// image -> screened, transformed plane stack (degrid direction)
static int image_to_planes(pfbg_plan* pl, cudaStream_t s, const void* x, const void* beam) {
  if (pl->fused) return DISPATCH(run_fused_fwd, pl, s, x, beam);
  if (pl->nbatch > 1) return fail(PFBG_ERR_STATE, "batched plans need the fused plane transforms");
  CKRC(cufft_setup(pl));
  CKRC(DISPATCH(run_img2grid, pl, s, x, beam));
  return fft_exec(pl, s, CUFFT_FORWARD);
}
// plane stack -> image with the fused epilogue (grid direction)
static int planes_to_image(pfbg_plan* pl, cudaStream_t s, const void* beam, const void* xin, double inv_wsum,
                           double eta, void* out) {
  if (pl->fused) return DISPATCH(run_fused_inv, pl, s, beam, xin, inv_wsum, eta, out);
  if (pl->nbatch > 1) return fail(PFBG_ERR_STATE, "batched plans need the fused plane transforms");
  CKRC(cufft_setup(pl));
  CKRC(fft_exec(pl, s, CUFFT_INVERSE));
  return DISPATCH(run_grid2img, pl, s, beam, xin, inv_wsum, eta, out);
}
static int zero_planes(pfbg_plan* pl, cudaStream_t s) {
  if (pl->fused) return DISPATCH(run_zero_window, pl, s);
  CK(cudaMemsetAsync(pl->grid.p, 0, pl->grid.bytes, s));
  return PFBG_OK;
}

// preconditions of pfbg_grid / pfbg_grid_psf / pfbg_degrid / pfbg_hessian; only the Hessian serves a split band
static int check_apply(const pfbg_plan* pl, bool split_ok) {
  if (pl->split_role && !split_ok) return fail(PFBG_ERR_STATE, "plan is part of a band split: only pfbg_hessian / pfbg_split_helper_serve");
  if (!pl->bound) return fail(PFBG_ERR_STATE, "no visibilities bound");
  if (!pl->grid.p) return fail(PFBG_ERR_STATE, "the plan has no plane stack (created with PFBG_PLAN_EXTERNAL_STACK): lend one with pfbg_plan_set_stack");
  return PFBG_OK;
}

extern "C" int pfbg_grid(pfbg_plan* pl, const void* vis, int64_t vis_rs, int64_t vis_cs, const void* wgt,
                         void* dirty, uint32_t flags, void* stream) {
  if (!pl || !dirty) return fail(PFBG_ERR_ARG, "null argument");
  CKRC(check_apply(pl, false));
  if (!vis && pl->nvis > 0) return fail(PFBG_ERR_ARG, "null vis");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = real_bytes(pl);
  const size_t img_bytes = img_elems(pl) * rb;
  pl->n_ev = 0;
  mark(pl, s);
  const void* dvis = vis;
  const void* dwgt = wgt;
  if (!dev && pl->nvis > 0) {
    bool bcast = (vis_rs == 0 && vis_cs == 0);
    if (!bcast && !(vis_cs == 1 && vis_rs == pl->gp.nchan)) return fail(PFBG_ERR_ARG, "host vis must be C-contiguous or a broadcast scalar");
    const size_t vb = bcast ? 2 * rb : (size_t)pl->nvis * 2 * rb;
    CKRC(fetch(pl, pl->vis_stage, vis, vb, false, s, &dvis));
    if (wgt) CKRC(fetch(pl, pl->wgt_stage, wgt, (size_t)pl->nvis * rb, false, s, &dwgt, (vb + 4095) & ~(size_t)4095));
  }
  if (!dwgt && pl->has_wgt) dwgt = pl->wgt.p;
  mark(pl, s);
  CKRC(zero_planes(pl, s));
  CKRC(DISPATCH(run_spread, pl, s, dvis, vis_rs, vis_cs, dwgt, 0, 1));
  mark(pl, s);
  void* dout = dirty;
  if (!dev) { CKRC(dev_alloc(pl, pl->img_out, img_bytes)); dout = pl->img_out.p; }
  CKRC(planes_to_image(pl, s, nullptr, nullptr, 1.0, 0.0, dout));
  mark(pl, s);
  if (!dev) CKRC(d2h_staged(pl, dirty, dout, img_bytes, s));
  mark(pl, s);
  return PFBG_OK;
}

extern "C" int pfbg_grid_psf(pfbg_plan* pl, double x0, double y0, double sign, const void* wgt, void* dirty,
                             uint32_t flags, void* stream) {
  if (!pl || !dirty) return fail(PFBG_ERR_ARG, "null argument");
  CKRC(check_apply(pl, false));
  if (x0 * x0 + y0 * y0 >= 1.0) return fail(PFBG_ERR_ARG, "phase centre outside the unit sphere");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = real_bytes(pl);
  const size_t img_bytes = img_elems(pl) * rb;
  pl->n_ev = 0;
  mark(pl, s);
  const void* dwgt = wgt;
  if (wgt && !dev && pl->nvis > 0) CKRC(fetch(pl, pl->wgt_stage, wgt, (size_t)pl->nvis * rb, false, s, &dwgt));
  if (!dwgt && pl->has_wgt) dwgt = pl->wgt.p;
  if (pl->nvis > 0) {
    CKRC(dev_alloc(pl, pl->vis_stage, (size_t)pl->nvis * 2 * rb));
    const double r2 = x0 * x0 + y0 * y0, nm1_0 = -r2 / (sqrt(1.0 - r2) + 1.0);
    const unsigned grd = (unsigned)((pl->nvis + 255) / 256);
    if (pl->precision == PFBG_F32)
      k_psf_ramp<float><<<grd, 256, 0, s>>>((const double*)pl->uvw.p, (const double*)pl->fscale.p, pl->nvis, pl->gp.nchan, x0, y0, nm1_0, sign, (float2*)pl->vis_stage.p);
    else
      k_psf_ramp<double><<<grd, 256, 0, s>>>((const double*)pl->uvw.p, (const double*)pl->fscale.p, pl->nvis, pl->gp.nchan, x0, y0, nm1_0, sign, (double2*)pl->vis_stage.p);
    LAUNCHED();
  }
  mark(pl, s);
  CKRC(zero_planes(pl, s));
  CKRC(DISPATCH(run_spread, pl, s, pl->vis_stage.p, (int64_t)pl->gp.nchan, (int64_t)1, dwgt, 0, 1));
  mark(pl, s);
  void* dout = dirty;
  if (!dev) { CKRC(dev_alloc(pl, pl->img_out, img_bytes)); dout = pl->img_out.p; }
  CKRC(planes_to_image(pl, s, nullptr, nullptr, 1.0, 0.0, dout));
  mark(pl, s);
  if (!dev) CKRC(d2h_staged(pl, dirty, dout, img_bytes, s));
  mark(pl, s);
  return PFBG_OK;
}

extern "C" int pfbg_degrid(pfbg_plan* pl, const void* dirty, void* vis, const void* wgt, uint32_t flags,
                           void* stream) {
  if (!pl || !dirty) return fail(PFBG_ERR_ARG, "null argument");
  CKRC(check_apply(pl, false));
  if (!vis && pl->nvis > 0) return fail(PFBG_ERR_ARG, "null vis");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = real_bytes(pl);
  const size_t img_bytes = img_elems(pl) * rb;
  const size_t vis_bytes = (size_t)pl->nvis * 2 * rb;
  pl->n_ev = 0;
  mark(pl, s);
  const void* dimg = dirty;
  CKRC(fetch(pl, pl->img_in, dirty, img_bytes, dev, s, &dimg));
  const void* dwgt = nullptr;
  if (flags & PFBG_APPLY_WGT) {
    dwgt = wgt;
    if (wgt && !dev) CKRC(fetch(pl, pl->wgt_stage, wgt, (size_t)pl->nvis * rb, false, s, &dwgt, (img_bytes + 4095) & ~(size_t)4095));
    if (!dwgt && pl->has_wgt) dwgt = pl->wgt.p;
  }
  mark(pl, s);
  CKRC(image_to_planes(pl, s, dimg, nullptr));
  mark(pl, s);
  void* dvis = vis;
  if (!dev && pl->nvis > 0) {
    CKRC(dev_alloc(pl, pl->vis_stage, vis_bytes));
    dvis = pl->vis_stage.p;
    // PFBG_NO_MASK_ZERO with host pointers: the masked samples of the caller's array make the round trip unchanged
    if (pl->has_mask && (flags & PFBG_NO_MASK_ZERO)) CKRC(h2d_staged(pl, dvis, vis, vis_bytes, s));
  }
  if (pl->nvis > 0) {
    const int zeroed = (pl->has_mask && !(flags & PFBG_NO_MASK_ZERO)) ? 1 : 0;
    if (zeroed) CK(cudaMemsetAsync(dvis, 0, vis_bytes, s));
    CKRC(DISPATCH(run_gather, pl, s, dwgt, dvis, nullptr, 1, zeroed));
  }
  mark(pl, s);
  if (!dev && pl->nvis > 0) CKRC(d2h_staged(pl, vis, dvis, vis_bytes, s));
  mark(pl, s);
  return PFBG_OK;
}

extern "C" int pfbg_hessian(pfbg_plan* pl, const void* x, const void* beam, double wsum, double eta, void* out,
                            uint32_t flags, void* stream) {
  if (!pl || !x || !out) return fail(PFBG_ERR_ARG, "null argument");
  CKRC(check_apply(pl, true));
  if (pl->split_role == 2) return fail(PFBG_ERR_STATE, "split helper plans only serve (pfbg_split_helper_serve)");
  if (pl->split_role == 1 && !(flags & PFBG_DEVICE_PTRS)) return fail(PFBG_ERR_STATE, "split plans take device pointers");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  const bool dev = flags & PFBG_DEVICE_PTRS;
  const size_t rb = real_bytes(pl);
  const size_t img_bytes = img_elems(pl) * rb;
  pl->n_ev = 0;
  mark(pl, s);
  const void *dx = x, *dbeam = beam;
  const bool pin_in = flags & PFBG_PINNED_IN, pin_out = flags & PFBG_PINNED_OUT;
  CKRC(fetch(pl, pl->img_in, x, img_bytes, dev, s, &dx, 0, pin_in));
  if (beam) {
    if (!dev && (flags & PFBG_BEAM_CACHED) && pl->beam_on_device && pl->img_beam.bytes >= img_bytes) {
      dbeam = pl->img_beam.p;  // same beam as the previous call (per-band constant, operators/hessian.py:91-98)
    } else {
      CKRC(fetch(pl, pl->img_beam, beam, img_bytes, dev, s, &dbeam, (img_bytes + 4095) & ~(size_t)4095));
      pl->beam_on_device = !dev;
    }
  }
  CKRC(dev_alloc(pl, pl->mvis, (size_t)(pl->nactive ? pl->nactive : 1) * 2 * rb));
  const void* dwgt = pl->has_wgt ? pl->wgt.p : nullptr;
  if (!dev) {
    // `if not x.any(): return zeros` (operators/hessian.py:47-48), checked on the device copy
    const int64_t npix = (int64_t)img_elems(pl);
    CK(cudaMemsetAsync(pl->flag.p, 0, 4, s));
    if (pl->precision == PFBG_F32)
      k_any_nonzero<float><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>((const float*)dx, npix, (int*)pl->flag.p);
    else
      k_any_nonzero<double><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>((const double*)dx, npix, (int*)pl->flag.p);
    LAUNCHED();
    int nz = 1;
    CK(cudaMemcpyAsync(&nz, pl->flag.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (!nz) {
      memset(out, 0, img_bytes);
      return PFBG_OK;
    }
  }
  const bool owner = pl->split_role == 1;
  if (owner) {  // publish x [* beam] to the helper GPU that transforms the last split_nq planes
    const int64_t npix = (int64_t)pl->gp.nx * pl->gp.ny;
    ++pl->split_step;
    if (pl->precision == PFBG_F32)
      k_share_image<float><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>(npix, (const float*)dx, (const float*)dbeam, (float*)pl->xshare.p);
    else
      k_share_image<double><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>(npix, (const double*)dx, (const double*)dbeam, (double*)pl->xshare.p);
    LAUNCHED();
    CKRC(split_signal(pl, s, 0));  // X_READY
  }
  mark(pl, s);
  // R (beam * x): pad + screen, FFT, gather (phase factors cancel against the adjoint)
  CKRC(image_to_planes(pl, s, dx, dbeam));
  if (owner) CKRC(split_wait(pl, s, 0));  // FWD_ARRIVED: the helper's planes are in the stack
  mark(pl, s);
  CKRC(DISPATCH(run_gather, pl, s, nullptr, nullptr, pl->mvis.p, 0));
  mark(pl, s);
  // R^H W: spread (weights applied on load), FFT, screen + crop + epilogue
  CKRC(zero_planes(pl, s));
  mark(pl, s);
  CKRC(DISPATCH(run_spread, pl, s, pl->mvis.p, 0, 0, dwgt, 1, 0));
  if (owner) CKRC(split_signal(pl, s, 1));  // GRID_DONE: the helper may fetch its planes
  mark(pl, s);
  void* dout = out;
  if (!dev) { CKRC(dev_alloc(pl, pl->img_out, img_bytes)); dout = pl->img_out.p; }
  CKRC(planes_to_image(pl, s, dbeam, eta != 0.0 ? dx : nullptr, wsum > 0.0 ? 1.0 / wsum : 1.0, eta, dout));
  mark(pl, s);
  if (!dev && pin_out) {
    CK(cudaMemcpyAsync(out, dout, img_bytes, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  } else if (!dev) CKRC(d2h_staged(pl, out, dout, img_bytes, s));
  mark(pl, s);
  return PFBG_OK;
}


// ---------------------------------------------------------------------------
// Band split across two GPUs (one process per GPU; SURVEY §8e, BASELINE north_star "bands are partitioned across
// the 8 GPUs"): when a job has as many bands as GPUs the heaviest band bounds the step (band 7 of C2 costs 1.7x
// band 0: more w-planes, a larger active uv window).  The plane transforms are the divisible half of a Hessian
// apply, so the owner of a heavy band hands the LAST nq planes to a helper GPU:
//   forward : helper reads x [* beam] from the owner, runs k_rows_fwd + k_cols_fwd on its planes; the column pass
//             stores the transformed columns straight into the owner's plane stack (peer-mapped, NVLink);
//   inverse : the helper's k_cols_inv loads the gridded columns of its planes from the owner's stack over NVLink,
//             k_rows_inv accumulates them into a local fp64 image, which one peer copy hands to the owner, whose
//             epilogue adds it to its own accumulator.
// The two processes never talk on the host after set-up: four flags in device memory (each polled by its owner,
// written by the peer after a system-scope fence) order the kernels of the two streams.
//   helper mailbox: [0] X_READY (owner -> helper), [1] GRID_DONE;  owner mailbox: [0] FWD_ARRIVED, [1] PARTIAL_ARRIVED
// Buffers cross the process boundary as CUDA IPC handles (pfbg_ipc_blob); within one process (tests) the raw
// pointer is used.
// ---------------------------------------------------------------------------
#include <unistd.h>
#include <map>
#include <mutex>

struct IpcBlob {
  cudaIpcMemHandle_t h;   // 64 bytes
  uint64_t offset;        // of the pointer inside the allocation the handle names
  uint64_t raw;           // the pointer itself (valid inside the exporting process)
  int64_t pid;
  int32_t device;
  int32_t pad;
};
static_assert(sizeof(IpcBlob) == PFBG_IPC_BLOB_BYTES, "pfbg_ipc_blob size");

static std::mutex g_ipc_mu;
static std::map<std::string, void*> g_ipc_open;  // handle bytes -> mapped base (a handle opens once per process)

static int ipc_export(const void* ptr, IpcBlob* b) {
  memset(b, 0, sizeof *b);
  // cudaMalloc may carve small allocations out of a larger block: the handle names the block
  typedef int (*range_fn)(unsigned long long*, size_t*, unsigned long long);
  static range_fn get_range = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &f, cudaEnableDefault, &q) != cudaSuccess) f = nullptr;
    return (range_fn)f;
  }();
  unsigned long long base = (unsigned long long)(uintptr_t)ptr;
  size_t size = 0;
  if (get_range && get_range(&base, &size, (unsigned long long)(uintptr_t)ptr) != 0) base = (unsigned long long)(uintptr_t)ptr;
  CK(cudaIpcGetMemHandle(&b->h, (void*)(uintptr_t)base));
  b->offset = (uint64_t)((uintptr_t)ptr - (uintptr_t)base);
  b->raw = (uint64_t)(uintptr_t)ptr;
  b->pid = (int64_t)getpid();
  int dev = 0;
  CK(cudaGetDevice(&dev));
  b->device = dev;
  return PFBG_OK;
}

static int ipc_open(const IpcBlob* b, int my_device, void** out) {
  *out = nullptr;
  if (b->pid == (int64_t)getpid()) {  // same process: the pointer is valid as it is
    if (b->device != my_device) {
      int can = 0;
      CK(cudaDeviceCanAccessPeer(&can, my_device, b->device));
      if (!can) return fail(PFBG_ERR_STATE, "device %d cannot access device %d", my_device, b->device);
      cudaError_t e = cudaDeviceEnablePeerAccess(b->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(PFBG_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
      cudaGetLastError();
    }
    *out = (void*)(uintptr_t)b->raw;
    return PFBG_OK;
  }
  std::lock_guard<std::mutex> lk(g_ipc_mu);
  const std::string key((const char*)&b->h, sizeof b->h);
  auto it = g_ipc_open.find(key);
  void* base = nullptr;
  if (it != g_ipc_open.end()) base = it->second;
  else {
    cudaError_t e = cudaIpcOpenMemHandle(&base, b->h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(PFBG_ERR_CUDA, "cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e)); }
    g_ipc_open[key] = base;
  }
  *out = (char*)base + b->offset;
  return PFBG_OK;
}

extern "C" int pfbg_ipc_export(const void* dev_ptr, pfbg_ipc_blob* blob) {
  if (!dev_ptr || !blob) return fail(PFBG_ERR_ARG, "null argument");
  return ipc_export(dev_ptr, (IpcBlob*)blob);
}
extern "C" int pfbg_ipc_open(int32_t device, const pfbg_ipc_blob* blob, void** dev_ptr) {
  if (!blob || !dev_ptr) return fail(PFBG_ERR_ARG, "null argument");
  CK(cudaSetDevice(device));
  return ipc_open((const IpcBlob*)blob, device, dev_ptr);
}
extern "C" int pfbg_ipc_close_all(void) {
  std::lock_guard<std::mutex> lk(g_ipc_mu);
  for (auto& kv : g_ipc_open) cudaIpcCloseMemHandle(kv.second);
  g_ipc_open.clear();
  cudaGetLastError();
  return PFBG_OK;
}

static const size_t kMailboxBytes = (size_t)2 << 20;  // its own allocation block
static const unsigned long long kSplitTimeoutNs = 20ull * 1000 * 1000 * 1000;

// CUDA loads kernels lazily and the first launch of a kernel synchronises the context: a launch issued while a flag
// wait spins on the same device would not start before the wait gives up.  Every kernel a split apply uses is
// therefore launched once at set-up, before any wait can spin.
static int split_warm_flags(pfbg_plan* pl) {
  unsigned long long* scratch = (unsigned long long*)pl->mailbox.p + 32;  // beyond the live slots and the time-out word
  k_flag_signal<<<1, 1>>>(scratch, 0ull);
  k_flag_wait<<<1, 1>>>(scratch, 0ull, 1000ull, (int*)(scratch + 1));
  if (pl->precision == PFBG_F32) k_share_image<float><<<1, 32>>>(0, nullptr, nullptr, nullptr);
  else k_share_image<double><<<1, 32>>>(0, nullptr, nullptr, nullptr);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return PFBG_OK;
}

static int split_signal(pfbg_plan* pl, cudaStream_t s, int slot) {
  k_flag_signal<<<1, 1, 0, s>>>(pl->peer_mailbox + slot, pl->split_step);
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}
static int split_wait(pfbg_plan* pl, cudaStream_t s, int slot) {
  k_flag_wait<<<1, 1, 0, s>>>((const unsigned long long*)pl->mailbox.p + slot, pl->split_step, kSplitTimeoutNs,
                              (int*)((char*)pl->mailbox.p + 64));
  LAUNCHED();
  CK(cudaGetLastError());
  return PFBG_OK;
}

extern "C" int pfbg_split_owner_init(pfbg_plan* pl, int32_t nq, pfbg_ipc_blob* blobs4) {
  if (!pl || !blobs4) return fail(PFBG_ERR_ARG, "null argument");
  if (!pl->fused) return fail(PFBG_ERR_STATE, "band split needs the fused plane transforms");
  if (pl->nbatch > 1) return fail(PFBG_ERR_STATE, "batched plans cannot be split");
  if (pl->split_role) return fail(PFBG_ERR_STATE, "plan is already part of a band split");
  if (nq < 1 || nq >= pl->gp.nplanes) return fail(PFBG_ERR_ARG, "nq=%d outside [1, nplanes)", nq);
  CK(cudaSetDevice(pl->device));
  const size_t npix = (size_t)pl->gp.nx * pl->gp.ny;
  CKRC(dev_alloc(pl, pl->xshare, npix * real_bytes(pl)));
  CKRC(dev_alloc(pl, pl->partial, npix * sizeof(double)));
  CKRC(dev_alloc(pl, pl->mailbox, kMailboxBytes));
  CK(cudaMemset(pl->mailbox.p, 0, 4096));
  CK(cudaMemset(pl->partial.p, 0, npix * sizeof(double)));
  IpcBlob* b = (IpcBlob*)blobs4;
  CKRC(ipc_export(pl->grid.p, &b[0]));
  CKRC(ipc_export(pl->xshare.p, &b[1]));
  CKRC(ipc_export(pl->partial.p, &b[2]));
  CKRC(ipc_export(pl->mailbox.p, &b[3]));
  pl->split_nq = nq;
  pl->split_step = 0;
  return PFBG_OK;
}

extern "C" int pfbg_split_owner_connect(pfbg_plan* pl, const pfbg_ipc_blob* helper_mailbox) {
  if (!pl || !helper_mailbox) return fail(PFBG_ERR_ARG, "null argument");
  if (pl->split_nq < 1 || pl->split_role) return fail(PFBG_ERR_STATE, "pfbg_split_owner_init first");
  CK(cudaSetDevice(pl->device));
  void* p = nullptr;
  CKRC(ipc_open((const IpcBlob*)helper_mailbox, pl->device, &p));
  pl->peer_mailbox = (unsigned long long*)p;
  CKRC(split_warm_flags(pl));
  if (pl->bound) {  // one whole (unsplit) apply on the shared image: loads every kernel of the path
    CK(cudaMemset(pl->xshare.p, 0, (size_t)pl->gp.nx * pl->gp.ny * real_bytes(pl)));
    CKRC(pfbg_hessian(pl, pl->xshare.p, nullptr, 0.0, 0.0, pl->xshare.p, PFBG_DEVICE_PTRS, nullptr));
    CK(cudaDeviceSynchronize());
  }
  pl->split_role = 1;
  return PFBG_OK;
}

extern "C" int pfbg_split_helper_create(const pfbg_plan_desc* d, int32_t nq, const int32_t* window4,
                                        const pfbg_ipc_blob* owner_blobs4, pfbg_plan** out,
                                        pfbg_ipc_blob* mailbox_out) {
  if (!d || !window4 || !owner_blobs4 || !out || !mailbox_out) return fail(PFBG_ERR_ARG, "null argument");
  if (nq < 1 || nq >= d->nplanes) return fail(PFBG_ERR_ARG, "nq=%d outside [1, nplanes)", nq);
  pfbg_plan* pl = nullptr;
  CKRC(plan_create_impl(d, nq, &pl));
  auto bail = [&](int rc) { pfbg_plan_destroy(pl); return rc; };
  if (!pl->fused) { fail(PFBG_ERR_STATE, "band split needs the fused plane transforms"); return bail(PFBG_ERR_STATE); }
  FusedTabs& ft = pl->ftabs;
  ft.a_lo = window4[0]; ft.a_len = window4[1]; ft.b_lo = window4[2]; ft.b_len = window4[3];
  if (ft.a_lo < 0 || ft.a_len < 1 || ft.a_lo + 0 >= pl->gp.nu || ft.a_len > pl->gp.nu || ft.b_lo < 0 || ft.b_len < 1 ||
      ft.b_lo >= pl->gp.nv || ft.b_len > pl->gp.nv || (ft.b_len % pl->col_c)) {
    fail(PFBG_ERR_ARG, "bad active window");
    return bail(PFBG_ERR_ARG);
  }
  int rc;
  const size_t npix = (size_t)pl->gp.nx * pl->gp.ny;
  if ((rc = dev_alloc(pl, pl->x_local, npix * real_bytes(pl))) || (rc = dev_alloc(pl, pl->mailbox, kMailboxBytes))) return bail(rc);
  if (cudaMemset(pl->mailbox.p, 0, 4096) != cudaSuccess) { fail(PFBG_ERR_CUDA, "memset failed"); return bail(PFBG_ERR_CUDA); }
  const IpcBlob* b = (const IpcBlob*)owner_blobs4;
  void* p[4] = {};
  for (int i = 0; i < 4; ++i)
    if ((rc = ipc_open(&b[i], pl->device, &p[i]))) return bail(rc);
  pl->peer_grid = p[0]; pl->peer_xshare = p[1]; pl->peer_partial = p[2]; pl->peer_mailbox = (unsigned long long*)p[3];
  if ((rc = ipc_export(pl->mailbox.p, (IpcBlob*)mailbox_out))) return bail(rc);
  pl->split_role = 2;
  pl->split_nq = nq;
  pl->split_step = 0;
  pl->bound = false;
  // dry run on the local stack (see split_warm_flags): transforms of the helper's planes, the peer copy of the image
  if ((rc = split_warm_flags(pl))) return bail(rc);
  {
    const int q0 = pl->gp.nplanes - nq;
    cudaError_t e = cudaMemcpy(pl->x_local.p, pl->peer_xshare, npix * real_bytes(pl), cudaMemcpyDefault);
    if (e != cudaSuccess) { fail(PFBG_ERR_CUDA, "peer copy from the owner failed: %s", cudaGetErrorString(e)); return bail(PFBG_ERR_CUDA); }
    cudaMemset(pl->x_local.p, 0, npix * real_bytes(pl));
    rc = pl->precision == PFBG_F32 ? run_fused_fwd<float>(pl, 0, pl->x_local.p, nullptr, q0, nq, nullptr)
                                   : run_fused_fwd<double>(pl, 0, pl->x_local.p, nullptr, q0, nq, nullptr);
    if (!rc) rc = pl->precision == PFBG_F32 ? run_fused_inv_acc<float>(pl, 0, q0, nq, nullptr)
                                            : run_fused_inv_acc<double>(pl, 0, q0, nq, nullptr);
    if (rc) return bail(rc);
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { fail(PFBG_ERR_CUDA, "helper dry run failed: %s", cudaGetErrorString(e)); return bail(PFBG_ERR_CUDA); }
  }
  *out = pl;
  return PFBG_OK;
}

// One Hessian apply worth of helper work, enqueued on `stream` (asynchronous; it waits on the owner's flags on the
// device).  Must be called once per pfbg_hessian call of the owner, in the same order.
extern "C" int pfbg_split_helper_serve(pfbg_plan* pl, void* stream) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  if (pl->split_role != 2) return fail(PFBG_ERR_STATE, "not a split helper");
  CK(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  const GParams& g = pl->gp;
  const int nq = pl->split_nq, q0 = g.nplanes - nq;
  const size_t npix = (size_t)g.nx * g.ny;
  ++pl->split_step;
  pl->n_ev = 0;
  mark(pl, s);
  CKRC(split_wait(pl, s, 0));  // X_READY
  mark(pl, s);
  CK(cudaMemcpyAsync(pl->x_local.p, pl->peer_xshare, npix * real_bytes(pl), cudaMemcpyDefault, s));
  if (pl->precision == PFBG_F32) CKRC(run_fused_fwd<float>(pl, s, pl->x_local.p, nullptr, q0, nq, pl->peer_grid));
  else CKRC(run_fused_fwd<double>(pl, s, pl->x_local.p, nullptr, q0, nq, pl->peer_grid));
  CKRC(split_signal(pl, s, 0));  // FWD_ARRIVED
  mark(pl, s);
  CKRC(split_wait(pl, s, 1));  // GRID_DONE
  mark(pl, s);
  if (pl->precision == PFBG_F32) CKRC(run_fused_inv_acc<float>(pl, s, q0, nq, pl->peer_grid));
  else CKRC(run_fused_inv_acc<double>(pl, s, q0, nq, pl->peer_grid));
  CK(cudaMemcpyAsync(pl->peer_partial, pl->accimg.p, npix * sizeof(double), cudaMemcpyDefault, s));
  CKRC(split_signal(pl, s, 1));  // PARTIAL_ARRIVED
  mark(pl, s);
  return PFBG_OK;
}

// Synchronises `stream` and reports whether any flag wait of this plan gave up (peer gone / calls out of step).
extern "C" int pfbg_split_status(pfbg_plan* pl, void* stream, int32_t* timed_out) {
  if (!pl || !timed_out) return fail(PFBG_ERR_ARG, "null argument");
  *timed_out = 0;
  if (!pl->split_role && pl->split_nq == 0) return PFBG_OK;
  CK(cudaSetDevice(pl->device));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  int t = 0;
  CK(cudaMemcpy(&t, (char*)pl->mailbox.p + 64, 4, cudaMemcpyDeviceToHost));
  *timed_out = t;
  return PFBG_OK;
}

// Leave the split: the owner transforms all its planes again.  Both sides must be idle (synchronise first).
extern "C" int pfbg_split_end(pfbg_plan* pl) {
  if (!pl) return fail(PFBG_ERR_ARG, "null plan");
  CK(cudaSetDevice(pl->device));
  CK(cudaDeviceSynchronize());
  if (pl->split_role == 2) return fail(PFBG_ERR_STATE, "destroy a helper plan instead");
  pl->split_role = 0;
  pl->split_nq = 0;
  pl->peer_mailbox = nullptr;
  return PFBG_OK;
}

// unit-test hook: the lean fp64 ES tap of the DMMA run kernels (runs_mma.cuh) at n positions x in [-1, 1]
__global__ void k_debug_es_fast64(const double* __restrict__ x, double beta, int64_t n, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = es_fast64(x[i], beta);
}
extern "C" int pfbg_debug_es_fast64(int32_t device, int64_t n, const double* x, double beta, double* out) {
  if (!x || !out || n < 1) return fail(PFBG_ERR_ARG, "bad argument");
  CK(cudaSetDevice(device));
  double *dx = nullptr, *dout = nullptr;
  CK(cudaMalloc(&dx, (size_t)n * 8));
  cudaError_t e = cudaMalloc(&dout, (size_t)n * 8);
  if (e == cudaSuccess) e = cudaMemcpy(dx, x, (size_t)n * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    k_debug_es_fast64<<<(unsigned)((n + 255) / 256), 256>>>(dx, beta, n, dout);
    LAUNCHED();
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost);
  cudaFree(dx);
  cudaFree(dout);
  if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "debug_es_fast64: %s", cudaGetErrorString(e));
  return PFBG_OK;
}

