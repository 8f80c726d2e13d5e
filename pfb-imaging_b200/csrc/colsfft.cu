// Translation unit of the pair-engine column transforms (cols2.cuh): tensor-map encoding, launch, and the unit-test
// hooks of both shared-memory FFT engines (fft.cuh, fft2.cuh).
#include <cuda.h>
#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include "cols2.cuh"
#include "fft_host.h"
#include "host.h"
#include "rows2.cuh"

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

// one block of four columns (two column pairs), 8 mbarrier slots, the two-level twiddle table, the u16 position table
static size_t cols2_smem(int nu) { return (size_t)nu * 32 + 64 + (size_t)((nu + 63) / 64 + 64) * 8 + (size_t)nu * 2; }

bool cols2_supported(int nu, int nv, int nx, const FftDesc& du) {
  if (nu > 65535) return false;
  if (!p2_dense_ok(du, 2)) return false;
  if (cols2_smem(nu) > kMaxSmem) return false;
  if ((nx / 2) % COLS2_BOX_SMALL || nu % COLS2_BOX_SMALL || nv % 32 || nx % 2) return false;
  return encode_fn() != nullptr;
}

// (2 nv floats, rows) view of the plane stack, boxes of 8 floats (four columns = one 32-byte sector per row) x `box_rows` rows, dense in shared
// memory (a 128-byte hardware swizzle of 16-byte-wide boxes faults on B200, so the first FFT stage swizzles instead)
static bool encode_map(CUtensorMap* m, const float2* stack, int nv, int64_t rows, int box_rows) {
  const cuuint64_t gdim[2] = {(cuuint64_t)2 * nv, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)nv * 8};
  const cuuint32_t box[2] = {8, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)stack, gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t cols2_launch(const Cols2Args& a, const float2* stack, int stack_planes, float2* out, cudaStream_t s,
                         const char** what) {
  static std::atomic<int> attr_done{0};
  *what = "";
  if (a.nq <= 0 || a.b_len <= 0) return cudaSuccess;
  alignas(64) CUtensorMap mbig, msmall;
  const int64_t rows = (int64_t)stack_planes * a.nu;
  if (!encode_map(&mbig, stack, a.nv, rows, COLS2_BOX_BIG) || !encode_map(&msmall, stack, a.nv, rows, COLS2_BOX_SMALL)) {
    *what = "cuTensorMapEncodeTiled";
    return cudaErrorInvalidValue;
  }
  int dev = 0, nsm = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) { *what = "device query"; return e; }
  if (!(attr_done.load() & (1 << (dev & 31)))) {
    e = cudaFuncSetAttribute(k_cols2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
    if (e != cudaSuccess) { *what = "cudaFuncSetAttribute(k_cols2)"; return e; }
    attr_done.fetch_or(1 << (dev & 31));
  }
  const int64_t nitems = (int64_t)a.nq * (a.b_len / 4);
  const int grid = (int)(nitems < nsm ? nitems : nsm);
  k_cols2<<<grid, COLS2_THREADS, cols2_smem(a.nu), s>>>(mbig, msmall, a, out);
  *what = "k_cols2 launch";
  return cudaGetLastError();
}

// ---- engine unit test: natural order in and out, NP pair elements per index --------------------------------------
// in / out: (batch, 2 NP, n) complex64
template <int NP>
__global__ void __launch_bounds__(256) k_fft2_debug(FftDesc d, const float2* __restrict__ tw, const int* __restrict__ rev,
                                                     const float2* __restrict__ in, float2* __restrict__ out, int inverse,
                                                     int aos) {
  extern __shared__ __align__(1024) unsigned char smem_raw1k[];
  unsigned char* smem_raw = smem_raw1k;
  float4* s = reinterpret_cast<float4*>(smem_raw);
  const int N = d.n, tid = threadIdx.x, nthr = blockDim.x;
  const float2* src = in + (size_t)blockIdx.x * 2 * NP * N;
  float2* dst = out + (size_t)blockIdx.x * 2 * NP * N;
  for (int e = tid; e < N * NP; e += nthr) {
    const int p = e % NP;
    const int n = aos == 2 ? rev[e / NP] : e / NP;  // DIT: position e / NP holds input rev[e / NP]
    const float2 v0 = src[(size_t)(2 * p) * N + n], v1 = src[(size_t)(2 * p + 1) * N + n];
    float4 v;
    if (aos == 1) v = make_float4(v0.x, v0.y, v1.x, v1.y);
    else if (!inverse) v = make_float4(v0.x, v1.x, v0.y, v1.y);
    else v = make_float4(v0.y, v1.y, v0.x, v1.x);
    s[aos == 1 ? e : sw2(e)] = v;
  }
  const P2Tw twt = p2_tw_fill(reinterpret_cast<float2*>(s + (size_t)N * NP), tw, N, tid, nthr);
  __syncthreads();
  if (aos == 2) p2_fft_dit<NP>(s, twt, d, tid, nthr);
  else p2_fft_dif<NP>(s, twt, d, aos ? (inverse ? P2_IN_AOS_SWAP : P2_IN_AOS) : P2_IN_PAIR, tid, nthr);
  for (int e = tid; e < N * NP; e += nthr) {
    const int pos = e / NP, p = e % NP;
    const float4 v = s[sw2(e)];
    const int k = aos == 2 ? pos : rev[pos];
    float2 o0, o1;
    if (!inverse) { o0 = make_float2(v.x, v.z); o1 = make_float2(v.y, v.w); }
    else { o0 = make_float2(v.z, v.x); o1 = make_float2(v.w, v.y); }
    dst[(size_t)(2 * p) * N + k] = o0;
    dst[(size_t)(2 * p + 1) * N + k] = o1;
  }
}

static cudaError_t fft2_debug_launch(const FftDesc& d, int np, const float2* tw, const int* rev, const float2* in,
                                     float2* out, int batch, int inverse, int aos) {
  const size_t sm = (size_t)d.n * np * 16 + (size_t)((d.n + 63) / 64 + 64) * 8;
  if (sm > kMaxSmem || (np != 1 && np != 2 && np != 4)) return cudaErrorInvalidValue;
  if (aos == 1 && !p2_dense_ok(d, np)) return cudaErrorInvalidValue;
  cudaError_t e;
#define FFT2_DEBUG_CASE(NPV)                                                                                          \
  e = cudaFuncSetAttribute(k_fft2_debug<NPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);       \
  if (e != cudaSuccess) return e;                                                                                      \
  k_fft2_debug<NPV><<<batch, 256, sm>>>(d, tw, rev, in, out, inverse, aos);
  if (np == 1) { FFT2_DEBUG_CASE(1) }
  else if (np == 2) { FFT2_DEBUG_CASE(2) }
  else { FFT2_DEBUG_CASE(4) }
#undef FFT2_DEBUG_CASE
  return cudaGetLastError();
}

extern "C" int pfbg_debug_fft2(int32_t device, int32_t n, int32_t np, int32_t batch, const void* in, void* out,
                               int32_t inverse, int32_t aos) {
  if (!in || !out || n < 2 || batch < 1) return fail(PFBG_ERR_ARG, "bad argument");
  CK(cudaSetDevice(device));
  FftDesc d;
  if (!factorize(n, d, 16)) return fail(PFBG_ERR_ARG, "n=%d is not 2^a 3^b 5^c 7^d 11^e", n);
  const std::vector<cx2<float>> tw = twiddles<float>(n);
  std::vector<int> rev, pos;
  digit_tables(d, rev, pos);
  const size_t bytes = (size_t)n * 8 * 2 * np * batch;
  TmpBufs t;
  void *dtw, *drev, *din, *dout;
  CKRC(t.get(&dtw, tw.data(), (size_t)n * 8, false, true, 0));
  CKRC(t.get(&drev, rev.data(), (size_t)n * 4, false, true, 0));
  CKRC(t.get(&din, in, bytes, false, true, 0));
  CKRC(t.get(&dout, out, bytes, false, false, 0));
  cudaError_t e = fft2_debug_launch(d, np, (const float2*)dtw, (const int*)drev, (const float2*)din, (float2*)dout, batch,
                                    inverse, aos);
  if (e != cudaSuccess) return fail(PFBG_ERR_CUDA, "fft2 debug launch: %s", cudaGetErrorString(e));
  LAUNCHED();
  CK(cudaMemcpy(out, dout, bytes, cudaMemcpyDeviceToHost));
  return PFBG_OK;
}

// ---- engine unit test of the one-plane FFT (fft.cuh) ---------------------------------------------------------------
template <typename T>
static int debug_fft_t(int n, int batch, const void* in, void* out, int mode, int inverse) {
  FftDesc d;
  if (!factorize(n, d, sizeof(T) == 4 ? 16 : 8)) return fail(PFBG_ERR_ARG, "n=%d is not 2^a 3^b 5^c 7^d 11^e", n);
  size_t bytes = (size_t)n * sizeof(cx2<T>);
  if (fft_smem_bytes<T>(n) > kMaxSmem) return fail(PFBG_ERR_ARG, "n=%d does not fit shared memory", n);
  const std::vector<cx2<T>> tw = twiddles<T>(n);
  std::vector<int> rev, pos;
  digit_tables(d, rev, pos);
  TmpBufs t;
  void *dtw, *drev, *dpos, *din, *dout;
  CKRC(t.get(&dtw, tw.data(), bytes, false, true, 0));
  CKRC(t.get(&drev, rev.data(), (size_t)n * 4, false, true, 0));
  CKRC(t.get(&dpos, pos.data(), (size_t)n * 4, false, true, 0));
  CKRC(t.get(&din, in, bytes * batch, false, true, 0));
  CKRC(t.get(&dout, out, bytes * batch, false, false, 0));
  CK(cudaFuncSetAttribute(k_fft_debug<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
  k_fft_debug<T><<<batch, 256, fft_smem_bytes<T>(n)>>>(d, (const cx2<T>*)dtw, (const int*)drev, (const int*)dpos, (const cx2<T>*)din,
                                        (cx2<T>*)dout, mode, inverse);
  LAUNCHED();
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, dout, bytes * batch, cudaMemcpyDeviceToHost));
  return PFBG_OK;
}

extern "C" int pfbg_debug_fft1d(int32_t precision, int32_t device, int32_t n, int32_t batch, const void* in,
                                void* out, int32_t mode, int32_t inverse) {
  if (!in || !out || n < 2 || batch < 1) return fail(PFBG_ERR_ARG, "bad argument");
  CK(cudaSetDevice(device));
  return precision == PFBG_F32 ? debug_fft_t<float>(n, batch, in, out, mode, inverse)
                               : debug_fft_t<double>(n, batch, in, out, mode, inverse);
}

// ---- row passes on the pair engine (rows2.cuh) --------------------------------------------------------------------
static size_t rows2_smem(int nv) { return (size_t)nv * 16 + (size_t)((nv + 63) / 64 + 64) * 8; }
static int rows2_threads(int nv) {
  const int t = ((nv / 16 + 1) / 2 + 31) & ~31;  // two butterflies of the widest stage per thread
  return t < 32 ? 32 : (t > ROWS2_THREADS ? ROWS2_THREADS : t);
}

bool rows2_supported(int nv) { return nv % 32 == 0 && rows2_smem(nv) <= kMaxSmem; }

template <typename K>
static cudaError_t rows2_attr(K kern) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  return e;
}

cudaError_t rows2_fwd_launch(const GParams& g, const FusedTabs& ft, int nq, bool fast, const float* x, const float* beam,
                             const float* corr, float2* stack_biased, cudaStream_t s) {
  static std::atomic<int> attr_done{0};
  if (nq & 1) return cudaErrorInvalidValue;  // every CTA transforms a full pair of planes
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (!(attr_done.load() & (1 << (dev & 31)))) {
    if ((e = rows2_attr(k_rows2_fwd<false>)) != cudaSuccess || (e = rows2_attr(k_rows2_fwd<true>)) != cudaSuccess) return e;
    attr_done.fetch_or(1 << (dev & 31));
  }
  const dim3 grid(nq / 2, g.nx);
  const int nt = rows2_threads(g.nv);
  const size_t sm = rows2_smem(g.nv);
  if (fast) k_rows2_fwd<true><<<grid, nt, sm, s>>>(g, ft, x, beam, corr, stack_biased);
  else k_rows2_fwd<false><<<grid, nt, sm, s>>>(g, ft, x, beam, corr, stack_biased);
  return cudaGetLastError();
}

cudaError_t rows2_inv_launch(const GParams& g, const FusedTabs& ft, int nq, bool fast, const float2* stack_biased,
                             double* accimg, cudaStream_t s) {
  static std::atomic<int> attr_done{0};
  if (nq & 1) return cudaErrorInvalidValue;  // every CTA transforms a full pair of planes
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (!(attr_done.load() & (1 << (dev & 31)))) {
    if ((e = rows2_attr(k_rows2_inv<false>)) != cudaSuccess || (e = rows2_attr(k_rows2_inv<true>)) != cudaSuccess) return e;
    attr_done.fetch_or(1 << (dev & 31));
  }
  const dim3 grid(nq / 2, g.nx);
  const int nt = rows2_threads(g.nv);
  const size_t sm = rows2_smem(g.nv);
  if (fast) k_rows2_inv<true><<<grid, nt, sm, s>>>(g, ft, stack_biased, accimg);
  else k_rows2_inv<false><<<grid, nt, sm, s>>>(g, ft, stack_biased, accimg);
  return cudaGetLastError();
}
