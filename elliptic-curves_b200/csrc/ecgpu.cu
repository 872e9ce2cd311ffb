// ecgpu.cu — kernels and C ABI of libecgpu.so (see include/ecgpu.h for the contract).
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
// There is no CPU fallback in this file: every compute entry launches sm_100a kernels or fails.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

// This file is compiled once per curve group (-DECG_TU=0..3) so that the groups build in parallel and the kernels of
// the headline curves keep their own translation unit:
//   ECG_TU 0: secp256k1, P-256, P-384 + every extern "C" entry (entries for other curves forward to their group)
//   ECG_TU 1: sm2, brainpoolP256r1/t1, bign-curve256v1 (8 limbs)   ECG_TU 2: brainpoolP384r1/t1 (12 limbs)
//   ECG_TU 3: P-224 (7 limbs), P-192 (6 limbs)                    ECG_TU 4: P-521 (17 limbs, 66-byte records)
// The groups 1-3 run the generic kernels over the generic Montgomery field policy (ecg_fe_mont.cuh).
#ifndef ECG_TU
#define ECG_TU 0
#endif

#include "../../include/ecgpu.h"
#include "ecg_kernels.cuh"
#if ECG_TU == 0 || ECG_TU == 4  // hash to curve: secp256k1, P-256, P-384 (group 0) and P-521 (group 4)
#include "ecg_h2c.cuh"
#endif
#if ECG_TU == 0
#include "ecg_microbench.cuh"
#endif
#if ECG_TU == 1  // SM2 public-key encryption (sm2 only)
#include "ecg_sm2pke.cuh"
#endif
#include "ecg_msm.cuh"

#define ECG_CURVE_COUNT 12
static inline int curve_group(int c) { return c <= 2 ? 0 : c <= 6 ? 1 : c <= 8 ? 2 : c <= 10 ? 3 : 4; }
// an entry point: extern "C" in group 0, an internal (hidden) function ecg_tuN_<name> in the other groups
#define ECG_CAT2(a, b) a##b
#define ECG_CAT(a, b) ECG_CAT2(a, b)
#if ECG_TU == 0
#define ECG_API(name) extern "C" ecg_status name
#else
#define ECG_API(name) __attribute__((visibility("hidden"))) ecg_status ECG_CAT(ECG_CAT(ECG_CAT(ecg_tu, ECG_TU), _), name)
#endif

// ------------------------------------------------------------------------------------------------
// host side
//
// A ctx owns, per device, two "lanes" (stream + grow-only device buffers + status words).  Device-pointer
// mode uses lane 0 only (optionally on the caller's stream).  Host-pointer mode cuts every per-element batch
// into chunks and alternates lanes, so the H2D copy of chunk c+1 and the D2H copy of chunk c-1 overlap the
// kernels of chunk c (PCIe is the only thing between the caller's buffers and the SMs).
enum { B_K = 0, B_P = 1, B_INF = 2, B_JAC = 3, B_SCR = 4, B_OUT = 5, B_OINF = 6, B_AUX = 7, B_A = 8, B_JAC2 = 9, B_TAB = 10, B_MSM = 11, B_FB1 = 12, B_FB2 = 13, B_X = 14, B_V1 = 15, B_V2 = 16, B_V3 = 17, B_V4 = 18, B_V5 = 19, B_V6 = 20, B_COUNT = 21 };
static const size_t HOST_CHUNK = (size_t)1 << 18;  // elements per pipelined chunk in host-pointer mode
static const size_t DEV_CHUNK = (size_t)1 << 22;   // device-pointer mode: bound the temporaries (tables 512-768 B/element)

struct Lane {
  cudaStream_t stream = nullptr;       // owned
  cudaStream_t user_stream = nullptr;  // optional override (lane 0, ecg_ctx_set_stream)
  bool use_user_stream = false;
  void* buf[B_COUNT] = {nullptr};
  size_t cap[B_COUNT] = {0};
  uint32_t* status = nullptr;    // 2 words: error flags, smallest offending index
  uint32_t* h_status = nullptr;  // pinned: 2 status words, then up to 256 bytes for one exported point (h_point())
  std::vector<cudaEvent_t> evs;  // event pairs bracketing the dominant kernel of every chunk of the current call (ecg_timing)
  size_t ev_used = 0;            // events of `evs` recorded by the current call (2 per chunk)
  bool used = false;  // touched by the current call
  cudaStream_t s() const { return use_user_stream ? user_stream : stream; }
  uint8_t* h_point() const { return reinterpret_cast<uint8_t*>(h_status + 2); }
};
struct DevState {
  int dev = 0;
  Lane lane[2];
  uint32_t* fb_table[ECG_CURVE_COUNT] = {nullptr};  // per curve, built lazily (like the reference's LazyLock table)
  int sm_count = 148;
};

struct ecg_ctx {
  std::vector<DevState> devs;
  unsigned flags = 0;
  std::string err;
  size_t err_index = (size_t)-1;
  uint64_t launches = 0;
  bool timing = false;    // ecg_timing_enable
  double dom_ms_sum = 0;  // accumulated device time of the dominant kernel (max over devices per call)
  uint64_t dom_calls = 0;
  bool skew = false;  // set by finish(): the bucket method declined a skewed input (MSM_SKEW_FLAG), the caller repeats per term
  bool devptr() const { return (flags & ECG_FLAG_DEVICE_PTRS) != 0; }
};

#define CU_TRY(ctx, call)                                                                                    \
  do {                                                                                                       \
    cudaError_t e_ = (call);                                                                                 \
    if (e_ != cudaSuccess) {                                                                                 \
      char m_[512];                                                                                          \
      snprintf(m_, sizeof m_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);  \
      (ctx)->err = m_;                                                                                       \
      return e_ == cudaErrorMemoryAllocation ? ECG_ENOMEM : ECG_ECUDA;                                       \
    }                                                                                                        \
  } while (0)
#define ST_TRY(expr)               \
  do {                             \
    ecg_status st_ = (expr);       \
    if (st_ != ECG_OK) return st_; \
  } while (0)
#define LAUNCHED(ctx)                \
  do {                               \
    (ctx)->launches++;               \
    CU_TRY(ctx, cudaGetLastError()); \
  } while (0)
// CUDA events around the dominant kernel of a call, on the launching stream (bench.py's roofline numerator)
// (one pair per chunk: a call cut into several chunks per lane accumulates all of them in finish())
static ecg_status dom_record(ecg_ctx* ctx, Lane& L) {
  if (!ctx->timing) return ECG_OK;
  if (L.ev_used == L.evs.size()) {
    cudaEvent_t e = nullptr;
    CU_TRY(ctx, cudaEventCreate(&e));
    L.evs.push_back(e);
  }
  CU_TRY(ctx, cudaEventRecord(L.evs[L.ev_used], L.s()));
  L.ev_used++;
  return ECG_OK;
}
#define DOM_BEGIN(ctx, L) ST_TRY(dom_record(ctx, L))
#define DOM_END(ctx, L) ST_TRY(dom_record(ctx, L))

static ecg_status ensure(ecg_ctx* ctx, Lane& L, int which, size_t bytes) {
  if (bytes <= L.cap[which]) return ECG_OK;
  if (L.buf[which]) {
    CU_TRY(ctx, cudaStreamSynchronize(L.s()));
    CU_TRY(ctx, cudaFree(L.buf[which]));
  }
  L.buf[which] = nullptr;
  L.cap[which] = 0;
  size_t want = bytes + bytes / 8 + 256;
  CU_TRY(ctx, cudaMalloc(&L.buf[which], want));
  L.cap[which] = want;
  return ECG_OK;
}

#if ECG_TU == 0
extern "C" const char* ecg_version(void) { return "ecgpu 0.3 (sm_100a)"; }

extern "C" ecg_status ecg_ctx_create(const int* device_ids, int n_devices, unsigned flags, ecg_ctx** out) {
  if (!out) return ECG_EINVAL;
  *out = nullptr;
  if (n_devices < 0 || n_devices > 64) return ECG_EINVAL;
  if ((flags & ECG_FLAG_DEVICE_PTRS) && n_devices > 1) return ECG_EINVAL;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) return ECG_ECUDA;  // no CPU fallback, by design
  ecg_ctx* ctx = new ecg_ctx();
  ctx->flags = flags;
  int nd = n_devices > 0 ? n_devices : 1;
  ctx->devs.resize(nd);
  for (int i = 0; i < nd; i++) {
    DevState& d = ctx->devs[i];
    d.dev = (device_ids && n_devices > 0) ? device_ids[i] : 0;
    if (d.dev < 0 || d.dev >= count) {
      ecg_ctx_destroy(ctx);
      return ECG_EINVAL;
    }
    bool ok = cudaSetDevice(d.dev) == cudaSuccess;
    for (int l = 0; ok && l < 2; l++) {
      Lane& L = d.lane[l];
      ok = cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking) == cudaSuccess &&
           cudaMalloc((void**)&L.status, 8) == cudaSuccess && cudaMallocHost((void**)&L.h_status, 8 + 256) == cudaSuccess;
    }
    if (!ok) {
      ecg_ctx_destroy(ctx);
      return ECG_ECUDA;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, d.dev) == cudaSuccess) d.sm_count = prop.multiProcessorCount;
  }
  *out = ctx;
  return ECG_OK;
}

extern "C" void ecg_ctx_destroy(ecg_ctx* ctx) {
  if (!ctx) return;
  for (DevState& d : ctx->devs) {
    cudaSetDevice(d.dev);
    for (int l = 0; l < 2; l++) {
      Lane& L = d.lane[l];
      if (L.stream) {
        cudaStreamSynchronize(L.stream);
        cudaStreamDestroy(L.stream);
      }
      for (int i = 0; i < B_COUNT; i++)
        if (L.buf[i]) cudaFree(L.buf[i]);
      if (L.status) cudaFree(L.status);
      if (L.h_status) cudaFreeHost(L.h_status);
      for (cudaEvent_t e : L.evs) cudaEventDestroy(e);
    }
    for (int i = 0; i < ECG_CURVE_COUNT; i++)
      if (d.fb_table[i]) cudaFree(d.fb_table[i]);
  }
  delete ctx;
}

extern "C" const char* ecg_last_error(const ecg_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
extern "C" size_t ecg_last_error_index(const ecg_ctx* ctx) { return ctx ? ctx->err_index : (size_t)-1; }
extern "C" uint64_t ecg_kernel_launches(const ecg_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" ecg_status ecg_timing_enable(ecg_ctx* ctx, int on) {
  if (!ctx) return ECG_EINVAL;
  ctx->timing = on != 0;
  ctx->dom_ms_sum = 0;
  ctx->dom_calls = 0;
  return ECG_OK;
}
extern "C" ecg_status ecg_timing_read(const ecg_ctx* ctx, double* dominant_kernel_ms_sum, uint64_t* calls) {
  if (!ctx || !dominant_kernel_ms_sum || !calls) return ECG_EINVAL;
  *dominant_kernel_ms_sum = ctx->dom_ms_sum;
  *calls = ctx->dom_calls;
  return ECG_OK;
}

extern "C" ecg_status ecg_ctx_set_stream(ecg_ctx* ctx, void* cuda_stream) {
  if (!ctx) return ECG_EINVAL;
  Lane& L = ctx->devs[0].lane[0];
  L.user_stream = (cudaStream_t)cuda_stream;
  L.use_user_stream = cuda_stream != nullptr;
  return ECG_OK;
}

#endif  // ECG_TU == 0

// Shard [0,n) into contiguous per-device ranges (SURVEY.md section 8(e)).
struct Shard {
  size_t off, cnt;
};
static std::vector<Shard> make_shards(size_t n, size_t ndev) {
  std::vector<Shard> v(ndev);
  size_t base = n / ndev, rem = n % ndev, off = 0;
  for (size_t i = 0; i < ndev; i++) {
    size_t c = base + (i < rem ? 1 : 0);
    v[i] = {off, c};
    off += c;
  }
  return v;
}

// operands of one chunk as seen by the kernels
struct DevPtrs {
  const uint8_t *k = nullptr, *p = nullptr, *inf = nullptr, *a = nullptr;
  uint8_t *out = nullptr, *oinf = nullptr;
};

// Make elements [off, off+cnt) of `src` (stride bytes each) available on the lane: in device-pointer mode that is
// pointer arithmetic, in host mode an async H2D copy into the lane's slot.
static ecg_status stage_in(ecg_ctx* ctx, Lane& L, int slot, const uint8_t* src, size_t off, size_t cnt, size_t stride,
                           const uint8_t** dst) {
  if (!src) {
    *dst = nullptr;
    return ECG_OK;
  }
  if (ctx->devptr()) {
    // the kernels read 32/64/96-byte records with 32-bit loads (ecg_io.cuh load_be32)
    if ((stride % 4 == 0) && (reinterpret_cast<uintptr_t>(src) & 3)) {
      ctx->err = "device pointer not 4-byte aligned";
      return ECG_EINVAL;
    }
    *dst = src + off * stride;
    return ECG_OK;
  }
  ST_TRY(ensure(ctx, L, slot, cnt * stride));
  CU_TRY(ctx, cudaMemcpyAsync(L.buf[slot], src + off * stride, cnt * stride, cudaMemcpyHostToDevice, L.s()));
  *dst = (const uint8_t*)L.buf[slot];
  return ECG_OK;
}
static ecg_status stage_out(ecg_ctx* ctx, Lane& L, size_t off, size_t cnt, uint8_t* out, size_t ostride, uint8_t* oinf,
                            DevPtrs& dp) {
  if (ctx->devptr()) {
    if ((ostride % 4 == 0) && (reinterpret_cast<uintptr_t>(out) & 3)) {
      ctx->err = "device pointer not 4-byte aligned";
      return ECG_EINVAL;
    }
    dp.out = out + off * ostride;
    dp.oinf = oinf ? oinf + off : nullptr;
    if (!dp.oinf) {
      ST_TRY(ensure(ctx, L, B_OINF, cnt));
      dp.oinf = (uint8_t*)L.buf[B_OINF];
    }
    return ECG_OK;
  }
  ST_TRY(ensure(ctx, L, B_OUT, cnt * ostride));
  ST_TRY(ensure(ctx, L, B_OINF, cnt));
  dp.out = (uint8_t*)L.buf[B_OUT];
  dp.oinf = (uint8_t*)L.buf[B_OINF];
  return ECG_OK;
}
static ecg_status copy_back(ecg_ctx* ctx, Lane& L, size_t off, size_t cnt, uint8_t* out, size_t ostride, uint8_t* oinf,
                            const DevPtrs& dp) {
  if (ctx->devptr()) return ECG_OK;
  CU_TRY(ctx, cudaMemcpyAsync(out + off * ostride, dp.out, cnt * ostride, cudaMemcpyDeviceToHost, L.s()));
  if (oinf) CU_TRY(ctx, cudaMemcpyAsync(oinf + off, dp.oinf, cnt, cudaMemcpyDeviceToHost, L.s()));
  return ECG_OK;
}
static ecg_status begin_lane(ecg_ctx* ctx, Lane& L) {
  if (L.used) return ECG_OK;
  CU_TRY(ctx, cudaMemsetAsync(L.status, 0, 4, L.s()));
  CU_TRY(ctx, cudaMemsetAsync(L.status + 1, 0xFF, 4, L.s()));
  L.used = true;
  return ECG_OK;
}
// ECG_FLAG_ZEROIZE: scrub everything the lane holds that was derived from the caller's inputs (stream-ordered, after
// the call's last kernel and copy).  Outputs the caller asked for live in the caller's buffers and are not touched;
// the fixed-base table is public data.
static const int ZEROIZE_SLOTS[] = {B_K, B_A, B_P, B_INF, B_X, B_JAC, B_JAC2, B_SCR, B_TAB, B_MSM, B_FB1, B_FB2, B_AUX,
                                    B_OUT, B_OINF, B_V1, B_V2, B_V3, B_V4, B_V5, B_V6};
static ecg_status zeroize_lane(ecg_ctx* ctx, Lane& L) {
  for (int slot : ZEROIZE_SLOTS)
    if (L.buf[slot]) CU_TRY(ctx, cudaMemsetAsync(L.buf[slot], 0, L.cap[slot], L.s()));
  return ECG_OK;
}

// Wait for every lane touched by this call; fold validation status and kernel timing into the ctx.
static ecg_status finish(ecg_ctx* ctx) {
  ecg_status rc = ECG_OK;
  size_t first = (size_t)-1;
  float dom_ms = 0;
  bool any_timed = false;
  for (DevState& d : ctx->devs) {
    float dev_ms = 0;
    for (int l = 0; l < 2; l++) {
      Lane& L = d.lane[l];
      if (!L.used) continue;
      L.used = false;
      CU_TRY(ctx, cudaSetDevice(d.dev));
      if (ctx->flags & ECG_FLAG_ZEROIZE) ST_TRY(zeroize_lane(ctx, L));
      CU_TRY(ctx, cudaMemcpyAsync(L.h_status, L.status, 8, cudaMemcpyDeviceToHost, L.s()));
      CU_TRY(ctx, cudaStreamSynchronize(L.s()));
      CU_TRY(ctx, cudaGetLastError());
      for (size_t e = 0; e + 1 < L.ev_used; e += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, L.evs[e], L.evs[e + 1]) == cudaSuccess) dev_ms += ms;
        any_timed = true;
      }
      L.ev_used = 0;
      if (L.h_status[0] & ERRF_SKEW) ctx->skew = true;
      if ((L.h_status[0] & (ERRF_SCALAR | ERRF_POINT)) && (size_t)L.h_status[1] < first) {
        first = L.h_status[1];
        rc = (L.h_status[0] & ERRF_POINT) ? ECG_ENOT_ON_CURVE : ECG_ESCALAR_RANGE;
      }
    }
    if (dev_ms > dom_ms) dom_ms = dev_ms;
  }
  if (any_timed) {
    ctx->dom_ms_sum += dom_ms;
    ctx->dom_calls++;
  }
  if (rc != ECG_OK) {
    ctx->err_index = first;
    ctx->err = rc == ECG_ESCALAR_RANGE ? "scalar out of range (>= n)" : "point not on curve / coordinate >= p";
  }
  return rc;
}
// abandon a call after a host-side failure: drain what was enqueued so buffers can be reused
static ecg_status fail(ecg_ctx* ctx, ecg_status rc) {
  std::string saved = ctx->err;
  for (DevState& d : ctx->devs)
    for (int l = 0; l < 2; l++)
      if (d.lane[l].used) {
        cudaSetDevice(d.dev);
        if (ctx->flags & ECG_FLAG_ZEROIZE) (void)zeroize_lane(ctx, d.lane[l]);
        cudaStreamSynchronize(d.lane[l].s());
        d.lane[l].used = false;
        d.lane[l].ev_used = 0;
      }
  ctx->err = saved;
  return rc;
}

static inline unsigned grid_for(size_t n, unsigned block) { return (unsigned)((n + block - 1) / block); }

// bytes per field element / scalar at the ABI (32; 48 for P-384) and 32-bit limbs per field element
static inline size_t flimbs(ecg_curve c) {
  switch ((int)c) {
    case ECG_NISTP384: case ECG_BP384R1: case ECG_BP384T1: return 12;
    case ECG_NISTP224: return 7;
    case ECG_NISTP192: return 6;
    case ECG_NISTP521: return 17;
    default: return 8;
  }
}
// bytes per canonical record at the ABI: 4 per limb, except P-521 (66 bytes in 17 limbs); bytes of one Jacobian point in
// the internal SoA form (three NL-word coordinates)
static inline size_t fbytes(ecg_curve c) { return c == ECG_NISTP521 ? 66 : 4 * flimbs(c); }
static inline size_t jbytes(ecg_curve c) { return 12 * flimbs(c); }
static inline bool curve_le(ecg_curve c) { return c == ECG_BIGNP256; }
// (0 : 1 : 0) as three canonical records in the curve's byte order
static void identity_xyz(uint8_t* z, ecg_curve c) {
  const size_t fb = fbytes(c);
  memset(z, 0, 3 * fb);
  z[curve_le(c) ? fb : 2 * fb - 1] = 1;
}
// ECG_INLINE_LOOPS=0 (environment) keeps the call-based field operations in the one-point-operation-per-iteration
// kernels (fixed-base, bucket accumulation): measurement knob, default = inlined
static bool inline_loops() {
  static const bool v = []() {
    const char* e = getenv("ECG_INLINE_LOOPS");
    return !(e && e[0] == '0');
  }();
  return v;
}
// FOR_CURVE(curve, statement): run the statement with CV bound to the curve's parameter struct; FOR_CURVE_INL: to the
// all-inlined variant of the curve (ecg_curves.cuh) where one exists.  Each translation unit knows its own group.
#if ECG_TU == 0
#define FOR_CURVE_INL(curve, ...)         \
  do {                                    \
    if ((curve) == ECG_SECP256K1) {       \
      typedef CurveK256I CV;              \
      __VA_ARGS__;                        \
    } else if ((curve) == ECG_NISTP256) { \
      typedef CurveP256I CV;              \
      __VA_ARGS__;                        \
    } else {                              \
      typedef CurveP384I CV;              \
      __VA_ARGS__;                        \
    }                                     \
  } while (0)
#define FOR_CURVE(curve, ...)             \
  do {                                    \
    if ((curve) == ECG_SECP256K1) {       \
      typedef CurveK256 CV;               \
      __VA_ARGS__;                        \
    } else if ((curve) == ECG_NISTP256) { \
      typedef CurveP256 CV;               \
      __VA_ARGS__;                        \
    } else {                              \
      typedef CurveP384 CV;               \
      __VA_ARGS__;                        \
    }                                     \
  } while (0)
#elif ECG_TU == 1
#define FOR_CURVE(curve, ...)             \
  do {                                    \
    if ((curve) == ECG_SM2) {             \
      typedef CurveSm2 CV;                \
      __VA_ARGS__;                        \
    } else if ((curve) == ECG_BP256R1) {  \
      typedef CurveBp256r1 CV;            \
      __VA_ARGS__;                        \
    } else if ((curve) == ECG_BP256T1) {  \
      typedef CurveBp256t1 CV;            \
      __VA_ARGS__;                        \
    } else {                              \
      typedef CurveBignP256 CV;           \
      __VA_ARGS__;                        \
    }                                     \
  } while (0)
#define FOR_CURVE_INL FOR_CURVE
#elif ECG_TU == 2
#define FOR_CURVE(curve, ...)             \
  do {                                    \
    if ((curve) == ECG_BP384R1) {         \
      typedef CurveBp384r1 CV;            \
      __VA_ARGS__;                        \
    } else {                              \
      typedef CurveBp384t1 CV;            \
      __VA_ARGS__;                        \
    }                                     \
  } while (0)
#define FOR_CURVE_INL FOR_CURVE
#elif ECG_TU == 3
#define FOR_CURVE(curve, ...)             \
  do {                                    \
    if ((curve) == ECG_NISTP224) {        \
      typedef CurveP224 CV;               \
      __VA_ARGS__;                        \
    } else {                              \
      typedef CurveP192 CV;               \
      __VA_ARGS__;                        \
    }                                     \
  } while (0)
#define FOR_CURVE_INL FOR_CURVE
#else
#define FOR_CURVE(curve, ...) \
  do {                        \
    typedef CurveP521 CV;     \
    __VA_ARGS__;              \
  } while (0)
#define FOR_CURVE_INL FOR_CURVE
#endif

template <class F>
static ecg_status launch_normalize(ecg_ctx* ctx, DevState& d, Lane& L, size_t n, const uint32_t* jac, uint8_t* out, uint8_t* oinf,
                                   bool x_only) {
  ST_TRY(ensure(ctx, L, B_SCR, n * 4 * F::NL));
  // ~32 elements per thread amortise the per-thread inversion, but never leave SMs idle for small batches
  size_t want_threads = std::max<size_t>((n + 31) / 32, std::min<size_t>(n, (size_t)d.sm_count * 256));
  if (x_only)
    normalize_kernel<F, true><<<grid_for(want_threads, 256), 256, 0, L.s()>>>(jac, n, (uint32_t*)L.buf[B_SCR], out, oinf);
  else
    normalize_kernel<F, false><<<grid_for(want_threads, 256), 256, 0, L.s()>>>(jac, n, (uint32_t*)L.buf[B_SCR], out, oinf);
  LAUNCHED(ctx);
  return ECG_OK;
}
static ecg_status launch_norm(ecg_ctx* ctx, DevState& d, Lane& L, ecg_curve curve, size_t n, const uint32_t* jac, uint8_t* out,
                              uint8_t* oinf, bool x_only = false) {
  FOR_CURVE(curve, return launch_normalize<CV::F>(ctx, d, L, n, jac, out, oinf, x_only));
  return ECG_EINVAL;
}

// launch geometry of the variable-base kernels (registers set the occupancy; tables are in global memory)
static const int K_BLOCK = 256, K_MINBLK = 2;  // secp256k1: <= 128 registers -> 16 warps/SM; phase-synchronised inlined body (ecg_kernels.cuh)
static const int KG_BLOCK = 128, KG_MINBLK = 4;  // secp256k1 a*G + b*P kernel: call-based body (mul = call, sqr inlined: OPT 7)
static const int P_BLOCK = 128, P_MINBLK = 5;  // P-256   : <= 96 registers -> 20 warps/SM (Montgomery field: 34.09 vs 34.65 ms at (128,4), tools/kbench.cu)

static const int Q_BLOCK = 128, Q_MINBLK = 3;  // P-384   : 12-limb values, <= 168 registers -> 12 warps/SM
#define Q_TAB_WORDS (8 * 36) /* 8 Jacobian entries x 36 words */

// the curves on the generic Montgomery field (groups 1-3): call-based field operations, 8 Jacobian table entries
static const int X_BLOCK = 128;
template <int NL>
struct XGeom {
  static constexpr int MINBLK = NL > 12 ? 2 : NL > 8 ? 3 : 4;
};
static size_t vb_block(ecg_curve c) { return c == ECG_SECP256K1 ? K_BLOCK : c == ECG_NISTP256 ? P_BLOCK : c == ECG_NISTP384 ? Q_BLOCK : X_BLOCK; }
// (the constant-time secp256k1 kernel runs 128-thread blocks: a table slot sized for 256-thread blocks covers it, since the
//  slot of block b starts at b * BLOCK * words and 128-thread blocks need half as much per block)
static size_t vb_minblk(ecg_curve c) {
  return c == ECG_SECP256K1 ? K_MINBLK : c == ECG_NISTP256 ? P_MINBLK : c == ECG_NISTP384 ? Q_MINBLK : (flimbs(c) > 12 ? 2 : flimbs(c) > 8 ? 3 : 4);
}
static size_t vb_tab_words(ecg_curve c) { return c == ECG_SECP256K1 ? K_TAB_WORDS : 8 * 3 * flimbs(c); }

static size_t wave_elems(const DevState& d, ecg_curve curve) { return (size_t)d.sm_count * vb_minblk(curve) * vb_block(curve); }

// per-block window-table slots for a launch of n elements
static ecg_status ensure_tab(ecg_ctx* ctx, Lane& L, ecg_curve curve, size_t n) {
  size_t block = vb_block(curve);
  size_t words = vb_tab_words(curve);
  size_t blocks = (n + block - 1) / block;
  return ensure(ctx, L, B_TAB, blocks * block * words * 4);
}

// k*P for one chunk -> Jacobian SoA in `jac`; `status` / `base` locate validation errors
static ecg_status launch_varbase(ecg_ctx* ctx, DevState& d, Lane& L, ecg_curve curve, size_t n, const DevPtrs& dp, uint32_t* jac,
                                 uint32_t* status, size_t base) {
  (void)d;
  ST_TRY(ensure_tab(ctx, L, curve, n));
  uint32_t* gtab = (uint32_t*)L.buf[B_TAB];
  DOM_BEGIN(ctx, L);
  if (ctx->flags & ECG_FLAG_CONSTTIME) {  // masked table selects, branch-free sign folding; dp.p == nullptr: P = G
#if ECG_TU == 0
    if (curve == ECG_SECP256K1)
      k256_varbase_ct_kernel<KG_BLOCK, KG_MINBLK><<<grid_for(n, KG_BLOCK), KG_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab, status, base);
    else if (curve == ECG_NISTP256)
      generic_varbase_kernel<CurveP256, P_BLOCK, P_MINBLK, true><<<grid_for(n, P_BLOCK), P_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab, status, base);
    else
      generic_varbase_kernel<CurveP384, Q_BLOCK, Q_MINBLK, true><<<grid_for(n, Q_BLOCK), Q_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab, status, base);
#else
    FOR_CURVE(curve, (generic_varbase_kernel<CV, X_BLOCK, XGeom<CV::F::NL>::MINBLK, true><<<grid_for(n, X_BLOCK), X_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac,
                                                                                                                                gtab, status, base)));
#endif
    LAUNCHED(ctx);
    DOM_END(ctx, L);
    return ECG_OK;
  }
#if ECG_TU == 0
  if (curve == ECG_SECP256K1)
    k256_varbase_kernel<K_BLOCK, K_MINBLK><<<grid_for(n, K_BLOCK), K_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab, status, base);
  else if (curve == ECG_NISTP256)
    generic_varbase_kernel<CurveP256, P_BLOCK, P_MINBLK><<<grid_for(n, P_BLOCK), P_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab, status, base);
  else
    generic_varbase_kernel<CurveP384, Q_BLOCK, Q_MINBLK><<<grid_for(n, Q_BLOCK), Q_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab, status, base);
#else
  FOR_CURVE(curve, (generic_varbase_kernel<CV, X_BLOCK, XGeom<CV::F::NL>::MINBLK><<<grid_for(n, X_BLOCK), X_BLOCK, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, jac, gtab,
                                                                                                                        status, base)));
#endif
  LAUNCHED(ctx);
  DOM_END(ctx, L);
  return ECG_OK;
}

// every curve the hot path serves; curve_256() = the two 256-bit curves the widening entries (verification, SEC1
// decompression, a*G + b*P, field sqrt) are written for
static bool curve_ok(ecg_curve c) { return (int)c >= 0 && (int)c < ECG_CURVE_COUNT && curve_group((int)c) == ECG_TU; }
static bool curve_256(ecg_curve c) { return c == ECG_SECP256K1 || c == ECG_NISTP256; }

// ---- fixed-base table ------------------------------------------------------------------------------
// Built on the device with the variable-base kernel itself: entry (i, j) = ((2j+1) << 16 i mod n) * G.
// Scalars of the fixed-base table entries, (2j + 1) 2^(16 i) mod n, as records in the curve's byte order.  Built by modular
// additions (B_i = 2^(16 i) mod n by doubling; entry j + 1 = entry j + 2 B_i), so that any group order below 2^(32 nl)
// works, however far below (P-521: n < 2^521 in 544-bit limbs).
struct HostMod {
  int nl;
  uint32_t n[19];
  void add(uint32_t* r, const uint32_t* a, const uint32_t* b) const {  // r = a + b mod n, inputs < n
    uint32_t t[19];
    uint64_t c = 0;
    for (int i = 0; i <= nl; i++) {
      c += (uint64_t)(i < nl ? a[i] : 0) + (i < nl ? b[i] : 0);
      t[i] = (uint32_t)c;
      c >>= 32;
    }
    bool ge = true;
    for (int i = nl; i >= 0; i--)
      if (t[i] != n[i]) {
        ge = t[i] > n[i];
        break;
      }
    if (ge) {
      uint64_t bw = 0;
      for (int i = 0; i <= nl; i++) {
        uint64_t d = (uint64_t)t[i] - n[i] - bw;
        t[i] = (uint32_t)d;
        bw = (d >> 63) & 1;
      }
    }
    for (int i = 0; i < nl; i++) r[i] = t[i];
  }
};
static void scalar_record(uint8_t* out, const uint32_t* v, int nl, size_t fb, bool le) {
  for (size_t byte = 0; byte < fb; byte++) {
    uint8_t b = (uint8_t)(v[byte >> 2] >> (8 * (byte & 3)));  // byte of weight 256^byte
    out[le ? byte : fb - 1 - byte] = b;
  }
  (void)nl;
}
static const uint32_t H_K256_N[8] = {0xD0364141u, 0xBFD25E8Cu, 0xAF48A03Bu, 0xBAAEDCE6u, 0xFFFFFFFEu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
static const uint32_t H_P256_N[8] = {0xFC632551u, 0xF3B9CAC2u, 0xA7179E84u, 0xBCE6FAADu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0x00000000u, 0xFFFFFFFFu};
static const uint8_t H_K256_G[64] = {
    0x79, 0xBE, 0x66, 0x7E, 0xF9, 0xDC, 0xBB, 0xAC, 0x55, 0xA0, 0x62, 0x95, 0xCE, 0x87, 0x0B, 0x07, 0x02, 0x9B, 0xFC, 0xDB, 0x2D, 0xCE,
    0x28, 0xD9, 0x59, 0xF2, 0x81, 0x5B, 0x16, 0xF8, 0x17, 0x98, 0x48, 0x3A, 0xDA, 0x77, 0x26, 0xA3, 0xC4, 0x65, 0x5D, 0xA4, 0xFB, 0xFC,
    0x0E, 0x11, 0x08, 0xA8, 0xFD, 0x17, 0xB4, 0x48, 0xA6, 0x85, 0x54, 0x19, 0x9C, 0x47, 0xD0, 0x8F, 0xFB, 0x10, 0xD4, 0xB8};
static const uint8_t H_P256_G[64] = {
    0x6B, 0x17, 0xD1, 0xF2, 0xE1, 0x2C, 0x42, 0x47, 0xF8, 0xBC, 0xE6, 0xE5, 0x63, 0xA4, 0x40, 0xF2, 0x77, 0x03, 0x7D, 0x81, 0x2D, 0xEB,
    0x33, 0xA0, 0xF4, 0xA1, 0x39, 0x45, 0xD8, 0x98, 0xC2, 0x96, 0x4F, 0xE3, 0x42, 0xE2, 0xFE, 0x1A, 0x7F, 0x9B, 0x8E, 0xE7, 0xEB, 0x4A,
    0x7C, 0x0F, 0x9E, 0x16, 0x2B, 0xCE, 0x33, 0x57, 0x6B, 0x31, 0x5E, 0xCE, 0xCB, 0xB6, 0x40, 0x68, 0x37, 0xBF, 0x51, 0xF5};

static const uint32_t H_P384_N[12] = {0xCCC52973u, 0xECEC196Au, 0x48B0A77Au, 0x581A0DB2u, 0xF4372DDFu, 0xC7634D81u,
                                      0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
static const uint8_t H_P384_G[96] = {
    0xAA, 0x87, 0xCA, 0x22, 0xBE, 0x8B, 0x05, 0x37, 0x8E, 0xB1, 0xC7, 0x1E, 0xF3, 0x20, 0xAD, 0x74, 0x6E, 0x1D, 0x3B, 0x62, 0x8B, 0xA7, 0x9B, 0x98,
    0x59, 0xF7, 0x41, 0xE0, 0x82, 0x54, 0x2A, 0x38, 0x55, 0x02, 0xF2, 0x5D, 0xBF, 0x55, 0x29, 0x6C, 0x3A, 0x54, 0x5E, 0x38, 0x72, 0x76, 0x0A, 0xB7,
    0x36, 0x17, 0xDE, 0x4A, 0x96, 0x26, 0x2C, 0x6F, 0x5D, 0x9E, 0x98, 0xBF, 0x92, 0x92, 0xDC, 0x29, 0xF8, 0xF4, 0x1D, 0xBD, 0x28, 0x9A, 0x14, 0x7C,
    0xE9, 0xDA, 0x31, 0x13, 0xB5, 0xF0, 0xB8, 0xC0, 0x0A, 0x60, 0xB1, 0xCE, 0x1D, 0x7E, 0x81, 0x9D, 0x7A, 0x43, 0x1D, 0x7C, 0x90, 0xEA, 0x0E, 0x5F};

static ecg_status ensure_fb_table(ecg_ctx* ctx, DevState& d, ecg_curve curve) {
  if (d.fb_table[curve]) return ECG_OK;
  Lane& L = d.lane[0];
  const int nl = (int)flimbs(curve);
  const size_t fb = fbytes(curve);
  const int nwin = 2 * nl;  // FB_WINDOWS_NL
  const size_t np = (size_t)nwin * FB_ENTRIES + 1;
  // built in pieces of FB_PIECE points so that the lane's window-table slots (512-768 B per element) and the
  // temporaries stay small: 2^16 points need 33-50 MB of slots instead of 268-402 MB for one launch over all of them
  const size_t FB_PIECE = (size_t)1 << 16;
  std::vector<uint8_t> hk(np * fb), hp(FB_PIECE * 2 * fb);
  const uint32_t* n_le = curve == ECG_SECP256K1 ? H_K256_N : curve == ECG_NISTP256 ? H_P256_N : H_P384_N;
  const uint8_t* g = curve == ECG_SECP256K1 ? H_K256_G : curve == ECG_NISTP256 ? H_P256_G : H_P384_G;
  bool le = false;
  for (int e = 0; e < ECG_EXT_CURVE_COUNT; e++)
    if (ECG_EXT_CURVES[e].id == (int)curve) {
      n_le = ECG_EXT_CURVES[e].n;
      g = ECG_EXT_CURVES[e].g;
      le = ECG_EXT_CURVES[e].le != 0;
    }
  {
    HostMod M;
    M.nl = nl;
    memset(M.n, 0, sizeof M.n);
    for (int i = 0; i < nl; i++) M.n[i] = n_le[i];
    uint32_t Bi[19] = {1}, B2[19], cur[19];  // B_i = 2^(16 i) mod n
    for (int i = 0; i <= nwin; i++) {
      if (i == nwin) {  // the implicit top digit: 2^(16 nwin) = 2^(32 nl) mod n
        scalar_record(&hk[(np - 1) * fb], Bi, nl, fb, le);
        break;
      }
      M.add(B2, Bi, Bi);
      memcpy(cur, Bi, sizeof cur);
      for (uint32_t j = 0; j < FB_ENTRIES; j++) {
        scalar_record(&hk[((size_t)i * FB_ENTRIES + j) * fb], cur, nl, fb, le);
        M.add(cur, cur, B2);
      }
      for (int d = 0; d < FB_W; d++) M.add(Bi, Bi, Bi);
    }
  }
  for (size_t i = 0; i < FB_PIECE; i++) memcpy(&hp[i * 2 * fb], g, 2 * fb);
  // temporaries are released on every exit path; `table` is released unless it is handed to the DevState
  struct Scratch {
    void* p[8] = {nullptr};
    ~Scratch() {
      for (void* q : p)
        if (q) cudaFree(q);
    }
  } tmp;
  CU_TRY(ctx, cudaMalloc(&tmp.p[0], np * fb));
  CU_TRY(ctx, cudaMalloc(&tmp.p[1], FB_PIECE * 2 * fb));
  CU_TRY(ctx, cudaMalloc(&tmp.p[2], FB_PIECE * 2 * fb));
  CU_TRY(ctx, cudaMalloc(&tmp.p[3], FB_PIECE));
  CU_TRY(ctx, cudaMalloc(&tmp.p[4], FB_PIECE * 12 * (size_t)nl));  // Jacobian SoA, NL words per coordinate
  CU_TRY(ctx, cudaMalloc(&tmp.p[5], FB_PIECE * 4 * (size_t)nl));   // inversion scratch
  CU_TRY(ctx, cudaMalloc(&tmp.p[6], np * 8 * (size_t)nl));         // the table: x, y in internal form
  CU_TRY(ctx, cudaMalloc(&tmp.p[7], 8));  // private status: building the table must not disturb a caller's validation state
  uint8_t *dk = (uint8_t*)tmp.p[0], *dpnt = (uint8_t*)tmp.p[1], *dxy = (uint8_t*)tmp.p[2], *dinf = (uint8_t*)tmp.p[3];
  uint32_t *jac = (uint32_t*)tmp.p[4], *scr = (uint32_t*)tmp.p[5], *table = (uint32_t*)tmp.p[6], *st = (uint32_t*)tmp.p[7];
  CU_TRY(ctx, cudaMemsetAsync(st, 0, 8, L.s()));
  CU_TRY(ctx, cudaMemcpyAsync(dk, hk.data(), np * fb, cudaMemcpyHostToDevice, L.s()));
  CU_TRY(ctx, cudaMemcpyAsync(dpnt, hp.data(), FB_PIECE * 2 * fb, cudaMemcpyHostToDevice, L.s()));
  bool saved_timing = ctx->timing;
  ctx->timing = false;
  ecg_status rc = ECG_OK;
  for (size_t lo = 0; lo < np && rc == ECG_OK; lo += FB_PIECE) {
    size_t cnt = std::min(FB_PIECE, np - lo);
    DevPtrs dp;
    dp.k = dk + fb * lo;
    dp.p = dpnt;
    rc = launch_varbase(ctx, d, L, curve, cnt, dp, jac, st, lo);
    if (rc != ECG_OK) break;
    size_t want_threads = std::max<size_t>((cnt + 31) / 32, std::min<size_t>(cnt, (size_t)d.sm_count * 256));
    FOR_CURVE(curve, normalize_kernel<CV::F><<<grid_for(want_threads, 256), 256, 0, L.s()>>>(jac, cnt, scr, dxy, dinf);
              affine_to_table_kernel<CV><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dxy, cnt, table + lo * 2 * nl));
    ctx->launches += 2;
    if (cudaGetLastError() != cudaSuccess) {
      ctx->err = "fixed-base table build: kernel launch failed";
      rc = ECG_ECUDA;
    }
  }
  ctx->timing = saved_timing;
  // nothing may still be using the temporaries when they are freed; lane 1 (and any caller stream) may use the table
  // from now on: it was completed with a full synchronize
  cudaError_t se = cudaStreamSynchronize(L.s());
  if (rc != ECG_OK) return rc;
  CU_TRY(ctx, se);
  tmp.p[6] = nullptr;  // keep the table
  d.fb_table[curve] = table;
  return ECG_OK;
}

// ---- per-element batch driver ------------------------------------------------------------------------
// What one chunk does is the only thing that differs between ecg_mul_batch, ecg_mul_gen_batch, ecg_mul_gen_add_batch,
// ecg_batch_normalize and ecg_field_op_batch:
struct BatchOp {
  enum Kind { MUL, MULGEN, MULGENADD, NORMALIZE, FIELD, SCHNORR, ECDSA, DECOMPRESS, FSQRT, RECOVER } kind;
  ecg_curve curve;
  int fop = 0;  // field op, the ECDSA low-S flag, or NORMALIZE's "homogeneous input" flag
  bool x_only = false;  // MUL: write x coordinates only (ostride 32)
  const uint8_t *k = nullptr, *a = nullptr, *p = nullptr, *inf = nullptr;  // host or device, per ctx flags
  const uint8_t* x = nullptr;  // extra 2 FB-byte-stride input (ECDSA public keys)
  size_t xstride = 64;
  size_t kstride = 32;  // scalars / field elements / messages: fbytes(curve) for the hot-path entries
  size_t pstride = 64;
  uint8_t *out = nullptr, *oinf = nullptr;
  uint8_t* aux_out = nullptr;  // third output array (decompress: validity flags)
  size_t ostride = 64;
};

// the generic twins of the a*G + b*P / ECDSA kernels serve every curve except secp256k1 and P-256: in group 0 that is P-384
#if ECG_TU == 0
#define ECDSA_FOR_CURVE(...)  \
  do {                        \
    typedef CurveP384 CV;     \
    __VA_ARGS__;              \
  } while (0)
static const int GB = Q_BLOCK;
#define ECDSA_MINBLK Q_MINBLK
#else
#define ECDSA_FOR_CURVE(...) FOR_CURVE(op.curve, __VA_ARGS__)
static const int GB = X_BLOCK;
#define ECDSA_MINBLK XGeom<CV::F::NL>::MINBLK
#endif

static ecg_status run_chunk(ecg_ctx* ctx, DevState& d, Lane& L, const BatchOp& op, size_t off, size_t cnt) {
  DevPtrs dp;
  ST_TRY(begin_lane(ctx, L));
  ST_TRY(stage_in(ctx, L, B_K, op.k, off, cnt, op.kstride, &dp.k));
  ST_TRY(stage_in(ctx, L, B_A, op.a, off, cnt, op.kstride, &dp.a));
  ST_TRY(stage_in(ctx, L, B_P, op.p, off, cnt, op.pstride, &dp.p));
  ST_TRY(stage_in(ctx, L, B_INF, op.inf, off, cnt, 1, &dp.inf));
  const uint8_t* dx = nullptr;
  ST_TRY(stage_in(ctx, L, B_X, op.x, off, cnt, op.xstride, &dx));
  ST_TRY(stage_out(ctx, L, off, cnt, op.out, op.ostride, op.oinf, dp));
  if ((op.kind == BatchOp::DECOMPRESS || op.kind == BatchOp::FSQRT) && !curve_256(op.curve)) {
    // generic twins: y = rhs^((p+1)/4) for every curve with p = 3 (mod 4)
    if (op.kind == BatchOp::DECOMPRESS) {
      ST_TRY(ensure(ctx, L, B_V4, cnt));
      uint8_t* vvalid = (ctx->devptr() && op.aux_out) ? op.aux_out + off : (uint8_t*)L.buf[B_V4];
      ECDSA_FOR_CURVE((decompress_generic_kernel<CV, SqrtExp<CV>::T><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.p, cnt, dp.out, dp.oinf, vvalid)));
      LAUNCHED(ctx);
      if (!ctx->devptr() && op.aux_out) CU_TRY(ctx, cudaMemcpyAsync(op.aux_out + off, vvalid, cnt, cudaMemcpyDeviceToHost, L.s()));
    } else {
      ECDSA_FOR_CURVE((field_sqrt_generic_kernel<CV, SqrtExp<CV>::T><<<grid_for(cnt, 128), 128, 0, L.s()>>>(cnt, dp.k, dp.out, dp.oinf, L.status, off)));
      LAUNCHED(ctx);
    }
    return copy_back(ctx, L, off, cnt, op.out, op.ostride, op.oinf, dp);
  }
  if (op.kind == BatchOp::ECDSA && !curve_256(op.curve)) {
    // ECDSA for the other curves: generic front end -> (u1, u2, Q) -> u1*G + u2*Q -> affine -> verdict (the 256-bit path
    // below, record sizes by the curve)
    const size_t fb = fbytes(op.curve), nl = flimbs(op.curve);
    ST_TRY(ensure(ctx, L, B_V1, cnt * 2 * fb));
    ST_TRY(ensure(ctx, L, B_V2, cnt * fb));
    ST_TRY(ensure(ctx, L, B_V3, cnt * fb));
    ST_TRY(ensure(ctx, L, B_V4, cnt));
    ST_TRY(ensure(ctx, L, B_V5, cnt * 2 * fb));
    ST_TRY(ensure(ctx, L, B_V6, cnt));
    ST_TRY(ensure(ctx, L, B_JAC, cnt * jbytes(op.curve)));
    ST_TRY(ensure(ctx, L, B_SCR, cnt * 4 * nl));
    ST_TRY(ensure_tab(ctx, L, op.curve, cnt));
    uint8_t *vp = (uint8_t*)L.buf[B_V1], *va = (uint8_t*)L.buf[B_V2], *vb = (uint8_t*)L.buf[B_V3], *vok = (uint8_t*)L.buf[B_V4];
    uint8_t *vxy = (uint8_t*)L.buf[B_V5], *vinf = (uint8_t*)L.buf[B_V6];
    uint32_t* vj = (uint32_t*)L.buf[B_JAC];
    size_t want_threads = std::max<size_t>((cnt + 31) / 32, std::min<size_t>(cnt, (size_t)d.sm_count * 128));
#if ECG_TU == 1
    const bool sm2dsa = (op.fop & 2) != 0;  // ecg_sm2dsa_verify_batch: another front end and verdict around the same a*G + b*P
    if (sm2dsa)
      sm2dsa_prep_kernel<CurveSm2><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.p, dx, cnt, vp, va, vb, vok);
    else
#else
    const bool sm2dsa = false;
#endif
      ECDSA_FOR_CURVE((ecdsa_prep_generic_kernel<CV><<<grid_for(want_threads, 128), 128, 0, L.s()>>>(dp.k, dp.p, dx, cnt, op.fop, (uint32_t*)L.buf[B_SCR], vp,
                                                                                                va, vb, vok)));
    LAUNCHED(ctx);
    DOM_BEGIN(ctx, L);
    ECDSA_FOR_CURVE((mul_gen_add_generic_kernel<CV, GB, ECDSA_MINBLK><<<grid_for(cnt, GB), GB, 0, L.s()>>>(va, vb, vp, nullptr, cnt, d.fb_table[op.curve], vj,
                                                                                                     (uint32_t*)L.buf[B_TAB], L.status, off)));
    LAUNCHED(ctx);
    DOM_END(ctx, L);
    ST_TRY(launch_norm(ctx, d, L, op.curve, cnt, vj, vxy, vinf));
#if ECG_TU == 1
    if (sm2dsa)
      sm2dsa_check_kernel<CurveSm2><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.k, dp.p, vxy, vinf, vok, cnt, dp.out);
    else
#endif
      ECDSA_FOR_CURVE((ecdsa_check_generic_kernel<CV><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.p, vxy, vinf, vok, cnt, dp.out)));
    (void)sm2dsa;
    LAUNCHED(ctx);
    return copy_back(ctx, L, off, cnt, op.out, op.ostride, nullptr, dp);
  }
#if ECG_TU == 0
  if (op.kind == BatchOp::DECOMPRESS) {
    // out = xy (64 B), oinf = identity flags, valid flags go to a third host array staged through B_V4
    ST_TRY(ensure(ctx, L, B_V4, cnt));
    uint8_t* vvalid = (ctx->devptr() && op.aux_out) ? op.aux_out + off : (uint8_t*)L.buf[B_V4];
    if (op.curve == ECG_SECP256K1)
      decompress_kernel<CurveK256><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.p, cnt, dp.out, dp.oinf, vvalid);
    else
      decompress_kernel<CurveP256><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.p, cnt, dp.out, dp.oinf, vvalid);
    LAUNCHED(ctx);
    if (!ctx->devptr() && op.aux_out) CU_TRY(ctx, cudaMemcpyAsync(op.aux_out + off, vvalid, cnt, cudaMemcpyDeviceToHost, L.s()));
    return copy_back(ctx, L, off, cnt, op.out, op.ostride, op.oinf, dp);
  }
  if (op.kind == BatchOp::FSQRT) {
    if (op.curve == ECG_SECP256K1)
      field_sqrt_kernel<CurveK256><<<grid_for(cnt, 128), 128, 0, L.s()>>>(cnt, dp.k, dp.out, dp.oinf, L.status, off);
    else
      field_sqrt_kernel<CurveP256><<<grid_for(cnt, 128), 128, 0, L.s()>>>(cnt, dp.k, dp.out, dp.oinf, L.status, off);
    LAUNCHED(ctx);
    return copy_back(ctx, L, off, cnt, op.out, op.ostride, op.oinf, dp);
  }
  if (op.kind == BatchOp::SCHNORR || op.kind == BatchOp::ECDSA || op.kind == BatchOp::RECOVER) {
    // front end -> (a, b, P) -> a*G + b*P -> affine -> verdict (or, for key recovery, the point itself), all on the device
    ST_TRY(ensure(ctx, L, B_V1, cnt * 64));
    ST_TRY(ensure(ctx, L, B_V2, cnt * 32));
    ST_TRY(ensure(ctx, L, B_V3, cnt * 32));
    ST_TRY(ensure(ctx, L, B_V4, cnt));
    ST_TRY(ensure(ctx, L, B_V5, cnt * 64));
    ST_TRY(ensure(ctx, L, B_V6, cnt));
    ST_TRY(ensure(ctx, L, B_JAC, cnt * 96));
    ST_TRY(ensure_tab(ctx, L, op.curve, cnt));
    uint8_t *vp = (uint8_t*)L.buf[B_V1], *va = (uint8_t*)L.buf[B_V2], *vb = (uint8_t*)L.buf[B_V3], *vok = (uint8_t*)L.buf[B_V4];
    uint8_t *vxy = (uint8_t*)L.buf[B_V5], *vinf = (uint8_t*)L.buf[B_V6];
    uint32_t* vj = (uint32_t*)L.buf[B_JAC];
    const bool k1c = op.curve == ECG_SECP256K1;
    if (op.kind == BatchOp::SCHNORR) {
      schnorr_prep_kernel<<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.k, dp.a, dp.p, cnt, vp, va, vb, vok);
    } else if (op.kind == BatchOp::RECOVER) {
      ST_TRY(ensure(ctx, L, B_SCR, cnt * 32));
      size_t want_threads = std::max<size_t>((cnt + 31) / 32, std::min<size_t>(cnt, (size_t)d.sm_count * 128));
      if (k1c) {
        ecdsa_recover_point_kernel<CurveK256><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.p, dp.inf, cnt, op.fop, vp, vok);
        ecdsa_recover_prep_kernel<CurveK256><<<grid_for(want_threads, 128), 128, 0, L.s()>>>(dp.k, dp.p, vok, cnt, (uint32_t*)L.buf[B_SCR], va, vb);
      } else {
        ecdsa_recover_point_kernel<CurveP256><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.p, dp.inf, cnt, op.fop, vp, vok);
        ecdsa_recover_prep_kernel<CurveP256><<<grid_for(want_threads, 128), 128, 0, L.s()>>>(dp.k, dp.p, vok, cnt, (uint32_t*)L.buf[B_SCR], va, vb);
      }
      LAUNCHED(ctx);
    } else {
      ST_TRY(ensure(ctx, L, B_SCR, cnt * 32));
      size_t want_threads = std::max<size_t>((cnt + 31) / 32, std::min<size_t>(cnt, (size_t)d.sm_count * 128));
      if (k1c)
        ecdsa_prep_kernel<CurveK256><<<grid_for(want_threads, 128), 128, 0, L.s()>>>(dp.k, dp.p, dx, cnt, op.fop, (uint32_t*)L.buf[B_SCR], vp, va, vb, vok);
      else
        ecdsa_prep_kernel<CurveP256><<<grid_for(want_threads, 128), 128, 0, L.s()>>>(dp.k, dp.p, dx, cnt, op.fop, (uint32_t*)L.buf[B_SCR], vp, va, vb, vok);
    }
    LAUNCHED(ctx);
    DOM_BEGIN(ctx, L);
    if (k1c)
      mul_gen_add_kernel<CurveK256, KG_BLOCK, KG_MINBLK, true><<<grid_for(cnt, KG_BLOCK), KG_BLOCK, 0, L.s()>>>(
          va, vb, vp, nullptr, cnt, d.fb_table[op.curve], vj, (uint32_t*)L.buf[B_TAB], L.status, off);
    else
      mul_gen_add_kernel<CurveP256, P_BLOCK, P_MINBLK, false><<<grid_for(cnt, P_BLOCK), P_BLOCK, 0, L.s()>>>(
          va, vb, vp, nullptr, cnt, d.fb_table[op.curve], vj, (uint32_t*)L.buf[B_TAB], L.status, off);
    LAUNCHED(ctx);
    DOM_END(ctx, L);
    if (op.kind == BatchOp::RECOVER) {  // the recovered key goes out as x || y; the identity-flag array becomes the verdict
      ST_TRY(launch_norm(ctx, d, L, op.curve, cnt, vj, dp.out, dp.oinf));
      ecdsa_recover_finish_kernel<><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.out, dp.oinf, vok, cnt);
      LAUNCHED(ctx);
      return copy_back(ctx, L, off, cnt, op.out, op.ostride, op.oinf, dp);
    }
    ST_TRY(launch_norm(ctx, d, L, op.curve, cnt, vj, vxy, vinf));
    if (op.kind == BatchOp::SCHNORR)
      schnorr_check_kernel<<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.p, vxy, vinf, vok, cnt, dp.out);
    else if (k1c)
      ecdsa_check_kernel<CurveK256><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.p, vxy, vinf, vok, cnt, dp.out);
    else
      ecdsa_check_kernel<CurveP256><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.p, vxy, vinf, vok, cnt, dp.out);
    LAUNCHED(ctx);
    return copy_back(ctx, L, off, cnt, op.out, op.ostride, nullptr, dp);
  }
#else
  (void)dx;
#endif
  uint32_t* jac = nullptr;
  if (op.kind != BatchOp::FIELD) {
    ST_TRY(ensure(ctx, L, B_JAC, cnt * jbytes(op.curve)));
    jac = (uint32_t*)L.buf[B_JAC];
  }
  switch (op.kind) {
    case BatchOp::MUL:
      ST_TRY(launch_varbase(ctx, d, L, op.curve, cnt, dp, jac, L.status, off));
      break;
    case BatchOp::MULGEN:
      if (ctx->flags & ECG_FLAG_CONSTTIME) {  // no table indexed by 16 secret bits: the variable-base routine with P = G
        DevPtrs g = dp;
        g.p = nullptr;
        g.inf = nullptr;
        ST_TRY(launch_varbase(ctx, d, L, op.curve, cnt, g, jac, L.status, off));
        break;
      }
      DOM_BEGIN(ctx, L);
      if (inline_loops())
        FOR_CURVE_INL(op.curve, fixedbase_kernel<CV><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.k, cnt, d.fb_table[op.curve], jac, L.status, off));
      else
        FOR_CURVE(op.curve, fixedbase_kernel<CV><<<grid_for(cnt, 128), 128, 0, L.s()>>>(dp.k, cnt, d.fb_table[op.curve], jac, L.status, off));
      LAUNCHED(ctx);
      DOM_END(ctx, L);
      break;
    case BatchOp::MULGENADD:
      if (!curve_256(op.curve)) {  // generic twin (record sizes by the curve)
        ST_TRY(ensure_tab(ctx, L, op.curve, cnt));
        DOM_BEGIN(ctx, L);
        ECDSA_FOR_CURVE((mul_gen_add_generic_kernel<CV, GB, ECDSA_MINBLK><<<grid_for(cnt, GB), GB, 0, L.s()>>>(dp.a, dp.k, dp.p, dp.inf, cnt, d.fb_table[op.curve], jac,
                                                                                                         (uint32_t*)L.buf[B_TAB], L.status, off)));
        LAUNCHED(ctx);
        DOM_END(ctx, L);
        break;
      }
#if ECG_TU == 0
      ST_TRY(ensure_tab(ctx, L, op.curve, cnt));
      DOM_BEGIN(ctx, L);
      if (op.curve == ECG_SECP256K1)
        mul_gen_add_kernel<CurveK256, KG_BLOCK, KG_MINBLK, true><<<grid_for(cnt, KG_BLOCK), KG_BLOCK, 0, L.s()>>>(
            dp.a, dp.k, dp.p, dp.inf, cnt, d.fb_table[op.curve], jac, (uint32_t*)L.buf[B_TAB], L.status, off);
      else
        mul_gen_add_kernel<CurveP256, P_BLOCK, P_MINBLK, false><<<grid_for(cnt, P_BLOCK), P_BLOCK, 0, L.s()>>>(
            dp.a, dp.k, dp.p, dp.inf, cnt, d.fb_table[op.curve], jac, (uint32_t*)L.buf[B_TAB], L.status, off);
      LAUNCHED(ctx);
      DOM_END(ctx, L);
#endif
      break;
    case BatchOp::NORMALIZE:
      if (op.fop)
        FOR_CURVE(op.curve, import_jac_kernel<CV, true><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.p, cnt, jac, L.status, off));
      else
        FOR_CURVE(op.curve, import_jac_kernel<CV, false><<<grid_for(cnt, 256), 256, 0, L.s()>>>(dp.p, cnt, jac, L.status, off));
      LAUNCHED(ctx);
      break;
    case BatchOp::SCHNORR:
    case BatchOp::ECDSA:
    case BatchOp::DECOMPRESS:
    case BatchOp::FSQRT:
      break;  // handled above
    case BatchOp::FIELD:
      FOR_CURVE(op.curve, field_op_kernel<CV><<<grid_for(cnt, 256), 256, 0, L.s()>>>(op.fop, cnt, dp.k, dp.a, dp.out, L.status, off));
      LAUNCHED(ctx);
      break;
  }
  if (op.kind != BatchOp::FIELD) ST_TRY(launch_norm(ctx, d, L, op.curve, cnt, jac, dp.out, dp.oinf, op.x_only));
  return copy_back(ctx, L, off, cnt, op.out, op.ostride, op.oinf, dp);
}

// Chunks of one device's range in host-pointer mode.  Two things cost time when a batch is cut into chunks: the first
// chunk's upload and the last chunk's download are not hidden behind a kernel of the other lane, and every chunk whose
// size is not a whole number of waves (all threads of the scalar-multiplication kernels run equally long, so a wave
// ends sharply) wastes part of its last wave.  So chunks are whole waves: 1, 2, then 3 waves, ending with one wave plus
// whatever is left.  `wave` = SMs x resident blocks x block size of the variable-base kernels.
static std::vector<Shard> chunk_schedule(size_t cnt, size_t wave) {
  std::vector<Shard> v;
  const size_t maxc = std::max(wave, HOST_CHUNK / wave * wave);
  size_t off = 0, next = wave;
  while (off < cnt) {
    size_t left = cnt - off;
    size_t c = std::min(next, left);
    size_t rest = left - c;
    if (rest > 0 && rest < wave)
      c = left >= 2 * wave ? (left - wave) / wave * wave : left;  // no tiny tail
    else if (rest == 0 && left > 2 * wave)
      c = (left - wave) / wave * wave;  // split the final chunk so that the exposed download is small
    v.push_back({off, c});
    off += c;
    next = std::min(next + wave, maxc);
  }
  return v;
}

static ecg_status run_batch_inner(ecg_ctx* ctx, const BatchOp& op, size_t n) {
  std::vector<Shard> shards = make_shards(n, ctx->devs.size());
  bool need_table = (op.kind == BatchOp::MULGEN && !(ctx->flags & ECG_FLAG_CONSTTIME)) || op.kind == BatchOp::MULGENADD ||
                    op.kind == BatchOp::SCHNORR || op.kind == BatchOp::ECDSA || op.kind == BatchOp::RECOVER;
  for (size_t i = 0; i < ctx->devs.size(); i++) {
    if (shards[i].cnt == 0) continue;
    DevState& d = ctx->devs[i];
    CU_TRY(ctx, cudaSetDevice(d.dev));
    if (need_table) {
      ecg_status st = ensure_fb_table(ctx, d, op.curve);
      if (st != ECG_OK) return fail(ctx, st);
    }
  }
  if (ctx->devptr()) {
    DevState& d = ctx->devs[0];
    for (size_t lo = 0; lo < n; lo += DEV_CHUNK) {
      ecg_status st = run_chunk(ctx, d, d.lane[0], op, lo, std::min(DEV_CHUNK, n - lo));
      if (st != ECG_OK) return fail(ctx, st);
    }
    return finish(ctx);
  }
  // host mode: interleave chunks across devices and lanes so copies and kernels of different chunks overlap
  std::vector<std::vector<Shard>> sched(shards.size());
  size_t maxchunks = 0;
  for (size_t i = 0; i < shards.size(); i++) {
    sched[i] = chunk_schedule(shards[i].cnt, wave_elems(ctx->devs[i], op.curve));
    maxchunks = std::max(maxchunks, sched[i].size());
  }
  for (size_t c = 0; c < maxchunks; c++) {
    for (size_t i = 0; i < ctx->devs.size(); i++) {
      if (c >= sched[i].size()) continue;
      DevState& d = ctx->devs[i];
      CU_TRY(ctx, cudaSetDevice(d.dev));
      ecg_status st = run_chunk(ctx, d, d.lane[c & 1], op, shards[i].off + sched[i][c].off, sched[i][c].cnt);
      if (st != ECG_OK) return fail(ctx, st);
    }
  }
  return finish(ctx);
}

// every error exit (including CUDA failures inside finish()) leaves the lanes reset: fail() is idempotent
static ecg_status run_batch(ecg_ctx* ctx, const BatchOp& op, size_t n) {
  ecg_status st = run_batch_inner(ctx, op, n);
  return st == ECG_OK ? st : fail(ctx, st);
}

// ---- entry points -------------------------------------------------------------------------------------
// group 0 owns the extern "C" symbols and hands calls for the other groups' curves to their translation units
#if ECG_TU == 0
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_mul_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_mul_gen_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_batch_normalize(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_batch_normalize_hom(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_mul_batch_x(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_x, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_field_op_batch(ecg_ctx* ctx, ecg_curve curve, int fop, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_lincomb_partial(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xyz);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_point_sum(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_lincomb(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_mul_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_mul_gen_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_batch_normalize(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_batch_normalize_hom(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_mul_batch_x(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_x, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_field_op_batch(ecg_ctx* ctx, ecg_curve curve, int fop, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_lincomb_partial(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xyz);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_point_sum(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_lincomb(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_mul_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_mul_gen_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_batch_normalize(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_batch_normalize_hom(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_mul_batch_x(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_x, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_field_op_batch(ecg_ctx* ctx, ecg_curve curve, int fop, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_lincomb_partial(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xyz);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_point_sum(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_lincomb(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_mul_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_mul_gen_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_batch_normalize(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_batch_normalize_hom(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_mul_batch_x(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_x, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_field_op_batch(ecg_ctx* ctx, ecg_curve curve, int fop, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_lincomb_partial(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xyz);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_point_sum(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_lincomb(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_sm2dsa_verify_batch(ecg_ctx* ctx, size_t n, const uint8_t* e32, const uint8_t* sig64, const uint8_t* Q_xy, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_sm2pke_encrypt_batch(ecg_ctx* ctx, size_t n, const uint8_t* msgs, const uint64_t* offsets,
                                                                                const uint8_t* k32, const uint8_t* Pb_xy, int mode, int compressed,
                                                                                uint8_t* out, uint8_t* status);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_sm2pke_decrypt_batch(ecg_ctx* ctx, size_t n, const uint8_t* cts, const uint64_t* offsets,
                                                                                const uint8_t* d32, int mode, uint8_t* out, uint64_t* pt_len,
                                                                                uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_mul_gen_add_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, const uint8_t* b, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_ecdsa_verify_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64, const uint8_t* Q_xy, int low_s_only, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_mul_gen_add_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, const uint8_t* b, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_ecdsa_verify_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64, const uint8_t* Q_xy, int low_s_only, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_mul_gen_add_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, const uint8_t* b, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_ecdsa_verify_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64, const uint8_t* Q_xy, int low_s_only, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_mul_gen_add_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, const uint8_t* b, const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_ecdsa_verify_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64, const uint8_t* Q_xy, int low_s_only, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_decompress_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* sec1_33, uint8_t* out_xy, uint8_t* out_inf, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu1_ecg_field_sqrt_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, uint8_t* out, uint8_t* is_square);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_decompress_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* sec1_33, uint8_t* out_xy, uint8_t* out_inf, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu2_ecg_field_sqrt_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, uint8_t* out, uint8_t* is_square);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_decompress_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* sec1_33, uint8_t* out_xy, uint8_t* out_inf, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu3_ecg_field_sqrt_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, uint8_t* out, uint8_t* is_square);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_decompress_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* sec1_33, uint8_t* out_xy, uint8_t* out_inf, uint8_t* valid);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_field_sqrt_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, uint8_t* out, uint8_t* is_square);
#define ECG_FORWARD(name, ...)                                     \
  do {                                                             \
    if ((int)curve >= 0 && (int)curve < ECG_CURVE_COUNT) {         \
      switch (curve_group((int)curve)) {                           \
        case 1: return ecg_tu1_##name(__VA_ARGS__);                \
        case 2: return ecg_tu2_##name(__VA_ARGS__);                \
        case 3: return ecg_tu3_##name(__VA_ARGS__);                \
        case 4: return ecg_tu4_##name(__VA_ARGS__);                \
        default: break;                                            \
      }                                                            \
    }                                                              \
  } while (0)
#else
#define ECG_FORWARD(name, ...) ((void)0)
#endif

ECG_API(ecg_mul_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                                    const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_mul_batch, ctx, curve, n, k, P_xy, P_inf, out_xy, out_inf);
  if (n == 0) return ECG_OK;
  if (!k || !P_xy || !out_xy || !curve_ok(curve)) {
    ctx->err = "ecg_mul_batch: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::MUL;
  op.curve = curve;
  op.kstride = fbytes(curve);
  op.pstride = op.ostride = 2 * fbytes(curve);
  op.k = k;
  op.p = P_xy;
  op.inf = P_inf;
  op.out = out_xy;
  op.oinf = out_inf;
  return run_batch(ctx, op, n);
}

ECG_API(ecg_mul_gen_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, uint8_t* out_xy,
                                        uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_mul_gen_batch, ctx, curve, n, k, out_xy, out_inf);
  if (n == 0) return ECG_OK;
  if (!k || !out_xy || !curve_ok(curve)) {
    ctx->err = "ecg_mul_gen_batch: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::MULGEN;
  op.curve = curve;
  op.kstride = fbytes(curve);
  op.ostride = 2 * fbytes(curve);
  op.k = k;
  op.out = out_xy;
  op.oinf = out_inf;
  return run_batch(ctx, op, n);
}

ECG_API(ecg_mul_gen_add_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, const uint8_t* b,
                               const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_mul_gen_add_batch, ctx, curve, n, a, b, P_xy, P_inf, out_xy, out_inf);
  if (n == 0) return ECG_OK;
  if (!a || !b || !P_xy || !out_xy || !curve_ok(curve)) {
    ctx->err = "ecg_mul_gen_add_batch: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::MULGENADD;
  op.curve = curve;
  op.kstride = fbytes(curve);
  op.pstride = op.ostride = 2 * fbytes(curve);
  op.a = a;
  op.k = b;
  op.p = P_xy;
  op.inf = P_inf;
  op.out = out_xy;
  op.oinf = out_inf;
  return run_batch(ctx, op, n);
}

ECG_API(ecg_decompress_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* sec1_33, uint8_t* out_xy,
                              uint8_t* out_inf, uint8_t* valid) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_decompress_batch, ctx, curve, n, sec1_33, out_xy, out_inf, valid);
  if (n == 0) return ECG_OK;
  if (!sec1_33 || !out_xy || !out_inf || !valid || !curve_ok(curve)) {
    ctx->err = "ecg_decompress_batch: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::DECOMPRESS;
  op.curve = curve;
  op.p = sec1_33;
  op.pstride = fbytes(curve) + 1;
  op.ostride = 2 * fbytes(curve);
  op.out = out_xy;
  op.oinf = out_inf;
  op.aux_out = valid;
  return run_batch(ctx, op, n);
}
#if ECG_TU == 0

extern "C" ecg_status ecg_schnorr_verify_batch(ecg_ctx* ctx, size_t n, const uint8_t* pk_x, const uint8_t* msg32, const uint8_t* sig64,
                                                uint8_t* valid) {
  if (!ctx) return ECG_EINVAL;
  if (n == 0) return ECG_OK;
  if (!pk_x || !msg32 || !sig64 || !valid) {
    ctx->err = "ecg_schnorr_verify_batch: null pointer";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::SCHNORR;
  op.curve = ECG_SECP256K1;
  op.k = pk_x;
  op.a = msg32;
  op.p = sig64;
  op.out = valid;
  op.ostride = 1;
  return run_batch(ctx, op, n);
}

#endif  // ECG_TU == 0
ECG_API(ecg_ecdsa_verify_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64,
                                const uint8_t* Q_xy, int low_s_only, uint8_t* valid) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_ecdsa_verify_batch, ctx, curve, n, z32, sig64, Q_xy, low_s_only, valid);
  if (n == 0) return ECG_OK;
  // ECDSA is defined by the reference for every curve here except sm2 (SM2DSA) and bign-curve256v1 (its own scheme)
  if (!z32 || !sig64 || !Q_xy || !valid || !curve_ok(curve) || curve == ECG_SM2 || curve == ECG_BIGNP256) {
    ctx->err = "ecg_ecdsa_verify_batch: null pointer or a curve without ECDSA";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::ECDSA;
  op.curve = curve;
  op.fop = low_s_only ? 1 : 0;
  op.kstride = fbytes(curve);
  op.pstride = op.xstride = 2 * fbytes(curve);
  op.k = z32;
  op.p = sig64;
  op.x = Q_xy;
  op.out = valid;
  op.ostride = 1;
  return run_batch(ctx, op, n);
}
#if ECG_TU == 0
ECG_API(ecg_ecdsa_recover_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64, const uint8_t* recid,
                                 int low_s_only, uint8_t* out_xy, uint8_t* valid) {
  if (!ctx) return ECG_EINVAL;
  if (n == 0) return ECG_OK;
  if (!z32 || !sig64 || !recid || !out_xy || !valid || !curve_256(curve)) {
    ctx->err = "ecg_ecdsa_recover_batch: null pointer, or a curve other than secp256k1 / P-256";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::RECOVER;
  op.curve = curve;
  op.fop = low_s_only ? 1 : 0;
  op.kstride = 32;
  op.pstride = 64;
  op.k = z32;
  op.p = sig64;
  op.inf = recid;
  op.out = out_xy;
  op.ostride = 64;
  op.oinf = valid;
  return run_batch(ctx, op, n);
}
#endif

// SM2DSA: TU 1 holds sm2; the public entry (TU 0) forwards there like every other sm2 call
ECG_API(ecg_sm2dsa_verify_batch)(ecg_ctx* ctx, size_t n, const uint8_t* e32, const uint8_t* sig64, const uint8_t* Q_xy, uint8_t* valid) {
  if (!ctx) return ECG_EINVAL;
#if ECG_TU == 0
  return ecg_tu1_ecg_sm2dsa_verify_batch(ctx, n, e32, sig64, Q_xy, valid);
#elif ECG_TU == 1
  if (n == 0) return ECG_OK;
  if (!e32 || !sig64 || !Q_xy || !valid) {
    ctx->err = "ecg_sm2dsa_verify_batch: null pointer";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::ECDSA;
  op.curve = ECG_SM2;
  op.fop = 2;
  op.kstride = 32;
  op.pstride = op.xstride = 64;
  op.k = e32;
  op.p = sig64;
  op.x = Q_xy;
  op.out = valid;
  op.ostride = 1;
  return run_batch(ctx, op, n);
#else
  return ECG_EINVAL;
#endif
}

#if ECG_TU == 1
// ---- SM2 public-key encryption (ecg_sm2pke.cuh): one pass on device 0, lane 0 ---------------------------------------
// front end -> variable-base [k]Pb / [d]C1 -> affine (x2, y2) -> (encryption: [k]G -> affine C1) -> KDF / C3 / layout
static ecg_status sm2pke_run(ecg_ctx* ctx, bool enc, size_t n, const uint8_t* data, const uint64_t* offsets, const uint8_t* key32,
                             const uint8_t* pb_xy, int mode, int compressed, uint8_t* out, uint8_t* verdict, uint64_t* pt_len) {
  DevState& d = ctx->devs[0];
  Lane& L = d.lane[0];
  CU_TRY(ctx, cudaSetDevice(d.dev));
  const bool ct = (ctx->flags & ECG_FLAG_CONSTTIME) != 0;
  if (enc && !ct) ST_TRY(ensure_fb_table(ctx, d, ECG_SM2));
  ST_TRY(begin_lane(ctx, L));
  const size_t ovh = enc ? 32 + (compressed ? 33 : 65) : 0;
  const uint8_t *ddata = data, *dkey = key32, *dpb = pb_xy;
  const uint64_t* doffs = offsets;
  uint8_t *dout = out, *dverdict = verdict;
  uint64_t* dlen = pt_len;
  uint64_t base = 0;
  size_t out_bytes = 0;
  if (!ctx->devptr()) {
    base = offsets[0];
    const size_t total = (size_t)(offsets[n] - base);
    out_bytes = total + n * ovh;
    ST_TRY(ensure(ctx, L, B_P, total + 16));
    ST_TRY(ensure(ctx, L, B_K, (n + 1) * 8));
    ST_TRY(ensure(ctx, L, B_A, n * 32));
    if (total) CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_P], data + base, total, cudaMemcpyHostToDevice, L.s()));
    CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_K], offsets, (n + 1) * 8, cudaMemcpyHostToDevice, L.s()));
    CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_A], key32, n * 32, cudaMemcpyHostToDevice, L.s()));
    ddata = (const uint8_t*)L.buf[B_P];
    doffs = (const uint64_t*)L.buf[B_K];
    dkey = (const uint8_t*)L.buf[B_A];
    if (enc) {
      ST_TRY(ensure(ctx, L, B_X, n * 64));
      CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_X], pb_xy, n * 64, cudaMemcpyHostToDevice, L.s()));
      dpb = (const uint8_t*)L.buf[B_X];
    }
    ST_TRY(ensure(ctx, L, B_OUT, out_bytes + 16));
    ST_TRY(ensure(ctx, L, B_OINF, n));
    dout = (uint8_t*)L.buf[B_OUT];
    dverdict = (uint8_t*)L.buf[B_OINF];
    if (!enc) {
      ST_TRY(ensure(ctx, L, B_AUX, n * 8));
      dlen = (uint64_t*)L.buf[B_AUX];
    }
  }
  ST_TRY(ensure(ctx, L, B_V1, n * 64));
  ST_TRY(ensure(ctx, L, B_V2, n * 32));
  ST_TRY(ensure(ctx, L, B_V4, n));
  ST_TRY(ensure(ctx, L, B_V5, n * 64));
  ST_TRY(ensure(ctx, L, B_V6, n));
  ST_TRY(ensure(ctx, L, B_JAC, n * jbytes(ECG_SM2)));
  uint8_t *vp = (uint8_t*)L.buf[B_V1], *vk = (uint8_t*)L.buf[B_V2], *vok = (uint8_t*)L.buf[B_V4];
  uint8_t *vxy = (uint8_t*)L.buf[B_V5], *vinf = (uint8_t*)L.buf[B_V6];
  if (enc)
    sm2pke_enc_prep_kernel<CurveSm2><<<grid_for(n, 128), 128, 0, L.s()>>>(doffs, n, dkey, dpb, vk, vp, vok);
  else
    sm2pke_dec_prep_kernel<CurveSm2><<<grid_for(n, 128), 128, 0, L.s()>>>(ddata, doffs, base, n, dkey, vk, vp, vok);
  LAUNCHED(ctx);
  DevPtrs dp;
  dp.k = vk;
  dp.p = vp;
  ST_TRY(launch_varbase(ctx, d, L, ECG_SM2, n, dp, (uint32_t*)L.buf[B_JAC], L.status, 0));
  ST_TRY(launch_norm(ctx, d, L, ECG_SM2, n, (uint32_t*)L.buf[B_JAC], vxy, vinf));
  const uint8_t* c1xy = nullptr;
  if (enc) {  // C1 = [k]G: the fixed-base table, or under ECG_FLAG_CONSTTIME the variable-base routine with P = G
    ST_TRY(ensure(ctx, L, B_JAC2, n * jbytes(ECG_SM2)));
    ST_TRY(ensure(ctx, L, B_V3, n * 64));
    ST_TRY(ensure(ctx, L, B_INF, n));
    uint32_t* jac2 = (uint32_t*)L.buf[B_JAC2];
    if (ct) {
      DevPtrs g;
      g.k = vk;
      ST_TRY(launch_varbase(ctx, d, L, ECG_SM2, n, g, jac2, L.status, 0));
    } else {
      DOM_BEGIN(ctx, L);
      fixedbase_kernel<CurveSm2><<<grid_for(n, 128), 128, 0, L.s()>>>(vk, n, d.fb_table[ECG_SM2], jac2, L.status, 0);
      LAUNCHED(ctx);
      DOM_END(ctx, L);
    }
    ST_TRY(launch_norm(ctx, d, L, ECG_SM2, n, jac2, (uint8_t*)L.buf[B_V3], (uint8_t*)L.buf[B_INF]));
    c1xy = (const uint8_t*)L.buf[B_V3];
  }
  if (enc)
    sm2pke_kdf_kernel<true><<<grid_for(n, 128), 128, 0, L.s()>>>(ddata, doffs, base, n, mode, compressed, vxy, c1xy, vok, dout, dverdict, nullptr);
  else
    sm2pke_kdf_kernel<false><<<grid_for(n, 128), 128, 0, L.s()>>>(ddata, doffs, base, n, mode, 0, vxy, nullptr, vok, dout, dverdict, dlen);
  LAUNCHED(ctx);
  if (!ctx->devptr()) {
    if (out_bytes) CU_TRY(ctx, cudaMemcpyAsync(out, dout, out_bytes, cudaMemcpyDeviceToHost, L.s()));
    CU_TRY(ctx, cudaMemcpyAsync(verdict, dverdict, n, cudaMemcpyDeviceToHost, L.s()));
    if (!enc) CU_TRY(ctx, cudaMemcpyAsync(pt_len, dlen, n * 8, cudaMemcpyDeviceToHost, L.s()));
  }
  return ECG_OK;
}

static ecg_status sm2pke_entry(ecg_ctx* ctx, bool enc, size_t n, const uint8_t* data, const uint64_t* offsets, const uint8_t* key32,
                               const uint8_t* pb_xy, int mode, int compressed, uint8_t* out, uint8_t* verdict, uint64_t* pt_len) {
  const char* who = enc ? "ecg_sm2pke_encrypt_batch" : "ecg_sm2pke_decrypt_batch";
  if (n == 0) return ECG_OK;
  if (!offsets || !key32 || !out || !verdict || (enc && !pb_xy) || (!enc && !pt_len) || n > ((size_t)1 << 31)) {
    ctx->err = std::string(who) + ": null pointer";
    return ECG_EINVAL;
  }
  if (mode != 0 && mode != 1) {
    ctx->err = std::string(who) + ": mode must be 0 (C1C3C2) or 1 (C1C2C3)";
    return ECG_EINVAL;
  }
  if (ctx->devptr()) {
    if (!data || (reinterpret_cast<uintptr_t>(offsets) & 7) || (reinterpret_cast<uintptr_t>(key32) & 3) ||
        (reinterpret_cast<uintptr_t>(pb_xy) & 3) || (reinterpret_cast<uintptr_t>(pt_len) & 7)) {
      ctx->err = std::string(who) + ": null device pointer, or offsets / pt_len not 8-byte aligned, or keys not 4-byte aligned";
      return ECG_EINVAL;
    }
  } else {
    for (size_t i = 0; i < n; i++)
      if (offsets[i + 1] < offsets[i]) {
        ctx->err = std::string(who) + ": offsets must be non-decreasing";
        return ECG_EINVAL;
      }
    if (!data && offsets[n] != offsets[0]) {
      ctx->err = std::string(who) + ": null data buffer";
      return ECG_EINVAL;
    }
  }
  ecg_status st = sm2pke_run(ctx, enc, n, data, offsets, key32, pb_xy, mode, compressed, out, verdict, pt_len);
  if (st != ECG_OK) return fail(ctx, st);
  st = finish(ctx);
  return st == ECG_OK ? st : fail(ctx, st);
}
#endif  // ECG_TU == 1

// SM2 public-key encryption: TU 1 holds sm2; the public entries (TU 0) forward there
ECG_API(ecg_sm2pke_encrypt_batch)(ecg_ctx* ctx, size_t n, const uint8_t* msgs, const uint64_t* offsets, const uint8_t* k32,
                                  const uint8_t* Pb_xy, int mode, int compressed, uint8_t* out, uint8_t* status) {
  if (!ctx) return ECG_EINVAL;
#if ECG_TU == 0
  return ecg_tu1_ecg_sm2pke_encrypt_batch(ctx, n, msgs, offsets, k32, Pb_xy, mode, compressed, out, status);
#elif ECG_TU == 1
  return sm2pke_entry(ctx, true, n, msgs, offsets, k32, Pb_xy, mode, compressed, out, status, nullptr);
#else
  return ECG_EINVAL;
#endif
}
ECG_API(ecg_sm2pke_decrypt_batch)(ecg_ctx* ctx, size_t n, const uint8_t* cts, const uint64_t* offsets, const uint8_t* d32, int mode,
                                  uint8_t* out, uint64_t* pt_len, uint8_t* valid) {
  if (!ctx) return ECG_EINVAL;
#if ECG_TU == 0
  return ecg_tu1_ecg_sm2pke_decrypt_batch(ctx, n, cts, offsets, d32, mode, out, pt_len, valid);
#elif ECG_TU == 1
  return sm2pke_entry(ctx, false, n, cts, offsets, d32, nullptr, mode, 0, out, valid, pt_len);
#else
  return ECG_EINVAL;
#endif
}

ECG_API(ecg_batch_normalize)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy,
                                          uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_batch_normalize, ctx, curve, n, xyz, out_xy, out_inf);
  if (n == 0) return ECG_OK;
  if (!xyz || !out_xy || !curve_ok(curve)) return ECG_EINVAL;
  BatchOp op;
  op.kind = BatchOp::NORMALIZE;
  op.curve = curve;
  op.ostride = 2 * fbytes(curve);
  op.p = xyz;
  op.pstride = 3 * fbytes(curve);
  op.out = out_xy;
  op.oinf = out_inf;
  return run_batch(ctx, op, n);
}

ECG_API(ecg_batch_normalize_hom)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy,
                                              uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_batch_normalize_hom, ctx, curve, n, xyz, out_xy, out_inf);
  if (n == 0) return ECG_OK;
  if (!xyz || !out_xy || !curve_ok(curve)) return ECG_EINVAL;
  BatchOp op;
  op.kind = BatchOp::NORMALIZE;
  op.curve = curve;
  op.ostride = 2 * fbytes(curve);
  op.fop = 1;  // homogeneous (X:Y:Z), x = X/Z
  op.p = xyz;
  op.pstride = 3 * fbytes(curve);
  op.out = out_xy;
  op.oinf = out_inf;
  return run_batch(ctx, op, n);
}

ECG_API(ecg_mul_batch_x)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                                      const uint8_t* P_inf, uint8_t* out_x, uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_mul_batch_x, ctx, curve, n, k, P_xy, P_inf, out_x, out_inf);
  if (n == 0) return ECG_OK;
  if (!k || !P_xy || !out_x || !curve_ok(curve)) {
    ctx->err = "ecg_mul_batch_x: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  BatchOp op;
  op.kind = BatchOp::MUL;
  op.curve = curve;
  op.kstride = fbytes(curve);
  op.pstride = 2 * fbytes(curve);
  op.k = k;
  op.p = P_xy;
  op.inf = P_inf;
  op.out = out_x;
  op.oinf = out_inf;
  op.ostride = fbytes(curve);
  op.x_only = true;
  return run_batch(ctx, op, n);
}

ECG_API(ecg_field_sqrt_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, uint8_t* out,
                              uint8_t* is_square) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_field_sqrt_batch, ctx, curve, n, a, out, is_square);
  if (n == 0) return ECG_OK;
  if (!a || !out || !is_square || !curve_ok(curve) || curve == ECG_NISTP224) return ECG_EINVAL;  // P-224: p = 1 (mod 4)
  BatchOp op;
  op.kind = BatchOp::FSQRT;
  op.curve = curve;
  op.k = a;
  op.kstride = fbytes(curve);
  op.out = out;
  op.oinf = is_square;
  op.ostride = fbytes(curve);
  return run_batch(ctx, op, n);
}

ECG_API(ecg_field_op_batch)(ecg_ctx* ctx, ecg_curve curve, int fop, size_t n, const uint8_t* a, const uint8_t* b,
                                         uint8_t* out) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_field_op_batch, ctx, curve, fop, n, a, b, out);
  if (n == 0) return ECG_OK;
  bool binary = (fop == ECG_FOP_ADD || fop == ECG_FOP_SUB || fop == ECG_FOP_MUL);
  if (!a || !out || (binary && !b) || fop < 0 || fop > ECG_FOP_INV || !curve_ok(curve)) return ECG_EINVAL;
  BatchOp op;
  op.kind = BatchOp::FIELD;
  op.curve = curve;
  op.kstride = fbytes(curve);
  op.fop = fop;
  op.k = a;
  op.a = binary ? b : nullptr;
  op.out = out;
  op.ostride = fbytes(curve);
  return run_batch(ctx, op, n);
}

// ---- lincomb ----------------------------------------------------------------------------------------
// Reduce n Jacobian points (SoA in `a`) to one, ping-ponging between a and b; *result = buffer holding it.
template <class C>
static ecg_status reduce_points(ecg_ctx* ctx, Lane& L, uint32_t* a, uint32_t* b, size_t n, uint32_t** result) {
  while (n > 1) {
    size_t m = (n + 31) / 32;
    jac_sum_kernel<C><<<grid_for(m, 128), 128, 0, L.s()>>>(a, n, b, m);
    LAUNCHED(ctx);
    std::swap(a, b);
    n = m;
  }
  *result = a;
  return ECG_OK;
}
static ecg_status reduce_points_c(ecg_ctx* ctx, Lane& L, ecg_curve curve, uint32_t* a, uint32_t* b, size_t n, uint32_t** result) {
  FOR_CURVE(curve, return reduce_points<CV>(ctx, L, a, b, n, result));
  return ECG_EINVAL;
}

// ---- bucket-method lincomb (ecg_msm.cuh) ------------------------------------------------------------
static const size_t MSM_MIN_TERMS = (size_t)1 << 13;   // below this the per-term kernel + tree sum is faster
static const size_t MSM_MAX_TERMS_DEFAULT = (size_t)1 << 24;  // per call (32-bit list offsets); larger shards are cut
// ECG_MSM_MAX_TERMS (environment) lowers the piece size so that tests can exercise the multi-piece path cheaply
static size_t msm_max_terms() {
  const char* e = getenv("ECG_MSM_MAX_TERMS");
  if (e) {
    size_t v = (size_t)strtoull(e, nullptr, 10);
    if (v >= MSM_MIN_TERMS && v <= MSM_MAX_TERMS_DEFAULT) return v;
  }
  return MSM_MAX_TERMS_DEFAULT;
}

// ECG_MSM_BUCKETS_PER_THREAD = 4 | 8 selects msm_bucket_sorted_kernel (experiment, default 1 = msm_bucket_kernel)
static int msm_buckets_per_thread() {
  const char* e = getenv("ECG_MSM_BUCKETS_PER_THREAD");
  int v = e ? atoi(e) : 1;
  return (v == 4 || v == 8) ? v : 1;
}

static MsmGeom msm_geometry(ecg_curve curve, size_t n) {
  MsmGeom g;
  bool glv = curve == ECG_SECP256K1;
  size_t nsub = glv ? 2 * n : n;
  int lg = 0;
  while (((size_t)1 << (lg + 1)) <= nsub) lg++;
  g.c = std::min(16, std::max(8, lg - 5));
  g.nbits = glv ? 128 : (int)(32 * flimbs(curve));
  while ((g.nbits + g.c - 1) / g.c > MSM_FINAL_THREADS) g.c++;  // msm_final_kernel: one thread per window (P-521: 544 bits -> c >= 9)
  g.W = (g.nbits + g.c - 1) / g.c;
  g.nbw = ((uint32_t)1 << (g.c + 1)) + 2;
  return g;
}

struct Carver {
  uint8_t* base;
  size_t off = 0;
  template <class T>
  T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

// Everything is enqueued without waiting; if the input turns out too skewed for the bucket method the result is
// garbage and finish() sets ctx->skew (the caller then repeats the call with per_term = true).
template <class C, class CI, bool GLV>
static ecg_status msm_run(ecg_ctx* ctx, Lane& L, const DevPtrs& dp, size_t n, size_t base, const MsmGeom& g, uint32_t** result) {
  const size_t nsub = GLV ? 2 * n : n;
  const size_t nb = (size_t)g.W * g.nbw;
  constexpr size_t NLc = C::F::NL;
  // recursion geometry of the weighted reduction
  std::vector<size_t> lens, nchs;
  size_t len = g.nbw - 1;
  for (;;) {
    const size_t chl = lens.empty() ? MSM_CH0 : MSM_CHU;  // chunk size of this level (ecg_msm.cuh)
    size_t nch = (len + chl - 1) / chl;
    lens.push_back(len);
    nchs.push_back(nch);
    if (nch == 1) break;
    len = nch;
  }
  const int levels = (int)lens.size();
  // carve the scratch arena (first pass sizes it, second pass hands out pointers)
  uint32_t *pts = nullptr, *count = nullptr, *cursor = nullptr, *offset = nullptr, *list = nullptr, *bkt = nullptr, *res = nullptr;
  uint32_t *blocksum = nullptr, *order = nullptr, *ohist = nullptr;
  int32_t* digits = nullptr;
  std::vector<uint32_t*> S(levels), X(levels);
  uint32_t* Rw = nullptr;
  for (int pass = 0; pass < 2; pass++) {
    Carver cv{pass ? (uint8_t*)L.buf[B_MSM] : nullptr};
    pts = cv.take<uint32_t>(nsub * 2 * NLc);
    digits = cv.take<int32_t>(nsub * (size_t)g.W);
    count = cv.take<uint32_t>(2 * nb + 4);  // count | cursor | maxcnt, cleared together
    cursor = count ? count + nb + 1 : nullptr;
    blocksum = cv.take<uint32_t>((nb + MSM_SCAN_CHUNK - 1) / MSM_SCAN_CHUNK + 1);
    offset = cv.take<uint32_t>(nb + 1);
    list = cv.take<uint32_t>(nsub * (size_t)g.W);
    bkt = cv.take<uint32_t>(nb * 3 * NLc);
    order = cv.take<uint32_t>(nb);
    ohist = cv.take<uint32_t>(MSM_ORDER_CLASSES + 1);
    for (int l = 0; l < levels; l++) {
      S[l] = cv.take<uint32_t>((size_t)g.W * nchs[l] * 3 * NLc);
      X[l] = cv.take<uint32_t>((size_t)g.W * nchs[l] * 3 * NLc);
    }
    Rw = cv.take<uint32_t>((size_t)g.W * 3 * NLc);
    res = cv.take<uint32_t>(3 * NLc);
    if (pass == 0) ST_TRY(ensure(ctx, L, B_MSM, cv.off + 256));
  }
  uint32_t* maxcnt = count + 2 * nb + 3;
  CU_TRY(ctx, cudaMemsetAsync(count, 0, (2 * nb + 4) * 4, L.s()));
  msm_prep_kernel<C, GLV><<<grid_for(n, 128), 128, 0, L.s()>>>(dp.k, dp.p, dp.inf, n, g, pts, digits, count, L.status, base);
  LAUNCHED(ctx);
  {
    unsigned sb = (unsigned)((nb + MSM_SCAN_CHUNK - 1) / MSM_SCAN_CHUNK);
    msm_scan_partial_kernel<0><<<sb, MSM_SCAN_BLOCK, 0, L.s()>>>(count, nb, blocksum, maxcnt);
    LAUNCHED(ctx);
    msm_scan_top_kernel<0><<<1, 1024, 0, L.s()>>>(blocksum, sb, offset, nb);
    LAUNCHED(ctx);
    msm_scan_final_kernel<0><<<sb, MSM_SCAN_BLOCK, 0, L.s()>>>(count, nb, blocksum, offset);
    LAUNCHED(ctx);
  }
  // one bucket thread adds its points serially: pathologically skewed inputs (e.g. thousands of identical terms) are
  // declined by the bucket kernel itself (MsmSkew, ecg_msm.cuh) — no host round trip here; finish() reports the flag
  // and the caller repeats the call on the per-term path, whose cost does not depend on the data
  const size_t avg = nsub / ((size_t)1 << (g.c - 1)) + 1;
  MsmSkew sk{maxcnt, 4096u, (uint32_t)std::min<size_t>(32 * avg, 0xFFFFFFFFu), L.status};
  msm_scatter_kernel<0><<<grid_for(nsub, 256), 256, 0, L.s()>>>(digits, nsub, g, offset, cursor, list);
  LAUNCHED(ctx);
  // bucket ids by decreasing population (ECG_MSM_ORDER=0 keeps the natural order: measurement knob)
  static const bool use_order = []() {
    const char* e = getenv("ECG_MSM_ORDER");
    return !(e && e[0] == '0');
  }();
  if (use_order) {
    CU_TRY(ctx, cudaMemsetAsync(ohist, 0, (MSM_ORDER_CLASSES + 1) * 4, L.s()));
    unsigned ob = (unsigned)std::min<size_t>((nb + 255) / 256, 592);
    msm_order_hist_kernel<0><<<ob, 256, 0, L.s()>>>(offset, nb, ohist);
    LAUNCHED(ctx);
    msm_order_scan_kernel<0><<<1, MSM_ORDER_CLASSES, 0, L.s()>>>(ohist);
    LAUNCHED(ctx);
    msm_order_scatter_kernel<0><<<ob, 256, 0, L.s()>>>(offset, nb, ohist, order);
    LAUNCHED(ctx);
  }
  DOM_BEGIN(ctx, L);
  switch (msm_buckets_per_thread()) {  // > 1: warp-balanced variant (ecg_msm.cuh), off unless the environment asks for it
#if ECG_TU == 0
    case 8:
      msm_bucket_sorted_kernel<C, 8><<<grid_for(nb, MSM_BS_BLOCK * 8), MSM_BS_BLOCK, 0, L.s()>>>(pts, list, offset, nb, bkt, sk);
      break;
    case 4:
      msm_bucket_sorted_kernel<C, 4><<<grid_for(nb, MSM_BS_BLOCK * 4), MSM_BS_BLOCK, 0, L.s()>>>(pts, list, offset, nb, bkt, sk);
      break;
#endif
    default:
      if (inline_loops())
        msm_bucket_kernel<CI><<<grid_for(nb, 128), 128, 0, L.s()>>>(pts, list, offset, nb, bkt, sk, use_order ? order : nullptr);
      else
        msm_bucket_kernel<C><<<grid_for(nb, 128), 128, 0, L.s()>>>(pts, list, offset, nb, bkt, sk, use_order ? order : nullptr);
  }
  LAUNCHED(ctx);
  DOM_END(ctx, L);
  // weighted reduction, level by level (ecg_msm.cuh)
  for (int l = 0; l < levels; l++) {
    const uint32_t* in = l == 0 ? bkt : S[l - 1];
    size_t n_in = l == 0 ? nb : (size_t)g.W * nchs[l - 1];
    size_t stride = l == 0 ? g.nbw : nchs[l - 1];
    size_t off = l == 0 ? 1 : 0;
    // rows below the top window only populate the first 2^(c-1) slots (level 0), i.e. ceil(that / CH^l) chunk totals at level l
    size_t len_low = ((size_t)1 << (g.c - 1));
    for (int q = 0; q < l; q++) len_low = (len_low + (q == 0 ? MSM_CH0 : MSM_CHU) - 1) / (q == 0 ? MSM_CH0 : MSM_CHU);
    msm_wreduce_kernel<C><<<grid_for((size_t)g.W * nchs[l], 128), 128, 0, L.s()>>>(in, n_in, stride, off, lens[l], std::min(len_low, lens[l]), g.W,
                                                                                 nchs[l], l == 0 ? nullptr : X[l - 1], l, S[l], X[l]);
    LAUNCHED(ctx);
  }
  msm_final_kernel<C><<<1, MSM_FINAL_THREADS, 0, L.s()>>>(X[levels - 1], S[levels - 1], g.W, g.c, levels - 1, Rw, res);
  LAUNCHED(ctx);
  *result = res;
  return ECG_OK;
}

// one shard -> one Jacobian point left in *result (SoA with n = 1, i.e. 24 consecutive words), on lane 0
static ecg_status lincomb_shard(ecg_ctx* ctx, DevState& d, ecg_curve curve, const Shard& sh, const uint8_t* k,
                                const uint8_t* P_xy, const uint8_t* P_inf, bool per_term, uint32_t** result) {
  Lane& L = d.lane[0];
  DevPtrs dp;
  const size_t fb = fbytes(curve), pt = jbytes(curve);  // bytes per scalar record / per Jacobian point in the internal SoA form
  ST_TRY(begin_lane(ctx, L));
  ST_TRY(stage_in(ctx, L, B_K, k, sh.off, sh.cnt, fb, &dp.k));
  ST_TRY(stage_in(ctx, L, B_P, P_xy, sh.off, sh.cnt, 2 * fb, &dp.p));
  ST_TRY(stage_in(ctx, L, B_INF, P_inf, sh.off, sh.cnt, 1, &dp.inf));
  if (ctx->flags & ECG_FLAG_CONSTTIME) per_term = true;  // the bucket method's memory access pattern IS the scalars
  if (sh.cnt >= MSM_MIN_TERMS && !per_term) {
    // bucket method, in pieces of at most MSM_MAX_TERMS terms whose partial sums are added at the end
    const size_t MSM_MAX_TERMS = msm_max_terms();
    size_t pieces = (sh.cnt + MSM_MAX_TERMS - 1) / MSM_MAX_TERMS;
    ST_TRY(ensure(ctx, L, B_JAC, pieces * pt + pt));
    ST_TRY(ensure(ctx, L, B_JAC2, pieces * pt + pt));
    uint32_t* parts = (uint32_t*)L.buf[B_JAC];
    for (size_t pc = 0; pc < pieces; pc++) {
      size_t lo = pc * MSM_MAX_TERMS, cnt = std::min(MSM_MAX_TERMS, sh.cnt - lo);
      DevPtrs q;
      q.k = dp.k + fb * lo;
      q.p = dp.p + 2 * fb * lo;
      q.inf = dp.inf ? dp.inf + lo : nullptr;
      MsmGeom g = msm_geometry(curve, cnt);
      uint32_t* r1 = nullptr;
#if ECG_TU == 0
      if (curve == ECG_SECP256K1)
        ST_TRY((msm_run<CurveK256, CurveK256I, true>(ctx, L, q, cnt, sh.off + lo, g, &r1)));
      else if (curve == ECG_NISTP256)
        ST_TRY((msm_run<CurveP256, CurveP256I, false>(ctx, L, q, cnt, sh.off + lo, g, &r1)));
      else
        ST_TRY((msm_run<CurveP384, CurveP384I, false>(ctx, L, q, cnt, sh.off + lo, g, &r1)));
#else
      FOR_CURVE(curve, ST_TRY((msm_run<CV, CV, false>(ctx, L, q, cnt, sh.off + lo, g, &r1))));
#endif
      if (pieces == 1) {
        *result = r1;
        return ECG_OK;
      }
      // gather piece results into an SoA array of `pieces` points (24 strided 4-byte copies)
      for (int w = 0; w < (int)(3 * flimbs(curve)); w++)
        CU_TRY(ctx, cudaMemcpyAsync(parts + (size_t)w * pieces + pc, r1 + w, 4, cudaMemcpyDeviceToDevice, L.s()));
    }
    return reduce_points_c(ctx, L, curve, parts, (uint32_t*)L.buf[B_JAC2], pieces, result);
  }
  // per-term path: one scalar multiplication per term in pieces of at most PT_CHUNK terms (bounds the window tables:
  // 512-768 B per term), each piece tree-summed to one point, the piece sums added at the end
  const size_t PT_CHUNK = (size_t)1 << 20;
  const size_t pieces = (sh.cnt + PT_CHUNK - 1) / PT_CHUNK;
  const size_t c0 = std::min(sh.cnt, PT_CHUNK);
  ST_TRY(ensure(ctx, L, B_FB1, c0 * pt));
  ST_TRY(ensure(ctx, L, B_FB2, ((c0 + 31) / 32) * pt + 256));
  ST_TRY(ensure(ctx, L, B_JAC, pieces * pt + pt));
  ST_TRY(ensure(ctx, L, B_JAC2, ((pieces + 31) / 32) * pt + pt));
  uint32_t* parts = (uint32_t*)L.buf[B_JAC];
  for (size_t pc = 0; pc < pieces; pc++) {
    size_t lo = pc * PT_CHUNK, cnt = std::min(PT_CHUNK, sh.cnt - lo);
    DevPtrs q;
    q.k = dp.k + fb * lo;
    q.p = dp.p + 2 * fb * lo;
    q.inf = dp.inf ? dp.inf + lo : nullptr;
    uint32_t* r1 = nullptr;
    ST_TRY(launch_varbase(ctx, d, L, curve, cnt, q, (uint32_t*)L.buf[B_FB1], L.status, sh.off + lo));
    ST_TRY(reduce_points_c(ctx, L, curve, (uint32_t*)L.buf[B_FB1], (uint32_t*)L.buf[B_FB2], cnt, &r1));
    if (pieces == 1) {
      *result = r1;
      return ECG_OK;
    }
    for (int w = 0; w < (int)(3 * flimbs(curve)); w++)
      CU_TRY(ctx, cudaMemcpyAsync(parts + (size_t)w * pieces + pc, r1 + w, 4, cudaMemcpyDeviceToDevice, L.s()));
  }
  return reduce_points_c(ctx, L, curve, parts, (uint32_t*)L.buf[B_JAC2], pieces, result);
}

static ecg_status export_point(ecg_ctx* ctx, Lane& L, ecg_curve curve, const uint32_t* jac1, uint8_t* dev_xyz) {
  FOR_CURVE(curve, export_jac_kernel<CV><<<1, 128, 0, L.s()>>>(jac1, 1, dev_xyz));
  LAUNCHED(ctx);
  return ECG_OK;
}

// One attempt at ecg_lincomb_partial (per_term = false: bucket method where it applies).
static ecg_status lincomb_partial_attempt(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                                          const uint8_t* P_inf, uint8_t* out_xyz, bool per_term) {
  DevState& d = ctx->devs[0];
  Lane& L = d.lane[0];
  Shard sh = {0, n};
  uint32_t* res = nullptr;
  ST_TRY(lincomb_shard(ctx, d, curve, sh, k, P_xy, P_inf, per_term, &res));
  uint8_t* dst = out_xyz;
  if (!ctx->devptr()) {
    ST_TRY(ensure(ctx, L, B_AUX, 256));
    dst = (uint8_t*)L.buf[B_AUX];
  }
  ST_TRY(export_point(ctx, L, curve, res, dst));
  if (!ctx->devptr()) CU_TRY(ctx, cudaMemcpyAsync(out_xyz, dst, 3 * fbytes(curve), cudaMemcpyDeviceToHost, L.s()));
  return ECG_OK;
}

ECG_API(ecg_lincomb_partial)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                                          const uint8_t* P_inf, uint8_t* out_xyz) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_lincomb_partial, ctx, curve, n, k, P_xy, P_inf, out_xyz);
  if (!out_xyz || !curve_ok(curve) || (n > 0 && (!k || !P_xy))) {
    ctx->err = "ecg_lincomb_partial: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  if (ctx->devs.size() != 1) {
    ctx->err = "ecg_lincomb_partial: single-device ctx only (use ecg_lincomb for a multi-device ctx)";
    return ECG_EINVAL;
  }
  DevState& d = ctx->devs[0];
  CU_TRY(ctx, cudaSetDevice(d.dev));
  if (n == 0) {  // empty sum = identity (0 : 1 : 0)
    const size_t fb = fbytes(curve);
    uint8_t z[208];
    identity_xyz(z, curve);
    if (ctx->devptr())
      CU_TRY(ctx, cudaMemcpy(out_xyz, z, 3 * fb, cudaMemcpyHostToDevice));
    else
      memcpy(out_xyz, z, 3 * fb);
    return ECG_OK;
  }
  ctx->skew = false;
  for (int attempt = 0; attempt < 2; attempt++) {
    ecg_status st = lincomb_partial_attempt(ctx, curve, n, k, P_xy, P_inf, out_xyz, attempt == 1);
    if (st != ECG_OK) return fail(ctx, st);
    st = finish(ctx);
    if (st != ECG_OK || !ctx->skew) return st;
    ctx->skew = false;  // the bucket method declined the input: once more, per term
  }
  return ECG_OK;
}

// m Jacobian points (X||Y||Z bytes, host or device per the ctx flags) -> affine sum (device 0 of the ctx, lane 0).
// Nothing is waited for: the caller finishes the lane.
static ecg_status point_sum_enqueue(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t* out_xy, uint8_t* out_inf,
                                    bool xyz_on_host) {
  DevState& d = ctx->devs[0];
  Lane& L = d.lane[0];
  CU_TRY(ctx, cudaSetDevice(d.dev));
  const size_t fb = fbytes(curve), pt = jbytes(curve), rec = 3 * fb;  // internal SoA point / X||Y||Z record at the ABI
  ST_TRY(begin_lane(ctx, L));
  ST_TRY(ensure(ctx, L, B_JAC, m * pt + pt));
  ST_TRY(ensure(ctx, L, B_JAC2, ((m + 31) / 32) * pt + pt));
  const uint8_t* dxyz = xyz;
  if (xyz_on_host) {
    ST_TRY(ensure(ctx, L, B_AUX, m * rec + 256));
    CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_AUX], xyz, m * rec, cudaMemcpyHostToDevice, L.s()));
    dxyz = (const uint8_t*)L.buf[B_AUX];
  }
  uint32_t* jac = (uint32_t*)L.buf[B_JAC];
  FOR_CURVE(curve, import_jac_kernel<CV><<<grid_for(m, 256), 256, 0, L.s()>>>(dxyz, m, jac, L.status, 0));
  LAUNCHED(ctx);
  uint32_t* res = nullptr;
  ST_TRY(reduce_points_c(ctx, L, curve, jac, (uint32_t*)L.buf[B_JAC2], m, &res));
  DevPtrs dp;
  ST_TRY(stage_out(ctx, L, 0, 1, out_xy, 2 * fb, out_inf, dp));
  ST_TRY(launch_norm(ctx, d, L, curve, 1, res, dp.out, dp.oinf));
  return copy_back(ctx, L, 0, 1, out_xy, 2 * fb, out_inf, dp);
}

ECG_API(ecg_point_sum)(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t* out_xy,
                                    uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_point_sum, ctx, curve, m, xyz, out_xy, out_inf);
  if (!out_xy || !out_inf || !curve_ok(curve) || (m > 0 && !xyz)) return ECG_EINVAL;
  if (ctx->devptr() && ((reinterpret_cast<uintptr_t>(xyz) | reinterpret_cast<uintptr_t>(out_xy)) & 3)) {
    ctx->err = "device pointer not 4-byte aligned";
    return ECG_EINVAL;
  }
  if (m == 0) {
    uint8_t z[137];
    memset(z, 0, sizeof z);
    if (ctx->devptr()) {
      CU_TRY(ctx, cudaSetDevice(ctx->devs[0].dev));
      CU_TRY(ctx, cudaMemcpy(out_xy, z, 2 * fbytes(curve), cudaMemcpyHostToDevice));
      z[0] = 1;
      CU_TRY(ctx, cudaMemcpy(out_inf, z, 1, cudaMemcpyHostToDevice));
    } else {
      memcpy(out_xy, z, 2 * fbytes(curve));
      *out_inf = 1;
    }
    return ECG_OK;
  }
  ecg_status st = point_sum_enqueue(ctx, curve, m, xyz, out_xy, out_inf, !ctx->devptr());
  if (st != ECG_OK) return fail(ctx, st);
  return finish(ctx);
}

// One attempt at ecg_lincomb: every device's shard is ENQUEUED (no waiting between devices), the per-device partial
// points come back through pinned host memory, device 0 adds them.
static ecg_status lincomb_attempt(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy, const uint8_t* P_inf,
                                  uint8_t* out_xy, uint8_t* out_inf, bool per_term, std::vector<uint8_t>& partial) {
  size_t nd = ctx->devs.size();
  std::vector<Shard> shards = make_shards(n, nd);
  if (nd == 1) {
    DevState& d = ctx->devs[0];
    Lane& L = d.lane[0];
    CU_TRY(ctx, cudaSetDevice(d.dev));
    uint32_t* res = nullptr;
    ST_TRY(lincomb_shard(ctx, d, curve, shards[0], k, P_xy, P_inf, per_term, &res));
    DevPtrs dp;
    ST_TRY(stage_out(ctx, L, 0, 1, out_xy, 2 * fbytes(curve), out_inf, dp));
    ST_TRY(launch_norm(ctx, d, L, curve, 1, res, dp.out, dp.oinf));
    return copy_back(ctx, L, 0, 1, out_xy, 2 * fbytes(curve), out_inf, dp);
  }
  for (size_t i = 0; i < nd; i++) {
    DevState& d = ctx->devs[i];
    Lane& L = d.lane[0];
    if (shards[i].cnt == 0) continue;
    CU_TRY(ctx, cudaSetDevice(d.dev));
    uint32_t* res = nullptr;
    ST_TRY(lincomb_shard(ctx, d, curve, shards[i], k, P_xy, P_inf, per_term, &res));
    ST_TRY(ensure(ctx, L, B_AUX, 256));
    ST_TRY(export_point(ctx, L, curve, res, (uint8_t*)L.buf[B_AUX]));
    CU_TRY(ctx, cudaMemcpyAsync(L.h_point(), L.buf[B_AUX], 3 * fbytes(curve), cudaMemcpyDeviceToHost, L.s()));
  }
  ST_TRY(finish(ctx));
  if (ctx->skew) return ECG_OK;  // the caller repeats per term
  for (size_t i = 0; i < nd; i++) {
    const size_t pt = 3 * fbytes(curve);
    identity_xyz(&partial[i * pt], curve);  // identity (0:1:0) for empty shards
    if (shards[i].cnt) memcpy(&partial[i * pt], ctx->devs[i].lane[0].h_point(), pt);
  }
  return point_sum_enqueue(ctx, curve, nd, partial.data(), out_xy, out_inf, true);
}

ECG_API(ecg_lincomb)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                                  const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  ECG_FORWARD(ecg_lincomb, ctx, curve, n, k, P_xy, P_inf, out_xy, out_inf);
  if (!out_xy || !out_inf || !curve_ok(curve) || (n > 0 && (!k || !P_xy))) {
    ctx->err = "ecg_lincomb: null pointer or unknown curve";
    return ECG_EINVAL;
  }
  if (n == 0) {
    uint8_t z[137];
    memset(z, 0, sizeof z);
    if (ctx->devptr()) {
      CU_TRY(ctx, cudaMemcpy(out_xy, z, 2 * fbytes(curve), cudaMemcpyHostToDevice));
      z[0] = 1;
      CU_TRY(ctx, cudaMemcpy(out_inf, z, 1, cudaMemcpyHostToDevice));
    } else {
      memcpy(out_xy, z, 2 * fbytes(curve));
      *out_inf = 1;
    }
    return ECG_OK;
  }
  std::vector<uint8_t> partial(ctx->devs.size() * 208, 0);
  ctx->skew = false;
  for (int attempt = 0; attempt < 2; attempt++) {
    ecg_status st = lincomb_attempt(ctx, curve, n, k, P_xy, P_inf, out_xy, out_inf, attempt == 1, partial);
    if (st != ECG_OK) return fail(ctx, st);
    st = finish(ctx);
    if (st != ECG_OK || !ctx->skew) return st;
    ctx->skew = false;  // the bucket method declined the input: once more, per term
  }
  return ECG_OK;
}

#if ECG_TU == 0 || ECG_TU == 4
// ---- hash to curve / hash to scalar (ecg_h2c.cuh) ---------------------------------------------------------------
// host-side SHA-256, only for a DST longer than 255 bytes (RFC 9380 section 5.3.3: DST = H("H2C-OVERSIZE-DST-" || DST))
static void host_sha256(const uint8_t* data, size_t len, uint8_t out[32]) {
  static const uint32_t K[64] = {
      0x428a2f98u, 0x71374491u, 0xb5c0fbcfu, 0xe9b5dba5u, 0x3956c25bu, 0x59f111f1u, 0x923f82a4u, 0xab1c5ed5u, 0xd807aa98u, 0x12835b01u,
      0x243185beu, 0x550c7dc3u, 0x72be5d74u, 0x80deb1feu, 0x9bdc06a7u, 0xc19bf174u, 0xe49b69c1u, 0xefbe4786u, 0x0fc19dc6u, 0x240ca1ccu,
      0x2de92c6fu, 0x4a7484aau, 0x5cb0a9dcu, 0x76f988dau, 0x983e5152u, 0xa831c66du, 0xb00327c8u, 0xbf597fc7u, 0xc6e00bf3u, 0xd5a79147u,
      0x06ca6351u, 0x14292967u, 0x27b70a85u, 0x2e1b2138u, 0x4d2c6dfcu, 0x53380d13u, 0x650a7354u, 0x766a0abbu, 0x81c2c92eu, 0x92722c85u,
      0xa2bfe8a1u, 0xa81a664bu, 0xc24b8b70u, 0xc76c51a3u, 0xd192e819u, 0xd6990624u, 0xf40e3585u, 0x106aa070u, 0x19a4c116u, 0x1e376c08u,
      0x2748774cu, 0x34b0bcb5u, 0x391c0cb3u, 0x4ed8aa4au, 0x5b9cca4fu, 0x682e6ff3u, 0x748f82eeu, 0x78a5636fu, 0x84c87814u, 0x8cc70208u,
      0x90befffau, 0xa4506cebu, 0xbef9a3f7u, 0xc67178f2u};
  uint32_t st[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
  std::vector<uint8_t> buf(data, data + len);
  buf.push_back(0x80);
  while (buf.size() % 64 != 56) buf.push_back(0);
  for (int i = 7; i >= 0; i--) buf.push_back((uint8_t)(((uint64_t)len * 8) >> (8 * i)));
  auto rotr = [](uint32_t x, int n) { return (x >> n) | (x << (32 - n)); };
  for (size_t off = 0; off < buf.size(); off += 64) {
    uint32_t w[64];
    for (int i = 0; i < 16; i++)
      w[i] = ((uint32_t)buf[off + 4 * i] << 24) | ((uint32_t)buf[off + 4 * i + 1] << 16) | ((uint32_t)buf[off + 4 * i + 2] << 8) | buf[off + 4 * i + 3];
    for (int i = 16; i < 64; i++)
      w[i] = w[i - 16] + (rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3)) + w[i - 7] + (rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10));
    uint32_t a = st[0], b = st[1], c = st[2], d = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
    for (int i = 0; i < 64; i++) {
      uint32_t t1 = h + (rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
      uint32_t t2 = (rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
      h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    st[0] += a; st[1] += b; st[2] += c; st[3] += d; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
  }
  for (int i = 0; i < 8; i++)
    for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(st[i] >> (24 - 8 * j));
}

// host-side SHA-384 / SHA-512 for the same purpose in the P-384 / P-521 suites
static void host_sha512(const uint8_t* data, size_t len, bool is384, uint8_t* out /* 48 or 64 bytes */) {
  static const uint64_t K[80] = {
      0x428a2f98d728ae22ull, 0x7137449123ef65cdull, 0xb5c0fbcfec4d3b2full, 0xe9b5dba58189dbbcull, 0x3956c25bf348b538ull, 0x59f111f1b605d019ull,
      0x923f82a4af194f9bull, 0xab1c5ed5da6d8118ull, 0xd807aa98a3030242ull, 0x12835b0145706fbeull, 0x243185be4ee4b28cull, 0x550c7dc3d5ffb4e2ull,
      0x72be5d74f27b896full, 0x80deb1fe3b1696b1ull, 0x9bdc06a725c71235ull, 0xc19bf174cf692694ull, 0xe49b69c19ef14ad2ull, 0xefbe4786384f25e3ull,
      0x0fc19dc68b8cd5b5ull, 0x240ca1cc77ac9c65ull, 0x2de92c6f592b0275ull, 0x4a7484aa6ea6e483ull, 0x5cb0a9dcbd41fbd4ull, 0x76f988da831153b5ull,
      0x983e5152ee66dfabull, 0xa831c66d2db43210ull, 0xb00327c898fb213full, 0xbf597fc7beef0ee4ull, 0xc6e00bf33da88fc2ull, 0xd5a79147930aa725ull,
      0x06ca6351e003826full, 0x142929670a0e6e70ull, 0x27b70a8546d22ffcull, 0x2e1b21385c26c926ull, 0x4d2c6dfc5ac42aedull, 0x53380d139d95b3dfull,
      0x650a73548baf63deull, 0x766a0abb3c77b2a8ull, 0x81c2c92e47edaee6ull, 0x92722c851482353bull, 0xa2bfe8a14cf10364ull, 0xa81a664bbc423001ull,
      0xc24b8b70d0f89791ull, 0xc76c51a30654be30ull, 0xd192e819d6ef5218ull, 0xd69906245565a910ull, 0xf40e35855771202aull, 0x106aa07032bbd1b8ull,
      0x19a4c116b8d2d0c8ull, 0x1e376c085141ab53ull, 0x2748774cdf8eeb99ull, 0x34b0bcb5e19b48a8ull, 0x391c0cb3c5c95a63ull, 0x4ed8aa4ae3418acbull,
      0x5b9cca4f7763e373ull, 0x682e6ff3d6b2b8a3ull, 0x748f82ee5defb2fcull, 0x78a5636f43172f60ull, 0x84c87814a1f0ab72ull, 0x8cc702081a6439ecull,
      0x90befffa23631e28ull, 0xa4506cebde82bde9ull, 0xbef9a3f7b2c67915ull, 0xc67178f2e372532bull, 0xca273eceea26619cull, 0xd186b8c721c0c207ull,
      0xeada7dd6cde0eb1eull, 0xf57d4f7fee6ed178ull, 0x06f067aa72176fbaull, 0x0a637dc5a2c898a6ull, 0x113f9804bef90daeull, 0x1b710b35131c471bull,
      0x28db77f523047d84ull, 0x32caab7b40c72493ull, 0x3c9ebe0a15c9bebcull, 0x431d67c49c100d4cull, 0x4cc5d4becb3e42b6ull, 0x597f299cfc657e2aull,
      0x5fcb6fab3ad6faecull, 0x6c44198c4a475817ull};
  uint64_t st[8];
  const uint64_t iv512[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                             0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
  const uint64_t iv384[8] = {0xcbbb9d5dc1059ed8ull, 0x629a292a367cd507ull, 0x9159015a3070dd17ull, 0x152fecd8f70e5939ull,
                             0x67332667ffc00b31ull, 0x8eb44a8768581511ull, 0xdb0c2e0d64f98fa7ull, 0x47b5481dbefa4fa4ull};
  for (int i = 0; i < 8; i++) st[i] = is384 ? iv384[i] : iv512[i];
  std::vector<uint8_t> buf(data, data + len);
  buf.push_back(0x80);
  while (buf.size() % 128 != 112) buf.push_back(0);
  for (int i = 0; i < 8; i++) buf.push_back(0);  // high half of the 128-bit length
  for (int i = 7; i >= 0; i--) buf.push_back((uint8_t)(((uint64_t)len * 8) >> (8 * i)));
  auto rotr = [](uint64_t x, int n) { return (x >> n) | (x << (64 - n)); };
  for (size_t off = 0; off < buf.size(); off += 128) {
    uint64_t w[80];
    for (int i = 0; i < 16; i++) {
      w[i] = 0;
      for (int j = 0; j < 8; j++) w[i] = (w[i] << 8) | buf[off + 8 * i + j];
    }
    for (int i = 16; i < 80; i++)
      w[i] = w[i - 16] + (rotr(w[i - 15], 1) ^ rotr(w[i - 15], 8) ^ (w[i - 15] >> 7)) + w[i - 7] + (rotr(w[i - 2], 19) ^ rotr(w[i - 2], 61) ^ (w[i - 2] >> 6));
    uint64_t a = st[0], b = st[1], c = st[2], d = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
    for (int i = 0; i < 80; i++) {
      uint64_t t1 = h + (rotr(e, 14) ^ rotr(e, 18) ^ rotr(e, 41)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
      uint64_t t2 = (rotr(a, 28) ^ rotr(a, 34) ^ rotr(a, 39)) + ((a & b) ^ (a & c) ^ (b & c));
      h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    st[0] += a; st[1] += b; st[2] += c; st[3] += d; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
  }
  const int nb = is384 ? 48 : 64;
  for (int i = 0; i < nb; i++) out[i] = (uint8_t)(st[i >> 3] >> (56 - 8 * (i & 7)));
}

// mode 0: hash_to_curve (RO), 1: encode_to_curve (NU), 2: hash_to_scalar
static ecg_status h2c_run(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs, const uint64_t* offsets, const uint8_t* dst,
                          size_t dst_len, int mode, uint8_t* out, uint8_t* out_inf) {
  DevState& d = ctx->devs[0];
  Lane& L = d.lane[0];
  CU_TRY(ctx, cudaSetDevice(d.dev));
  // DST_prime = DST || I2OSP(len(DST), 1), an oversize DST replaced by its hash (expand_msg.rs:76-95)
  uint8_t dst_prime[256];
  uint32_t dpl;
  if (dst_len > 255) {
    std::vector<uint8_t> salted;
    const char* salt = "H2C-OVERSIZE-DST-";
    salted.insert(salted.end(), salt, salt + 17);
    salted.insert(salted.end(), dst, dst + dst_len);
    // hashed with the suite's own hash (Domain::xmd<X>, expand_msg.rs:107-121)
    if (curve_256(curve)) {
      host_sha256(salted.data(), salted.size(), dst_prime);
      dpl = 32;
    } else {
      host_sha512(salted.data(), salted.size(), curve == ECG_NISTP384, dst_prime);
      dpl = curve == ECG_NISTP384 ? 48 : 64;
    }
    dst_prime[dpl] = (uint8_t)dpl;
    dpl += 1;
  } else {
    memcpy(dst_prime, dst, dst_len);
    dst_prime[dst_len] = (uint8_t)dst_len;
    dpl = (uint32_t)dst_len + 1;
  }
  ST_TRY(begin_lane(ctx, L));
  ST_TRY(ensure(ctx, L, B_A, 256));
  CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_A], dst_prime, dpl, cudaMemcpyHostToDevice, L.s()));  // pageable, <= 256 bytes: staged by the driver
  const uint8_t* dmsgs = msgs;
  const uint64_t* doffs = offsets;
  uint64_t base = 0;
  if (!ctx->devptr()) {
    base = offsets[0];
    const uint64_t total = offsets[n] - base;
    for (size_t i = 0; i < n; i++)
      if (offsets[i + 1] < offsets[i]) {
        ctx->err = "hash_to_curve: message offsets must be non-decreasing";
        return ECG_EINVAL;
      }
    ST_TRY(ensure(ctx, L, B_P, (size_t)total + 16));
    ST_TRY(ensure(ctx, L, B_K, (n + 1) * 8));
    if (total) CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_P], msgs + base, (size_t)total, cudaMemcpyHostToDevice, L.s()));
    CU_TRY(ctx, cudaMemcpyAsync(L.buf[B_K], offsets, (n + 1) * 8, cudaMemcpyHostToDevice, L.s()));
    dmsgs = (const uint8_t*)L.buf[B_P];
    doffs = (const uint64_t*)L.buf[B_K];
  } else if (reinterpret_cast<uintptr_t>(offsets) & 7) {
    ctx->err = "device pointer (offsets) not 8-byte aligned";
    return ECG_EINVAL;
  }
  const uint8_t* dprime = (const uint8_t*)L.buf[B_A];
  const size_t fb = fbytes(curve);
  DevPtrs dp;
// the suites: group 0 serves secp256k1 / P-256 (SHA-256) and P-384 (SHA-384), group 4 P-521 (SHA-512)
#if ECG_TU == 0
#define H2C_FOR_SUITE(...)                \
  do {                                    \
    if (curve == ECG_SECP256K1) {         \
      typedef CurveK256 CV;               \
      typedef FpMontT<MnK256> FN;         \
      __VA_ARGS__;                        \
    } else if (curve == ECG_NISTP256) {   \
      typedef CurveP256 CV;               \
      typedef FpMontT<MnP256> FN;         \
      __VA_ARGS__;                        \
    } else {                              \
      typedef CurveP384 CV;               \
      typedef FpMontT<MnP384> FN;         \
      __VA_ARGS__;                        \
    }                                     \
  } while (0)
#else
#define H2C_FOR_SUITE(...)        \
  do {                            \
    typedef CurveP521 CV;         \
    typedef FpMontT<MnP521> FN;   \
    __VA_ARGS__;                  \
  } while (0)
#endif
  if (mode == 2) {
    ST_TRY(stage_out(ctx, L, 0, n, out, fb, nullptr, dp));
    DOM_BEGIN(ctx, L);
    H2C_FOR_SUITE((h2s_kernel<CV, FN><<<grid_for(n, 128), 128, 0, L.s()>>>(dmsgs, doffs, base, n, dprime, dpl, dp.out)));
    LAUNCHED(ctx);
    DOM_END(ctx, L);
    return copy_back(ctx, L, 0, n, out, fb, nullptr, dp);
  }
  ST_TRY(stage_out(ctx, L, 0, n, out, 2 * fb, out_inf, dp));
  ST_TRY(ensure(ctx, L, B_JAC, n * jbytes(curve)));
  uint32_t* jac = (uint32_t*)L.buf[B_JAC];
  DOM_BEGIN(ctx, L);
  if (mode == 0)
    H2C_FOR_SUITE((h2c_kernel<CV, false><<<grid_for(n, 128), 128, 0, L.s()>>>(dmsgs, doffs, base, n, dprime, dpl, jac)));
  else
    H2C_FOR_SUITE((h2c_kernel<CV, true><<<grid_for(n, 128), 128, 0, L.s()>>>(dmsgs, doffs, base, n, dprime, dpl, jac)));
  LAUNCHED(ctx);
  DOM_END(ctx, L);
  ST_TRY(launch_norm(ctx, d, L, curve, n, jac, dp.out, dp.oinf));
  return copy_back(ctx, L, 0, n, out, 2 * fb, out_inf, dp);
}

static ecg_status h2c_entry(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs, const uint64_t* offsets, const uint8_t* dst,
                            size_t dst_len, int mode, uint8_t* out, uint8_t* out_inf) {
  if (!ctx) return ECG_EINVAL;
  const bool suite_here = ECG_TU == 0 ? (curve == ECG_SECP256K1 || curve == ECG_NISTP256 || curve == ECG_NISTP384) : curve == ECG_NISTP521;
  if (!suite_here || !dst || dst_len == 0 || dst_len > 65535) {  // ExpandMsgXmdError::EmptyDst
    ctx->err = "hash_to_curve: secp256k1 / P-256 / P-384 / P-521 only, and a non-empty domain separation tag is required";
    return ECG_EINVAL;
  }
  if (n == 0) return ECG_OK;
  if (!offsets || !out || (mode != 2 && !out_inf) || n > ((size_t)1 << 31)) {
    ctx->err = "hash_to_curve: null pointer";
    return ECG_EINVAL;
  }
  if (!msgs && (ctx->devptr() || offsets[n] != offsets[0])) {
    ctx->err = "hash_to_curve: null message buffer";
    return ECG_EINVAL;
  }
  ecg_status st = h2c_run(ctx, curve, n, msgs, offsets, dst, dst_len, mode, out, out_inf);
  if (st != ECG_OK) return fail(ctx, st);
  st = finish(ctx);
  return st == ECG_OK ? st : fail(ctx, st);
}

#if ECG_TU == 0
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_hash_to_curve_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs,
                                                                              const uint64_t* offsets, const uint8_t* dst, size_t dst_len,
                                                                              int nonuniform, uint8_t* out_xy, uint8_t* out_inf);
__attribute__((visibility("hidden"))) ecg_status ecg_tu4_ecg_hash_to_scalar_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs,
                                                                               const uint64_t* offsets, const uint8_t* dst, size_t dst_len, uint8_t* out);
#endif
ECG_API(ecg_hash_to_curve_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs, const uint64_t* offsets,
                                 const uint8_t* dst, size_t dst_len, int nonuniform, uint8_t* out_xy, uint8_t* out_inf) {
#if ECG_TU == 0
  if (ctx && curve == ECG_NISTP521) return ecg_tu4_ecg_hash_to_curve_batch(ctx, curve, n, msgs, offsets, dst, dst_len, nonuniform, out_xy, out_inf);
#endif
  return h2c_entry(ctx, curve, n, msgs, offsets, dst, dst_len, nonuniform ? 1 : 0, out_xy, out_inf);
}
ECG_API(ecg_hash_to_scalar_batch)(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs, const uint64_t* offsets,
                                  const uint8_t* dst, size_t dst_len, uint8_t* out) {
#if ECG_TU == 0
  if (ctx && curve == ECG_NISTP521) return ecg_tu4_ecg_hash_to_scalar_batch(ctx, curve, n, msgs, offsets, dst, dst_len, out);
#endif
  return h2c_entry(ctx, curve, n, msgs, offsets, dst, dst_len, 2, out, nullptr);
}
#endif  // ECG_TU == 0 || ECG_TU == 4

#if ECG_TU == 0
extern "C" ecg_status ecg_microbench(ecg_ctx* ctx, int which, int iters, double* ops_per_s, double* elapsed_ms) {
  if (!ctx || !ops_per_s || iters <= 0) return ECG_EINVAL;
  DevState& d = ctx->devs[0];
  Lane& L = d.lane[0];
  CU_TRY(ctx, cudaSetDevice(d.dev));
  ST_TRY(ensure(ctx, L, B_AUX, 256));
  uint32_t* out = (uint32_t*)L.buf[B_AUX];
  unsigned blocks = (unsigned)d.sm_count * 8, threads = 256;
  double per_thread_iter = 0;
  cudaEvent_t e0, e1;
  CU_TRY(ctx, cudaEventCreate(&e0));
  CU_TRY(ctx, cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {  // rep 0 = warm-up
    CU_TRY(ctx, cudaEventRecord(e0, L.s()));
    switch (which) {
      case 0: mb_imad_wide_kernel<<<blocks, threads, 0, L.s()>>>(out, iters, 12345u + rep); per_thread_iter = 32; break;
      case 1: mb_imad_kernel<<<blocks, threads, 0, L.s()>>>(out, iters, 12345u + rep); per_thread_iter = 64; break;
      case 2: mb_iadd_kernel<<<blocks, threads, 0, L.s()>>>(out, iters, 12345u + rep); per_thread_iter = 64; break;
      case 3: mb_fmul_kernel<FpK256><<<blocks, threads, 0, L.s()>>>(out, iters, 12345u + rep); per_thread_iter = 2; break;
      case 4: mb_fmul_kernel<FpP256><<<blocks, threads, 0, L.s()>>>(out, iters, 12345u + rep); per_thread_iter = 2; break;
      default:
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        return ECG_EINVAL;
    }
    ctx->launches++;
    CU_TRY(ctx, cudaEventRecord(e1, L.s()));
    CU_TRY(ctx, cudaEventSynchronize(e1));
    CU_TRY(ctx, cudaGetLastError());
    float ms = 0;
    CU_TRY(ctx, cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ops_per_s = (double)blocks * threads * (double)iters * per_thread_iter / (best * 1e-3);
  if (elapsed_ms) *elapsed_ms = best;
  return ECG_OK;
}
#endif  // ECG_TU == 0
