// Shared helpers for the csg2im sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#ifndef CSG_API
#define CSG_API extern "C" __attribute__((visibility("default")))
#endif

// Thread-local error text returned by csg_last_error(); no exception crosses the C ABI.
void csg_set_error(const char* fmt, ...);

#define CSG_REQUIRE(cond, ...)            \
  do {                                    \
    if (!(cond)) {                        \
      csg_set_error(__VA_ARGS__);         \
      return 1;                           \
    }                                     \
  } while (0)

// Launch errors are checked immediately (no deferred sync), SURVEY.md §8(b).
void csg_count_launch();
#define CSG_CHECK_LAUNCH(name)                                                      \
  do {                                                                              \
    csg_count_launch();                                                             \
    cudaError_t e__ = cudaGetLastError();                                           \
    if (e__ != cudaSuccess) {                                                       \
      csg_set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__));   \
      return 2;                                                                     \
    }                                                                               \
  } while (0)

#define CSG_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      csg_set_error("%s failed: %s", #call, cudaGetErrorString(e__));               \
      return 2;                                                                     \
    }                                                                               \
  } while (0)

// Optional live timing of kernel classes (csg_prof_enable / csg_prof_collect): CUDA events recorded on the
// launching stream around the launches of one entry point.  Disabled = one relaxed load per call.
struct CsgProfScope {
  int slot;
  cudaStream_t stream;
  CsgProfScope(int cls, double work, cudaStream_t s);
  ~CsgProfScope();
};
enum { CSG_PROF_GEMM_BF16 = 0, CSG_PROF_GEMM_F32 = 1, CSG_PROF_LAYOUT_FWD = 2, CSG_PROF_LAYOUT_BWD = 3,
       CSG_PROF_POOL = 4, CSG_PROF_ASSEMBLE = 5, CSG_PROF_CANON = 6, CSG_PROF_CLASSES = 8 };

static inline int csg_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// Programmatic dependent launch (PDL): a kernel launched through csg_launch_pdl may be scheduled while the previous
// kernel of the stream is still draining; it must execute CSG_PDL_WAIT() before its first global-memory access (a
// no-op when the kernel was launched the ordinary way).  Hides ~1-2 us of launch latency per kernel in the ~200-launch
// training step.
#define CSG_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
template <typename... KArgs, typename... Args>
static inline cudaError_t csg_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                         Args... args) {
  cudaLaunchConfig_t cfg;
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int csg_num_sms();   // SM count of the current device (cached per device)

// Asynchronous index-error record (api.cu): pinned, device-mapped {code, row, value, limit}; NULL if unavailable.
int* csg_async_err_ptr();
enum { CSG_ERR_TRIPLE_OBJECT = 1, CSG_ERR_TRIPLE_PREDICATE = 2, CSG_ERR_EMBED_ID = 3, CSG_ERR_CANON_TRIPLET = 4 };
__device__ __forceinline__ void csg_report_index(int* rec, int code, long long row, long long value, long long limit) {
  if (!rec) return;
  volatile int* v = rec;       // plain stores: concurrent offenders race, any one of them is a valid report
  v[1] = (int)row; v[2] = (int)value; v[3] = (int)limit;
  __threadfence_system();
  v[0] = code;
}

__device__ __forceinline__ float4 ld_f4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st_f4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// streaming (evict-first) 128-bit store: canvas tiles are written once and not re-read by the writer
__device__ __forceinline__ void st_f4_stream(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }
__device__ __forceinline__ float4 ld_f4_stream(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }

// s = p[0] + p[stride] + ... + p[(n-1)*stride] in exactly that order, with the loads issued U at a time (the ordered
// "final" passes of the deterministic reductions are latency-bound on their dependent load -> add chain otherwise)
template <int U>
__device__ __forceinline__ float ordered_sum(const float* __restrict__ p, size_t stride, int n) {
  float s = 0.f;
  int b = 0;
  for (; b + U <= n; b += U) {
    float x[U];
#pragma unroll
    for (int i = 0; i < U; ++i) x[i] = p[(size_t)(b + i) * stride];
#pragma unroll
    for (int i = 0; i < U; ++i) s += x[i];
  }
  for (; b < n; ++b) s += p[(size_t)b * stride];
  return s;
}

// ---- 16-bit activation formats of the tensor-core engine: bf16 or fp16, chosen per tensor (fp16 carries the forward
// activations / weights: 11 significant bits instead of 8 at the same tcgen05 kind::f16 rate; bf16 carries the
// gradients, whose range fp16 cannot hold).  Eight packed values <-> floats.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
__device__ __forceinline__ void unpack8_16(const uint4& u, float (&f)[8], bool fp16) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
  if (fp16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 x = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      f[2 * i] = x.x; f[2 * i + 1] = x.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    }
  }
}
__device__ __forceinline__ uint32_t pack2_16(float a, float b, bool fp16) {
  if (fp16) {      // saturating: an activation beyond +-65504 must not become inf
    __half2 h = __floats2half2_rn(fminf(fmaxf(a, -65504.f), 65504.f), fminf(fmaxf(b, -65504.f), 65504.f));
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8_16(const float (&f)[8], bool fp16) {
  uint4 u;
  u.x = pack2_16(f[0], f[1], fp16); u.y = pack2_16(f[2], f[3], fp16);
  u.z = pack2_16(f[4], f[5], fp16); u.w = pack2_16(f[6], f[7], fp16);
  return u;
}
__device__ __forceinline__ unsigned short cvt16(float a, bool fp16) {
  if (fp16) { __half h = __float2half_rn(fminf(fmaxf(a, -65504.f), 65504.f)); return *reinterpret_cast<unsigned short*>(&h); }
  __nv_bfloat16 h = __float2bfloat16_rn(a);
  return *reinterpret_cast<unsigned short*>(&h);
}
// x > 0 for either format: sign bit clear and magnitude non-zero
__device__ __forceinline__ bool pos16(uint32_t h) { return h != 0 && h < 0x8000u; }

// ---- element access of the layout canvas and its gradient: float, __nv_bfloat16 or __half.  The 16-bit stores round
// once to nearest even WITHOUT saturation (unlike pack2_16 / cvt16): the canvas is "the fp32 result, rounded", as
// Tensor.to(dtype) rounds it -- fp16 overflow is +-inf and NaN stays NaN.  Loads widen exactly.
__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float to_f32(__half x) { return __half2float(x); }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
template <> __device__ __forceinline__ __half from_f32<__half>(float x) { return __float2half_rn(x); }
__device__ __forceinline__ uint32_t pack2_rn(float a, float b, __nv_bfloat16*) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack2_rn(float a, float b, __half*) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
// streaming store of 4 consecutive elements (16 B for fp32, 8 B for 16-bit; p aligned to that)
__device__ __forceinline__ void st4_stream(float* p, float a, float b, float c, float d) { st_f4_stream(p, make_float4(a, b, c, d)); }
template <typename T>
__device__ __forceinline__ void st4_stream(T* p, float a, float b, float c, float d) {
  __stcs(reinterpret_cast<uint2*>(p), make_uint2(pack2_rn(a, b, (T*)nullptr), pack2_rn(c, d, (T*)nullptr)));
}
// 8 consecutive elements widened to fp32 (32 B for fp32 = two 16-B loads, 16 B for 16-bit = one; p aligned to 16 B)
__device__ __forceinline__ void ld8_f32(const float* p, float (&f)[8]) {
  const float4 a = ld_f4(p), b = ld_f4(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
__device__ __forceinline__ void ld8_f32(const __half* p, float (&f)[8]) { unpack8_16(*reinterpret_cast<const uint4*>(p), f, true); }
__device__ __forceinline__ void ld8_f32(const __nv_bfloat16* p, float (&f)[8]) {
  unpack8_16(*reinterpret_cast<const uint4*>(p), f, false);
}

// Calls f with a null pointer of the element type selected by fmt (0 fp32, 1 bf16, 2 fp16 -- the format codes of the
// entry points that take any of the three), so one launch site covers every format; any other code is an error.
#include <type_traits>
template <typename F>
static inline int csg_with_format(int fmt, F&& f) {
  switch (fmt) {
    case 0: return f((float*)nullptr);
    case 1: return f((__nv_bfloat16*)nullptr);
    case 2: return f((__half*)nullptr);
  }
  csg_set_error("element format %d is not 0 (fp32), 1 (bf16) or 2 (fp16)", fmt);
  return 1;
}
template <typename P> using csg_elem_t = std::remove_pointer_t<P>;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
