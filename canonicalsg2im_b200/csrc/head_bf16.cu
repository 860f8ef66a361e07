// Narrow output head of box_net (sg2im/model.py:58-60: Linear(D, H) -> ReLU -> Linear(H, 4)) for the bf16 engine.
// The wide first layer runs on the tcgen05 GEMMs; the 4-wide second layer is far below any GEMM tile, so it is a
// row-dot kernel forward and one fused kernel backward:
//   csg_head_fwd   y[r, j] = sum_k h[r, k] * w[j, k] + b[j]                       (h bf16, w / b / y fp32, j < NOUT <= 8)
//   csg_head_bwd   dh[r, k] = (h[r, k] > 0) * sum_j dy[r, j] * w[j, k]  (bf16, ReLU of the first layer folded in),
//                  dw[j, k] = sum_r dy[r, j] * h[r, k],  db[j] = sum_r dy[r, j]  (per-block partials summed in block
//                  order by a second kernel: deterministic)
// The same kernels, templated on the element type of h / dh (fp32, bf16, fp16) and with an optional sigmoid, are the
// 1x1 output convolution of the mask head (sg2im/model.py:62-75, mask_size > 0): csg_head_fwd_ex / csg_head_bwd_ex.
//   sigmoid:  y = sigmoid(h w^T + b) forward; backward takes y and folds sigmoid' = y (1 - y) into dy
#include "common.cuh"
#include <cuda_bf16.h>

namespace {

constexpr int HEAD_MAX_OUT = 8;
constexpr int HB_ROWS = 32;            // rows per block of the backward kernel

__device__ __forceinline__ float2 ld2_f32(const float* p) { return *reinterpret_cast<const float2*>(p); }
__device__ __forceinline__ float2 ld2_f32(const __nv_bfloat16* p) { return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p)); }
__device__ __forceinline__ float2 ld2_f32(const __half* p) { return __half22float2(*reinterpret_cast<const __half2*>(p)); }

template <typename TH, bool SIGMOID>
__global__ void __launch_bounds__(256) head_fwd_kernel(const TH* __restrict__ h, int ldh, const float* __restrict__ w,
                                                       const float* __restrict__ b, int M, int K, int NOUT,
                                                       float* __restrict__ y) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) float ws[];          // [NOUT][K]
  for (int i = threadIdx.x; i < NOUT * K; i += blockDim.x) ws[i] = w[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = blockIdx.x * 8 + warp; r < M; r += gridDim.x * 8) {
    float acc[HEAD_MAX_OUT];
#pragma unroll
    for (int j = 0; j < HEAD_MAX_OUT; ++j) acc[j] = 0.f;
    for (int k = lane * 2; k < K; k += 64) {
      const float2 x = ld2_f32(h + (size_t)r * ldh + k);
#pragma unroll
      for (int j = 0; j < HEAD_MAX_OUT; ++j)
        if (j < NOUT) acc[j] = fmaf(x.y, ws[j * K + k + 1], fmaf(x.x, ws[j * K + k], acc[j]));
    }
#pragma unroll
    for (int j = 0; j < HEAD_MAX_OUT; ++j)
      if (j < NOUT) {
        const float v = warp_sum(acc[j]);
        if (lane == 0) y[(size_t)r * NOUT + j] = SIGMOID ? 1.f / (1.f + expf(-(v + b[j]))) : v + b[j];
      }
  }
}

// thread = column k; a block walks HB_ROWS rows.  ysig (may be NULL): the sigmoid outputs, dy *= ysig (1 - ysig).
// relu: h is the output of a ReLU and dh takes its mask (h > 0); otherwise dh = dy w everywhere
template <typename TH, typename TD>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ ysig,
                                                       const TH* __restrict__ h, int ldh,
                                                       const float* __restrict__ w, int M, int K, int NOUT,
                                                       TD* __restrict__ dh, int lddh, float* __restrict__ partial,
                                                       bool relu) {
  CSG_PDL_WAIT();
  __shared__ float sdy[HB_ROWS][HEAD_MAX_OUT];
  const int r0 = blockIdx.x * HB_ROWS, nr = min(HB_ROWS, M - r0);
  for (int i = threadIdx.x; i < HB_ROWS * HEAD_MAX_OUT; i += blockDim.x) {
    const int r = i / HEAD_MAX_OUT, j = i % HEAD_MAX_OUT;
    float d = 0.f;
    if (r < nr && j < NOUT) {
      const size_t e = (size_t)(r0 + r) * NOUT + j;
      d = dy[e];
      if (ysig) d *= ysig[e] * (1.f - ysig[e]);
    }
    sdy[r][j] = d;
  }
  __syncthreads();
  float* out = partial + (size_t)blockIdx.x * (NOUT * K + HEAD_MAX_OUT);
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float wk[HEAD_MAX_OUT], acc[HEAD_MAX_OUT];
#pragma unroll
    for (int j = 0; j < HEAD_MAX_OUT; ++j) {
      wk[j] = j < NOUT ? w[(size_t)j * K + k] : 0.f;
      acc[j] = 0.f;
    }
    for (int r = 0; r < nr; ++r) {
      const float hv = to_f32(h[(size_t)(r0 + r) * ldh + k]);
      float g = 0.f;
#pragma unroll
      for (int j = 0; j < HEAD_MAX_OUT; ++j) {
        g = fmaf(sdy[r][j], wk[j], g);
        acc[j] = fmaf(sdy[r][j], hv, acc[j]);
      }
      dh[(size_t)(r0 + r) * lddh + k] = from_f32<TD>(hv > 0.f || !relu ? g : 0.f);
    }
#pragma unroll
    for (int j = 0; j < HEAD_MAX_OUT; ++j)
      if (j < NOUT) out[(size_t)j * K + k] = acc[j];
  }
  if (threadIdx.x < HEAD_MAX_OUT) {
    float sdb = 0.f;
    for (int r = 0; r < nr; ++r) sdb += sdy[r][threadIdx.x];
    out[(size_t)NOUT * K + threadIdx.x] = sdb;
  }
}

__global__ void head_bwd_final_kernel(const float* __restrict__ partial, int blocks, int K, int NOUT, float* __restrict__ dw,
                                      float* __restrict__ db) {
  CSG_PDL_WAIT();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int cells = NOUT * K + HEAD_MAX_OUT;
  if (i >= cells) return;
  const float a = ordered_sum<16>(partial + i, (size_t)cells, blocks);
  if (i < NOUT * K) dw[i] = a;
  else if (i - NOUT * K < NOUT) db[i - NOUT * K] = a;
}

// out[g][i] = sum of partial[g*HB_GROUP .. min(blocks, (g+1)*HB_GROUP))[i] in block order: the first level of a two-level
// ordered reduction when the backward runs on many blocks (the mask head: one row per output pixel)
constexpr int HB_GROUP = 64;
__global__ void head_bwd_group_kernel(const float* __restrict__ partial, int blocks, int cells, float* __restrict__ out) {
  CSG_PDL_WAIT();
  const int i = blockIdx.x * blockDim.x + threadIdx.x, g = blockIdx.y;
  if (i >= cells) return;
  const int b0 = g * HB_GROUP;
  out[(size_t)g * cells + i] = ordered_sum<16>(partial + (size_t)b0 * cells + i, (size_t)cells, min(HB_GROUP, blocks - b0));
}

// Launch sequences shared by the box head's entry points (bf16 / fp16 h, no sigmoid, one ordered reduction level) and the
// general ones (any format, optional sigmoid, two levels beyond HB_GROUP row blocks).
int head_fwd_launch(const void* h, int ldh, int h_fmt, const float* w, const float* b, int M, int K, int nout, bool sigmoid,
                    float* y, cudaStream_t stream) {
  if (M == 0) return 0;
  CSG_REQUIRE(nout >= 1 && nout <= HEAD_MAX_OUT && K > 0 && (K & 1) == 0 && (ldh & 1) == 0,
              "head_fwd: nout=%d must be in [1, 8], K=%d and ldh=%d even", nout, K, ldh);
  const size_t smem = (size_t)nout * K * sizeof(float);
  CSG_REQUIRE(smem <= 48 * 1024, "head_fwd: weight [%d, %d] does not fit shared memory", nout, K);
  int blocks = csg_div_up(M, 8);
  if (blocks > 4 * csg_num_sms()) blocks = 4 * csg_num_sms();
  return csg_with_format(h_fmt, [&](auto* tag) -> int {
    using TH = csg_elem_t<decltype(tag)>;
    const TH* hp = reinterpret_cast<const TH*>(h);
    if (sigmoid) CSG_CUDA(csg_launch_pdl(head_fwd_kernel<TH, true>, dim3(blocks), dim3(256), smem, stream, hp, ldh, w, b, M, K, nout, y));
    else CSG_CUDA(csg_launch_pdl(head_fwd_kernel<TH, false>, dim3(blocks), dim3(256), smem, stream, hp, ldh, w, b, M, K, nout, y));
    CSG_CHECK_LAUNCH("csg_head_fwd");
    return 0;
  });
}

size_t head_bwd_workspace(int M, int K, int nout, bool two_level) {
  const size_t blocks = csg_div_up(M > 0 ? M : 1, HB_ROWS), cells = (size_t)nout * K + HEAD_MAX_OUT;
  return (blocks + (two_level ? (blocks + HB_GROUP - 1) / HB_GROUP : 0)) * cells * sizeof(float) + 256;
}

int head_bwd_launch(const float* dy, const float* ysig, const void* h, int ldh, int h_fmt, const float* w, int M, int K,
                    int nout, void* dh, int lddh, int dh_fmt, bool relu, float* dw, float* db, bool two_level,
                    void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CSG_REQUIRE(nout >= 1 && nout <= HEAD_MAX_OUT && K > 0, "head_bwd: nout=%d must be in [1, 8]", nout);
  if (M == 0) {
    CSG_CUDA(cudaMemsetAsync(dw, 0, (size_t)nout * K * sizeof(float), stream));
    CSG_CUDA(cudaMemsetAsync(db, 0, (size_t)nout * sizeof(float), stream));
    return 0;
  }
  CSG_REQUIRE(workspace && workspace_bytes >= head_bwd_workspace(M, K, nout, two_level), "head_bwd: workspace too small");
  int blocks = csg_div_up(M, HB_ROWS);
  const int cells = nout * K + HEAD_MAX_OUT;
  float* partial = reinterpret_cast<float*>(workspace);
  int rc = csg_with_format(h_fmt, [&](auto* htag) -> int {
    using TH = csg_elem_t<decltype(htag)>;
    return csg_with_format(dh_fmt, [&](auto* dtag) -> int {
      using TD = csg_elem_t<decltype(dtag)>;
      CSG_CUDA(csg_launch_pdl(head_bwd_kernel<TH, TD>, dim3(blocks), dim3(256), 0, stream, dy, ysig, reinterpret_cast<const TH*>(h),
                              ldh, w, M, K, nout, reinterpret_cast<TD*>(dh), lddh, partial, relu));
      CSG_CHECK_LAUNCH("csg_head_bwd");
      return 0;
    });
  });
  if (rc) return rc;
  if (two_level && blocks > HB_GROUP) {
    const int groups = csg_div_up(blocks, HB_GROUP);
    float* grouped = partial + (size_t)blocks * cells;
    CSG_CUDA(csg_launch_pdl(head_bwd_group_kernel, dim3(csg_div_up(cells, 256), groups), dim3(256), 0, stream,
                            (const float*)partial, blocks, cells, grouped));
    CSG_CHECK_LAUNCH("csg_head_bwd group");
    partial = grouped;
    blocks = groups;
  }
  CSG_CUDA(csg_launch_pdl(head_bwd_final_kernel, dim3(csg_div_up(cells, 256)), dim3(256), 0, stream, (const float*)partial,
                          blocks, K, nout, dw, db));
  CSG_CHECK_LAUNCH("csg_head_bwd final");
  return 0;
}

}  // namespace

CSG_API int csg_head_fwd(const void* h, int ldh, const float* w, const float* b, int M, int K, int nout, float* y,
                         int h_fp16, cudaStream_t stream) {
  return head_fwd_launch(h, ldh, h_fp16 ? 2 : 1, w, b, M, K, nout, false, y, stream);
}

CSG_API size_t csg_head_bwd_workspace(int M, int K, int nout) { return head_bwd_workspace(M, K, nout, false); }

// dh [M, K] bf16 (pitch lddh), dw [nout, K] fp32, db [nout] fp32 are fully written.  One ordered reduction level over the
// row blocks, as the box head has always summed them.
CSG_API int csg_head_bwd(const float* dy, const void* h, int ldh, const float* w, int M, int K, int nout, void* dh, int lddh,
                         float* dw, float* db, int h_fp16, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return head_bwd_launch(dy, nullptr, h, ldh, h_fp16 ? 2 : 1, w, M, K, nout, dh, lddh, 1, true, dw, db, false, workspace,
                         workspace_bytes, stream);
}

CSG_API int csg_head_fwd_ex(const void* h, int ldh, int h_fmt, const float* w, const float* b, int M, int K, int nout,
                            int sigmoid, float* y, cudaStream_t stream) {
  return head_fwd_launch(h, ldh, h_fmt, w, b, M, K, nout, sigmoid != 0, y, stream);
}

CSG_API size_t csg_head_bwd_ex_workspace(int M, int K, int nout) { return head_bwd_workspace(M, K, nout, true); }

// dh is written in dh_fmt (0 fp32, 1 bf16, 2 fp16); more than HB_GROUP row blocks are reduced in two ordered levels
CSG_API int csg_head_bwd_ex(const float* dy, const float* y, const void* h, int ldh, int h_fmt, const float* w, int M, int K,
                            int nout, void* dh, int lddh, int dh_fmt, int relu, float* dw, float* db, void* workspace,
                            size_t workspace_bytes, cudaStream_t stream) {
  return head_bwd_launch(dy, y, h, ldh, h_fmt, w, M, K, nout, dh, lddh, dh_fmt, relu != 0, dw, db, true, workspace,
                         workspace_bytes, stream);
}
