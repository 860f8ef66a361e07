// Embedding lookups of Sg2LayoutModel.forward (sg2im/model.py:108-109, sg2im/attribute_embed.py:38-48) and the
// masked box regression loss that seeds the backward pass (sg2im/pix2pix_model.py:72-85), for sm_100a.
//
//   csg_embed_fwd   out[r, :] = table[idx[r], :]  written as fp32 or straight as bf16 (the operand type of the
//                   tensor-core GCN), so the [NT, E] fp32 predicate rows are never materialised;
//   csg_embed_bwd   dtable[v, :] = sum_{r: idx[r] = v} dout[r, :]  -- deterministic: every single-warp block walks a
//                   contiguous range of rows in order, accumulating into a private [V, E] table in shared memory;
//                   the per-block tables are then summed in block order (torch's embedding backward sorts the
//                   indices with a radix sort per call and accumulates with atomics);
//   csg_box_loss    per-image masked smooth-L1 box loss of the generator (bbox_pred_all / bbox_pred) and its gradient;
//   csg_mask_loss   binary cross-entropy mask loss of the generator (mean over every mask element) and its gradient.
#include "common.cuh"
#include <cuda_bf16.h>

namespace {

__device__ __forceinline__ float4 load_row4(const void* base, size_t elem, bool bf16) {
  if (bf16) {
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(base) + elem);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
    const float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
  }
  return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + elem);
}

// one warp per row, 4 columns per lane per step
__global__ void __launch_bounds__(256) embed_fwd_kernel(const float* __restrict__ table, const long long* __restrict__ idx,
                                                        long long idx_stride, int n, int V, int E,
                                                        void* __restrict__ out, int ld_out, int out_bf16, int* err) {
  CSG_PDL_WAIT();
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const int lane = threadIdx.x & 31;
  long long v = idx[(size_t)r * idx_stride];
  if (v < 0 || v >= V) {                             // nn.Embedding raises IndexError here: report, read row 0
    if (lane == 0) csg_report_index(err, CSG_ERR_EMBED_ID, r, v, V);
    v = 0;
  }
  const float* src = table + (size_t)v * E;
  for (int c = lane * 4; c < E; c += 128) {
    const float4 x = ld_f4(src + c);
    if (out_bf16) {      // 1 = bf16, 2 = fp16
      uint2 u;
      u.x = pack2_16(x.x, x.y, out_bf16 == 2);
      u.y = pack2_16(x.z, x.w, out_bf16 == 2);
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + (size_t)r * ld_out + c) = u;
    } else {
      st_f4(reinterpret_cast<float*>(out) + (size_t)r * ld_out + c, x);
    }
  }
}

// one-hot rows [n, ld] bf16 (ld >= V, a multiple of 8): row r is 1.0 at column idx[r] and 0 elsewhere.  With it the table
// gradient of a large bf16 lookup is the tensor-core product onehot^T dout (csg_gemm_bf16, mn_major): exact products,
// fp32 accumulation in a fixed split-K order, i.e. a deterministic segmented sum at GEMM speed.
__global__ void __launch_bounds__(256) onehot_bf16_kernel(const long long* __restrict__ idx, long long idx_stride, int n,
                                                          int V, int ld, uint4* __restrict__ out) {
  CSG_PDL_WAIT();
  const int per_row = ld >> 3;                                    // 16-byte pieces per row
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * per_row) return;
  const int r = (int)(i / per_row), c8 = (int)(i % per_row) * 8;
  const long long v = idx[(size_t)r * idx_stride];
  uint32_t w[4] = {0u, 0u, 0u, 0u};
  if (v >= c8 && v < c8 + 8 && v < V) {
    const int k = (int)(v - c8);
    w[k >> 1] = (k & 1) ? 0x3F800000u : 0x00003F80u;              // bf16 1.0 = 0x3F80
  }
  out[i] = make_uint4(w[0], w[1], w[2], w[3]);
}

constexpr int EB_UNROLL = 4;
// block b (one warp) owns rows [b * rows_per_block, ...) and vocabulary slice [v0, v0 + Vc)
__global__ void __launch_bounds__(32) embed_bwd_partial_kernel(const void* __restrict__ dout, int ld, int in_bf16,
                                                               const long long* __restrict__ idx, long long idx_stride,
                                                               int n, int rows_per_block, int v0, int Vc, int E,
                                                               float* __restrict__ partial) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) float acc[];     // [Vc][E]
  const int lane = threadIdx.x;
  for (int i = lane * 4; i < Vc * E; i += 128) st_f4(acc + i, make_float4(0.f, 0.f, 0.f, 0.f));
  __syncwarp();
  const int rbeg = blockIdx.x * rows_per_block, rend = min(rbeg + rows_per_block, n);
  for (int c = lane * 4; c < E; c += 128) {
    for (int r0 = rbeg; r0 < rend; r0 += EB_UNROLL) {
      float4 x[EB_UNROLL];
      int v[EB_UNROLL];
#pragma unroll
      for (int u = 0; u < EB_UNROLL; ++u) {
        const int r = r0 + u;
        v[u] = -1;
        x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < rend) {
          const long long vv = idx[(size_t)r * idx_stride] - v0;
          if (vv >= 0 && vv < Vc) {
            v[u] = (int)vv;
            x[u] = load_row4(dout, (size_t)r * ld + c, in_bf16 != 0);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < EB_UNROLL; ++u) {
        if (v[u] >= 0) {
          float* a = acc + (size_t)v[u] * E + c;
          float4 s = ld_f4(a);
          s.x += x[u].x; s.y += x[u].y; s.z += x[u].z; s.w += x[u].w;
          st_f4(a, s);
        }
      }
    }
  }
  __syncwarp();
  float* dst = partial + (size_t)blockIdx.x * Vc * E;
  for (int i = lane * 4; i < Vc * E; i += 128) st_f4(dst + i, ld_f4(acc + i));
}

__global__ void embed_bwd_final_kernel(const float* __restrict__ partial, int blocks, int cells, float* __restrict__ dtable) {
  CSG_PDL_WAIT();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cells) return;
  float a0 = 0.f, a1 = 0.f;
  int b = 0;
  for (; b + 1 < blocks; b += 2) {
    a0 += partial[(size_t)b * cells + i];
    a1 += partial[(size_t)(b + 1) * cells + i];
  }
  if (b < blocks) a0 += partial[(size_t)b * cells + i];
  dtable[i] = a0 + a1;
}

constexpr int EB_SMEM_MAX = 96 * 1024;
struct EbPlan { int Vc, blocks, rows_per_block; };
EbPlan embed_bwd_plan(int n, int V, int E) {
  EbPlan p;
  p.Vc = EB_SMEM_MAX / (E * 4);
  if (p.Vc > V) p.Vc = V;
  if (p.Vc < 1) p.Vc = 1;
  const int per_sm = (200 * 1024) / (p.Vc * E * 4 + 1024);
  int cap = csg_num_sms() * (per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm));
  int want = csg_div_up(n > 0 ? n : 1, 64);
  p.blocks = want < cap ? want : cap;
  p.rows_per_block = csg_div_up(n > 0 ? n : 1, p.blocks);
  p.rows_per_block = (p.rows_per_block + EB_UNROLL - 1) / EB_UNROLL * EB_UNROLL;
  p.blocks = csg_div_up(n > 0 ? n : 1, p.rows_per_block);
  return p;
}

__device__ __forceinline__ float block_sum_1024(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x < 32) {
    t = red[threadIdx.x];
    t = warp_sum(t);
    if (threadIdx.x == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

// pix2pix_model.py:72-85 on a flat batch.  One warp per image: count the real objects (objs != 0, or the sum of the
// attribute ids != 0 for multi-attribute objects), then loss_all[b] = weight * sum smooth_l1 / n_real and the gradient
// rows.  Lanes own rows b0 + lane, b0 + lane + 32, ...; the warp sums are xor trees, i.e. a fixed order.
constexpr int BL_WARPS = 8;
__global__ void __launch_bounds__(32 * BL_WARPS) box_loss_image_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                                     const long long* __restrict__ objs, int A,
                                                                     const int* __restrict__ obj_off, int B, float weight,
                                                                     float* __restrict__ loss_all, float* __restrict__ dpred) {
  CSG_PDL_WAIT();
  const int b = blockIdx.x * BL_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const int r0 = obj_off[b], r1 = obj_off[b + 1];
  auto is_real = [&](int r) {
    long long sum = 0;
    for (int k = 0; k < A; ++k) sum += objs[(size_t)r * A + k];
    return sum != 0;
  };
  float cnt = 0.f;
  for (int r = r0 + lane; r < r1; r += 32) cnt += is_real(r) ? 1.f : 0.f;
  cnt = warp_sum(cnt);
  const float inv = 1.f / cnt;                       // 0 real objects: 0 * inf = NaN below, as 0 / 0 in the reference
  const float gscale = weight * inv / (float)B;
  float sum = 0.f;
  for (int r = r0 + lane; r < r1; r += 32) {
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (is_real(r)) {
      const float4 g = ld_f4(gt + 4 * (size_t)r), p = ld_f4(pred + 4 * (size_t)r);
      const float d[4] = {p.x - g.x, p.y - g.y, p.z - g.z, p.w - g.w};
      float q[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float a = fabsf(d[k]);
        sum += a < 1.f ? 0.5f * d[k] * d[k] : a - 0.5f;
        q[k] = (a < 1.f ? d[k] : (d[k] > 0.f ? 1.f : -1.f)) * gscale;
      }
      o = make_float4(q[0], q[1], q[2], q[3]);
    }
    st_f4(dpred + 4 * (size_t)r, o);
  }
  sum = warp_sum(sum);
  if (lane == 0) loss_all[b] = weight * sum * inv;
}

// loss[0] = mean_b loss_all[b], summed in a fixed order (thread-strided partial sums, then a fixed tree)
__global__ void __launch_bounds__(1024) box_loss_mean_kernel(const float* __restrict__ loss_all, int B, float* __restrict__ loss) {
  CSG_PDL_WAIT();
  __shared__ float red[33];
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += 1024) s += loss_all[b];
  const float total = block_sum_1024(s, red);
  if (threadIdx.x == 0) loss[0] = total / (float)B;
}

// Mask term of the generator loss, weight * F.binary_cross_entropy(pred, target) (mean over all n elements), with
// torch's arithmetic: per element -(t max(log p, -100) + (1 - t) max(log(1 - p), -100)) written as torch's CPU kernel
// writes it, and d/dp = ((weight (p - t)) / max((1 - p) p, 1e-12)) / n, rounded step by step in the same order (the
// explicit _rn intrinsics keep nvcc from contracting them into FMAs), so a saturated p gives torch's bits: p == 1
// yields a finite d/dp that sigmoid' = 0 turns into an exact zero.  Block partials of the element losses in double, a
// fixed grid for a given n, one ordered final pass: two calls are bitwise equal.
constexpr int ML_THREADS = 256, ML_PER_THREAD = 8, ML_MAX_BLOCKS = 1024;
int mask_loss_blocks(long long n) {
  const long long b = (n + ML_THREADS * ML_PER_THREAD - 1) / (ML_THREADS * ML_PER_THREAD);
  return (int)(b < ML_MAX_BLOCKS ? b : ML_MAX_BLOCKS);
}

// std::max(a, b) = a < b ? b : a: a NaN first argument is returned (fmaxf would drop it)
__device__ __forceinline__ float std_max(float a, float b) { return a < b ? b : a; }

__device__ __forceinline__ double block_sum_double(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 32) {
    t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  return t;                                            // valid in thread 0
}

template <bool TARGET_I64>
__global__ void __launch_bounds__(ML_THREADS) mask_loss_partial_kernel(const float* __restrict__ pred,
                                                                      const void* __restrict__ target, long long n,
                                                                      float weight, float* __restrict__ dpred,
                                                                      double* __restrict__ partial) {
  CSG_PDL_WAIT();
  __shared__ double red[ML_THREADS / 32];
  const long long stride = (long long)gridDim.x * ML_THREADS;
  const float fn = (float)n;
  double s = 0.0;
  for (long long i0 = (long long)blockIdx.x * ML_THREADS + threadIdx.x; i0 < n; i0 += stride * ML_PER_THREAD) {
    float p[ML_PER_THREAD], t[ML_PER_THREAD];
#pragma unroll
    for (int k = 0; k < ML_PER_THREAD; ++k) {        // all loads in flight before the arithmetic
      const long long i = i0 + k * stride;
      p[k] = t[k] = 0.f;
      if (i < n) {
        p[k] = __ldcs(pred + i);
        t[k] = TARGET_I64 ? (float)__ldcs(static_cast<const long long*>(target) + i)
                          : __ldcs(static_cast<const float*>(target) + i);
      }
    }
#pragma unroll
    for (int k = 0; k < ML_PER_THREAD; ++k) {
      const long long i = i0 + k * stride;
      if (i < n) {
        const float l1 = std_max(log1pf(-p[k]), -100.f), l0 = std_max(logf(p[k]), -100.f);
        s += (double)__fsub_rn(__fmul_rn(__fsub_rn(t[k], 1.f), l1), __fmul_rn(t[k], l0));
        const float den = std_max(__fmul_rn(__fsub_rn(1.f, p[k]), p[k]), 1e-12f);
        __stcs(dpred + i, __fdiv_rn(__fdiv_rn(__fmul_rn(weight, __fsub_rn(p[k], t[k])), den), fn));
      }
    }
  }
  const double b = block_sum_double(s, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = b;
}

// loss[0] = weight * (sum of the block partials in block order / n); blocks == 0 (n == 0) reads nothing and gives 0 / 0
__global__ void __launch_bounds__(ML_MAX_BLOCKS) mask_loss_final_kernel(const double* __restrict__ partial, int blocks,
                                                                        long long n, float weight, float* __restrict__ loss) {
  CSG_PDL_WAIT();
  __shared__ double red[ML_MAX_BLOCKS / 32];
  const double v = (int)threadIdx.x < blocks ? partial[threadIdx.x] : 0.0;
  const double total = block_sum_double(v, red);
  if (threadIdx.x == 0) loss[0] = __fmul_rn((float)(total / (double)n), weight);
}

}  // namespace

CSG_API int csg_embed_fwd(const float* table, const long long* idx, long long idx_stride, int n, int V, int E,
                          void* out, int ld_out, int out_bf16, cudaStream_t stream) {
  if (n == 0) return 0;
  CSG_REQUIRE(V > 0 && E > 0 && (E & 3) == 0 && (ld_out & 3) == 0, "embed_fwd: E=%d / ld=%d must be multiples of 4", E, ld_out);
  CSG_CUDA(csg_launch_pdl(embed_fwd_kernel, dim3(csg_div_up((long long)n * 32, 256)), dim3(256), 0, stream, table, idx, idx_stride, n, V, E, out, ld_out,
                                                                          out_bf16, csg_async_err_ptr()));
  CSG_CHECK_LAUNCH("csg_embed_fwd");
  return 0;
}

CSG_API size_t csg_embed_bwd_workspace(int n, int V, int E) {
  const EbPlan p = embed_bwd_plan(n, V, E);
  return (size_t)p.blocks * p.Vc * E * sizeof(float) + 256;
}

// dtable [V, E] fp32 is fully written (rows of unused ids are zero).  dout: fp32 or bf16 rows with leading dimension ld.
CSG_API int csg_embed_bwd(const void* dout, int ld, int in_bf16, const long long* idx, long long idx_stride, int n,
                          int V, int E, float* dtable, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CSG_REQUIRE(V > 0 && E > 0 && (E & 3) == 0 && (ld & 3) == 0, "embed_bwd: E=%d / ld=%d must be multiples of 4", E, ld);
  CSG_REQUIRE(workspace_bytes >= csg_embed_bwd_workspace(n, V, E), "embed_bwd: workspace too small");
  if (n == 0) {
    CSG_CUDA(cudaMemsetAsync(dtable, 0, (size_t)V * E * sizeof(float), stream));
    return 0;
  }
  const EbPlan p = embed_bwd_plan(n, V, E);
  float* partial = reinterpret_cast<float*>(workspace);
  const size_t smem = (size_t)p.Vc * E * sizeof(float);
  CSG_CUDA(cudaFuncSetAttribute(embed_bwd_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (int v0 = 0; v0 < V; v0 += p.Vc) {
    const int vc = V - v0 < p.Vc ? V - v0 : p.Vc;
    CSG_CUDA(csg_launch_pdl(embed_bwd_partial_kernel, dim3(p.blocks), dim3(32), (size_t)vc * E * sizeof(float), stream, dout, ld, in_bf16, idx, idx_stride, n,
                                                                                      p.rows_per_block, v0, vc, E, partial));
    CSG_CHECK_LAUNCH("csg_embed_bwd partial");
    CSG_CUDA(csg_launch_pdl(embed_bwd_final_kernel, dim3(csg_div_up((long long)vc * E, 256)), dim3(256), 0, stream, partial, p.blocks, vc * E,
                                                                                  dtable + (size_t)v0 * E));
    CSG_CHECK_LAUNCH("csg_embed_bwd final");
  }
  return 0;
}

CSG_API int csg_onehot_bf16(const long long* idx, long long idx_stride, int n, int V, void* out, int ld,
                            cudaStream_t stream) {
  if (n == 0) return 0;
  CSG_REQUIRE(V > 0 && ld >= V && (ld & 7) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
              "onehot_bf16: ld=%d must be a multiple of 8 and >= V=%d, out 16-byte aligned", ld, V);
  const long long pieces = (long long)n * (ld >> 3);
  CSG_CUDA(csg_launch_pdl(onehot_bf16_kernel, dim3(csg_div_up(pieces, 256)), dim3(256), 0, stream, idx, idx_stride, n, V, ld, reinterpret_cast<uint4*>(out)));
  CSG_CHECK_LAUNCH("csg_onehot_bf16");
  return 0;
}

// Box regression term of the generator loss (pix2pix_model.py:72-85): loss_all[b] (G_losses["bbox_pred_all"]) =
// weight * sum over the real objects of image b of smooth_l1(pred - gt) / n_real(b); loss[0] (G_losses["bbox_pred"]) =
// mean_b loss_all[b]; dpred [NO, 4] = d loss[0] / d pred.  objs [NO, A] int64 class / attribute ids; a row is real iff
// its id (A == 1) or the sum of its ids (A > 1) is non-zero (the __image__ dummy and collate padding are 0).
CSG_API int csg_box_loss(const float* pred, const float* gt, const long long* objs, int A, const int* obj_off, int B,
                         double weight, float* loss, float* loss_all, float* dpred, cudaStream_t stream) {
  CSG_REQUIRE(B > 0 && A > 0, "box_loss: B=%d A=%d", B, A);
  CSG_CUDA(csg_launch_pdl(box_loss_image_kernel, dim3(csg_div_up(B, BL_WARPS)), dim3(32 * BL_WARPS), 0, stream, pred, gt, objs, A,
                          obj_off, B, (float)weight, loss_all, dpred));
  CSG_CHECK_LAUNCH("csg_box_loss image");
  CSG_CUDA(csg_launch_pdl(box_loss_mean_kernel, dim3(1), dim3(1024), 0, stream, (const float*)loss_all, B, loss));
  CSG_CHECK_LAUNCH("csg_box_loss mean");
  return 0;
}

CSG_API size_t csg_mask_loss_workspace(long long n) {
  return (size_t)(n > 0 ? mask_loss_blocks(n) : 0) * sizeof(double) + 256;
}

// Mask term of the generator loss (sg2im's compute_generator_loss): loss[0] = weight * F.binary_cross_entropy(pred,
// target), the mean over n elements, and dpred [n] = d loss[0] / d pred.  target_fmt 0: fp32 targets (soft targets in
// [0, 1] allowed), 1: int64.  n == 0: loss[0] = NaN (the mean of nothing) and nothing is read.
CSG_API int csg_mask_loss(const float* pred, const void* target, int target_fmt, long long n, double weight,
                          float* loss, float* dpred, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CSG_REQUIRE(n >= 0 && (target_fmt == 0 || target_fmt == 1), "mask_loss: n=%lld target_fmt=%d", n, target_fmt);
  CSG_REQUIRE(workspace_bytes >= csg_mask_loss_workspace(n), "mask_loss: workspace too small");
  double* partial = reinterpret_cast<double*>(workspace);
  const int blocks = n > 0 ? mask_loss_blocks(n) : 0;
  if (blocks > 0) {
    if (target_fmt == 1)
      CSG_CUDA(csg_launch_pdl(mask_loss_partial_kernel<true>, dim3(blocks), dim3(ML_THREADS), 0, stream, pred, target, n,
                              (float)weight, dpred, partial));
    else
      CSG_CUDA(csg_launch_pdl(mask_loss_partial_kernel<false>, dim3(blocks), dim3(ML_THREADS), 0, stream, pred, target,
                              n, (float)weight, dpred, partial));
    CSG_CHECK_LAUNCH("csg_mask_loss partial");
  }
  CSG_CUDA(csg_launch_pdl(mask_loss_final_kernel, dim3(1), dim3(ML_MAX_BLOCKS), 0, stream, (const double*)partial, blocks,
                          n, (float)weight, loss));
  CSG_CHECK_LAUNCH("csg_mask_loss final");
  return 0;
}
