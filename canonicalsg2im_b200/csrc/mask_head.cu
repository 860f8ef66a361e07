// Memory-bound kernels of the mask head of Sg2LayoutModel (sg2im/model.py:62-75, mask_size > 0):
//   per stage  Upsample(2, nearest) -> BatchNorm2d(C) -> Conv2d(C, C, 3, padding=1) -> ReLU,  then Conv2d(C, 1, 1) + sigmoid.
// Every convolution is a plain GEMM on the csg2im engines (csg_gemm_bf16 / csg_gemm_f32) over a patch matrix; the kernels
// here do everything around those GEMMs.  Activations are NHWC rows: a stage input of side s is x [O*s*s, C] with row
// (o*s + y)*s + x.
//
// Nearest upsampling copies every input pixel exactly four times, so the batch mean and biased variance of the
// upsampled tensor are those of the s x s input: BatchNorm is applied at low resolution and the (2s)^2 tensor is never
// materialised.  Only the unbiased correction of the running variance keeps the upsampled count 4n.
//   csg_mask_bn_fwd   per-channel batch statistics (shifted sums, fixed-order reduction) + running-buffer update, or the
//                     running buffers in eval mode -> mean, invstd and scale = gamma * invstd of the normalisation
//   csg_mask_patch    A[(o*S + Y)*S + X, c*9 + ky*3 + kx] = BN(x)[o, (Y+ky-1)/2, (X+kx-1)/2, c] inside the S x S = 2s x 2s
//                     image, 0 outside (the convolution's zero padding comes after BatchNorm): torch's own K order, so
//                     conv.weight.view(C, 9C) is the GEMM's B operand as it is
//   csg_mask_bn_bwd   G = the 2x2 block sums of the nine-tap adjoint of the patch map (fixed order, no atomics), then
//                     BatchNorm's backward at low resolution with the previous stage's ReLU mask folded in
#include "common.cuh"

namespace {

constexpr int MH_THREADS = 128;
constexpr int MH_STAT_ROWS = 256;      // rows per block of the statistics' partial sums (fixed: run-to-run identical)
constexpr int MH_BWD_ROWS = 32;        // low-resolution rows per block of the backward gather
constexpr int MH_PATCH_SMEM = 40 * 1024;

template <typename T> __device__ __forceinline__ float ldf(const T* p, size_t i) { return to_f32(p[i]); }

// part[b][0][c] = sum over the block's rows of (x - x[0, c]), part[b][1][c] = the same of its square.  Four accumulator
// pairs (rows r = 0, 1, 2, 3 mod 4) combined in a fixed order: deterministic, with four loads in flight per thread.
template <typename T>
__global__ void __launch_bounds__(MH_THREADS) bn_partial_kernel(const T* __restrict__ x, int n, int C, float* __restrict__ part) {
  CSG_PDL_WAIT();
  const int r0 = blockIdx.x * MH_STAT_ROWS, r1 = min(n, r0 + MH_STAT_ROWS);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float k = ldf(x, c);
    float s[4] = {0.f, 0.f, 0.f, 0.f}, q[4] = {0.f, 0.f, 0.f, 0.f};
    int r = r0;
    for (; r + 4 <= r1; r += 4) {
      float d[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) d[j] = ldf(x, (size_t)(r + j) * C + c) - k;
#pragma unroll
      for (int j = 0; j < 4; ++j) { s[j] += d[j]; q[j] = fmaf(d[j], d[j], q[j]); }
    }
    for (; r < r1; ++r) {          // at most 3 tail rows, into the first pair (a dynamic index would live on the stack)
      const float d = ldf(x, (size_t)r * C + c) - k;
      s[0] += d; q[0] = fmaf(d, d, q[0]);
    }
    part[(size_t)blockIdx.x * 2 * C + c] = (s[0] + s[1]) + (s[2] + s[3]);
    part[(size_t)blockIdx.x * 2 * C + C + c] = (q[0] + q[1]) + (q[2] + q[3]);
  }
}

// one thread per channel: batch statistics (training) or running buffers (eval) -> scale, mean, invstd
template <typename T>
__global__ void bn_final_kernel(const T* __restrict__ x, const float* __restrict__ part, int chunks, int n, int C,
                                const float* __restrict__ gamma, float* running_mean, float* running_var,
                                long long* num_batches, float momentum, float eps, int training, float* __restrict__ scale,
                                float* __restrict__ mean_out, float* __restrict__ invstd_out) {
  CSG_PDL_WAIT();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (training && c == 0 && num_batches) *num_batches += 1;
  if (c >= C || n == 0) return;
  float mean, var;
  if (training) {
    const float s = ordered_sum<8>(part + c, 2 * (size_t)C, chunks), q = ordered_sum<8>(part + C + c, 2 * (size_t)C, chunks);
    const float inv_n = 1.f / (float)n, md = s * inv_n;
    var = fmaxf(q * inv_n - md * md, 0.f);
    mean = ldf(x, c) + md;
    if (running_mean) {
      const float nu = 4.f * (float)n;       // element count of the upsampled tensor BatchNorm2d sees
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * (var * nu / (nu - 1.f));
    }
  } else {
    mean = running_mean[c];
    var = running_var[c];
  }
  const float inv = 1.f / sqrtf(var + eps);
  scale[c] = gamma[c] * inv;
  mean_out[c] = mean;
  invstd_out[c] = inv;
}

template <typename T> __device__ __forceinline__ void st_elem(T* p, float v) { *p = from_f32<T>(v); }

// A block owns `rb` consecutive output rows (one contiguous span of rb * 9C elements): a thread per channel writes the
// nine taps of its channel into shared memory, then the span is copied out with 16-byte stores.  BN(x) is evaluated as
// (x - mean) * scale + beta: with a near-zero batch variance scale is large, and x * scale + (beta - mean * scale) would
// lose beta to the rounding of the two large terms.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) patch_kernel(const TI* __restrict__ x, int O, int s, int C, const float* __restrict__ mean,
                                                    const float* __restrict__ scale, const float* __restrict__ beta,
                                                    TO* __restrict__ A, int rb) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TO* sm = reinterpret_cast<TO*>(smem_raw);
  const int S = 2 * s, K = 9 * C;
  const long long rows = (long long)O * S * S;
  for (long long row0 = (long long)blockIdx.x * rb; row0 < rows; row0 += (long long)gridDim.x * rb) {
    const int nr = (int)min((long long)rb, rows - row0);
    for (int i = threadIdx.x; i < nr * C; i += blockDim.x) {
      const int rr = i / C, c = i - rr * C;
      const long long row = row0 + rr;
      const int X = (int)(row % S), Y = (int)((row / S) % S);
      const long long o = row / ((long long)S * S);
      const float mu = mean[c], sc = scale[c], sh = beta[c];
      TO* dst = sm + (size_t)rr * K + c * 9;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int yy = Y + ky - 1;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int xx = X + kx - 1;
          float v = 0.f;
          if (yy >= 0 && yy < S && xx >= 0 && xx < S)
            v = fmaf(ldf(x, ((size_t)(o * s + (yy >> 1)) * s + (xx >> 1)) * C + c) - mu, sc, sh);
          st_elem(dst + ky * 3 + kx, v);
        }
      }
    }
    __syncthreads();
    const size_t nvec = (size_t)nr * K * sizeof(TO) / 16;
    uint4* out = reinterpret_cast<uint4*>(A + row0 * K);
    const uint4* src = reinterpret_cast<const uint4*>(sm);
    for (size_t i = threadIdx.x; i < nvec; i += blockDim.x) __stcs(out + i, src[i]);
    __syncthreads();
  }
}

// G[o, y, x, c] = sum over the 2x2 upsampled pixels (P, Q) of (y, x), in the order (0,0) (0,1) (1,0) (1,1), of
// sum over the taps (ky, kx) in row-major order of dA[(o, P - ky + 1, Q - kx + 1), c*9 + ky*3 + kx] (rows inside the
// image only) -- the adjoint of csg_mask_patch, each dA element read once.  The block also writes its per-channel partial
// sums of G and of G * xhat (xhat = (x - mean) * invstd), summed in row order.
template <typename TD, typename TX>
__global__ void __launch_bounds__(MH_THREADS) bn_bwd_gather_kernel(const TD* __restrict__ dA, const TX* __restrict__ x, int O, int s,
                                                                   int C, const float* __restrict__ mean,
                                                                   const float* __restrict__ invstd, float* __restrict__ G,
                                                                   float* __restrict__ part) {
  CSG_PDL_WAIT();
  const int S = 2 * s, K = 9 * C;
  const int n = O * s * s;
  const int r0 = blockIdx.x * MH_BWD_ROWS, r1 = min(n, r0 + MH_BWD_ROWS);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float mu = mean[c], inv = invstd[c];
    float sg = 0.f, sgx = 0.f;
    for (int r = r0; r < r1; ++r) {
      const int xl = r % s, yl = (r / s) % s, o = r / (s * s);
      float g = 0.f;
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const int P = 2 * yl + dy, Q = 2 * xl + dx;
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) {
            const int Y = P - ky + 1;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const int X = Q - kx + 1;
              if (Y >= 0 && Y < S && X >= 0 && X < S)
                g += ldf(dA, ((size_t)((size_t)o * S + Y) * S + X) * K + c * 9 + ky * 3 + kx);
            }
          }
        }
      G[(size_t)r * C + c] = g;
      const float xh = (ldf(x, (size_t)r * C + c) - mu) * inv;
      sg += g;
      sgx = fmaf(g, xh, sgx);
    }
    part[(size_t)blockIdx.x * 2 * C + c] = sg;
    part[(size_t)blockIdx.x * 2 * C + C + c] = sgx;
  }
}

__global__ void bn_bwd_final_kernel(const float* __restrict__ part, int chunks, int C, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta) {
  CSG_PDL_WAIT();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  dbeta[c] = ordered_sum<8>(part + c, 2 * (size_t)C, chunks);
  dgamma[c] = ordered_sum<8>(part + C + c, 2 * (size_t)C, chunks);
}

// dx = gamma * invstd * (G - (dbeta + xhat * dgamma) / n) (training) or gamma * invstd * G (eval), times (x > 0) when the
// input is the previous stage's ReLU output
template <typename TX, typename TO>
__global__ void __launch_bounds__(256) bn_bwd_dx_kernel(const float* __restrict__ G, const TX* __restrict__ x, int n, int C,
                                                        const float* __restrict__ gamma, const float* __restrict__ mean,
                                                        const float* __restrict__ invstd, const float* __restrict__ dgamma,
                                                        const float* __restrict__ dbeta, int training, int relu_mask,
                                                        TO* __restrict__ dx) {
  CSG_PDL_WAIT();
  const size_t total = (size_t)n * C;
  const float inv_n = 1.f / (float)n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const float xv = ldf(x, i), inv = invstd[c];
    float v = G[i];
    if (training) v -= (dbeta[c] + (xv - mean[c]) * inv * dgamma[c]) * inv_n;
    v *= gamma[c] * inv;
    if (relu_mask && !(xv > 0.f)) v = 0.f;
    st_elem(dx + i, v);
  }
}

size_t stat_chunks(int n) { return (size_t)csg_div_up(n, MH_STAT_ROWS); }
size_t bwd_chunks(int n) { return (size_t)csg_div_up(n, MH_BWD_ROWS); }
size_t align256(size_t b) { return (b + 255) / 256 * 256; }

}  // namespace

CSG_API size_t csg_mask_bn_fwd_workspace(int n, int C) {
  return align256(stat_chunks(n > 0 ? n : 1) * 2 * (size_t)C * sizeof(float));
}

CSG_API int csg_mask_bn_fwd(const void* x, int x_fmt, int n, int C, const float* gamma, float* running_mean,
                            float* running_var, long long* num_batches_tracked, double momentum, double eps, int training,
                            float* scale, float* mean, float* invstd, void* workspace, size_t workspace_bytes,
                            cudaStream_t stream) {
  CSG_REQUIRE(n >= 0 && C > 0, "mask_bn_fwd: bad sizes n=%d C=%d", n, C);
  CSG_REQUIRE(training || (running_mean && running_var), "mask_bn_fwd: eval mode needs the running buffers");
  CSG_REQUIRE(!training || n == 0 || (workspace && workspace_bytes >= csg_mask_bn_fwd_workspace(n, C)),
              "mask_bn_fwd: workspace too small");
  const int chunks = (int)stat_chunks(n);
  return csg_with_format(x_fmt, [&](auto* tag) -> int {
    using T = csg_elem_t<decltype(tag)>;
    const T* xp = reinterpret_cast<const T*>(x);
    float* part = reinterpret_cast<float*>(workspace);
    if (training && n > 0) {
      CSG_CUDA(csg_launch_pdl(bn_partial_kernel<T>, dim3(chunks), dim3(MH_THREADS), 0, stream, xp, n, C, part));
      CSG_CHECK_LAUNCH("csg_mask_bn_fwd partial");
    }
    if (n == 0 && !training) return 0;      // eval on an empty batch: nothing to compute, nothing to update
    CSG_CUDA(csg_launch_pdl(bn_final_kernel<T>, dim3(csg_div_up(C, MH_THREADS)), dim3(MH_THREADS), 0, stream, xp,
                            (const float*)part, chunks, n, C, gamma, running_mean, running_var, num_batches_tracked,
                            (float)momentum, (float)eps, training, scale, mean, invstd));
    CSG_CHECK_LAUNCH("csg_mask_bn_fwd final");
    return 0;
  });
}

CSG_API int csg_mask_patch(const void* x, int x_fmt, int O, int s, int C, const float* mean, const float* scale,
                           const float* beta, void* A, int a_fmt, cudaStream_t stream) {
  CSG_REQUIRE(O >= 0 && s > 0 && C > 0 && C % 8 == 0, "mask_patch: bad sizes O=%d s=%d C=%d (C must be a multiple of 8)",
              O, s, C);
  CSG_REQUIRE(((uintptr_t)A & 15) == 0, "mask_patch: A must be 16-byte aligned");
  if (O == 0) return 0;
  return csg_with_format(x_fmt, [&](auto* xtag) -> int {
    using TI = csg_elem_t<decltype(xtag)>;
    return csg_with_format(a_fmt, [&](auto* atag) -> int {
      using TO = csg_elem_t<decltype(atag)>;
      const size_t row_bytes = (size_t)9 * C * sizeof(TO);
      CSG_REQUIRE(row_bytes <= MH_PATCH_SMEM, "mask_patch: C=%d too wide for one row in shared memory", C);
      const int rb = (int)(MH_PATCH_SMEM / row_bytes < 8 ? MH_PATCH_SMEM / row_bytes : 8);
      const long long rows = (long long)O * 4 * s * s;
      long long blocks = (rows + rb - 1) / rb;
      if (blocks > 16ll * csg_num_sms()) blocks = 16ll * csg_num_sms();
      CSG_CUDA(csg_launch_pdl(patch_kernel<TI, TO>, dim3((unsigned)blocks), dim3(256), (size_t)rb * row_bytes, stream,
                              reinterpret_cast<const TI*>(x), O, s, C, mean, scale, beta, reinterpret_cast<TO*>(A), rb));
      CSG_CHECK_LAUNCH("csg_mask_patch");
      return 0;
    });
  });
}

CSG_API size_t csg_mask_bn_bwd_workspace(int n, int C) {
  const size_t nn = n > 0 ? n : 1;
  return align256(nn * C * sizeof(float)) + align256(bwd_chunks((int)nn) * 2 * (size_t)C * sizeof(float));
}

CSG_API int csg_mask_bn_bwd(const void* dA, int da_fmt, const void* x, int x_fmt, int O, int s, int C, const float* gamma,
                            const float* mean, const float* invstd, int training, int relu_mask, void* dx, int dx_fmt,
                            float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  CSG_REQUIRE(O >= 0 && s > 0 && C > 0, "mask_bn_bwd: bad sizes O=%d s=%d C=%d", O, s, C);
  const int n = O * s * s;
  if (n == 0) {
    CSG_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)C * sizeof(float), stream));
    CSG_CUDA(cudaMemsetAsync(dbeta, 0, (size_t)C * sizeof(float), stream));
    return 0;
  }
  CSG_REQUIRE(workspace && workspace_bytes >= csg_mask_bn_bwd_workspace(n, C), "mask_bn_bwd: workspace too small");
  float* G = reinterpret_cast<float*>(workspace);
  float* part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + align256((size_t)n * C * sizeof(float)));
  const int chunks = (int)bwd_chunks(n);
  return csg_with_format(x_fmt, [&](auto* xtag) -> int {
    using TX = csg_elem_t<decltype(xtag)>;
    const TX* xp = reinterpret_cast<const TX*>(x);
    int rc = csg_with_format(da_fmt, [&](auto* dtag) -> int {
      using TD = csg_elem_t<decltype(dtag)>;
      CSG_CUDA(csg_launch_pdl(bn_bwd_gather_kernel<TD, TX>, dim3(chunks), dim3(MH_THREADS), 0, stream,
                              reinterpret_cast<const TD*>(dA), xp, O, s, C, mean, invstd, G, part));
      CSG_CHECK_LAUNCH("csg_mask_bn_bwd gather");
      return 0;
    });
    if (rc) return rc;
    CSG_CUDA(csg_launch_pdl(bn_bwd_final_kernel, dim3(csg_div_up(C, MH_THREADS)), dim3(MH_THREADS), 0, stream,
                            (const float*)part, chunks, C, dgamma, dbeta));
    CSG_CHECK_LAUNCH("csg_mask_bn_bwd final");
    return csg_with_format(dx_fmt, [&](auto* otag) -> int {
      using TO = csg_elem_t<decltype(otag)>;
      long long blocks = ((long long)n * C + 255) / 256;
      if (blocks > 8ll * csg_num_sms()) blocks = 8ll * csg_num_sms();
      CSG_CUDA(csg_launch_pdl(bn_bwd_dx_kernel<TX, TO>, dim3((unsigned)blocks), dim3(256), 0, stream, (const float*)G, xp,
                              n, C, gamma, mean, invstd, (const float*)dgamma, (const float*)dbeta, training, relu_mask,
                              reinterpret_cast<TO*>(dx)));
      CSG_CHECK_LAUNCH("csg_mask_bn_bwd dx");
      return 0;
    });
  });
}
