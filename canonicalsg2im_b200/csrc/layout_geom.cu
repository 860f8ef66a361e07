// Layout compositor, the two secondary paths of sg2im/layout.py:
//
//   * test-mode occlusion compositor (masks_to_layout(test_mode=True), layout.py:72-76 + _pool_mask_samples
//     :135-147): objects are visited in ascending order of their total sampled mass and the first one whose
//     clean mask sample exceeds 0.5 owns the pixel.  Two launches: (1) per image, the mass of every object in
//     closed form and its rank; (2) a tiled single-pass compositor that finds the owner of each pixel and writes
//     every canvas element exactly once.  No host synchronisation (the reference calls .item() per object).
//   * gradients wrt boxes and (float) masks (autograd through F.grid_sample + _boxes_to_grid, layout.py:80-112):
//     one CTA per object walks the rows of its support, contracts the incoming gradient with the object's vector
//     once (g = sum_d dout * vec), and accumulates the box / mask-tap gradients in double in a fixed order.
//
// Both are HBM-light compared with the training compositor (layout.cu); they exist for completeness of the
// drop-in (inference canvases, box gradients), and are deterministic.  The predicted-mask training step takes d masks
// from the band-tiled kernel of layout.cu (csg_layout_bwd_vecs_masks), which falls back to this one on shapes the ring
// kernel does not serve.
#include "layout_common.cuh"

namespace {

constexpr int MAX_M = 64;   // mask resolution supported by these paths (shared-memory tables)

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// =====================================================================================================
// occlusion, pass 1: mass_j = sum_{d,y,x} vecs[j,d] * S_j(y,x) = (sum_d vecs[j,d]) * sum_{a,b} m[a,b] cy[a] cx[b]
// with cx[b] = sum_x (weight of mask column b at canvas column x); then order = argsort(mass) per image
// (ties by object index, NaN last as numpy does).
// =====================================================================================================
constexpr int ORD_WARPS = 8;

__global__ void __launch_bounds__(ORD_WARPS * 32) occlude_order_kernel(LayoutParams p, double* __restrict__ mass,
                                                                       int* __restrict__ order,
                                                                       int* __restrict__ img_flag) {
  __shared__ double cx[ORD_WARPS][MAX_M], cy[ORD_WARPS][MAX_M];
  __shared__ int s_flag;
  const int n = blockIdx.x;
  const int obeg = p.obj_off[n], oend = p.obj_off[n + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = p.M;
  if (threadIdx.x == 0) s_flag = 0;
  __syncthreads();
  for (int o = obeg + warp; o < oend; o += ORD_WARPS) {
    const float4 b = ld_f4(p.boxes + 4 * (size_t)o);
    if (box_poison(b)) { if (lane == 0) s_flag = 1; }
    for (int t = lane; t < S; t += 32) {
      double ax = 0.0, ay = 0.0;
      for (int x = 0; x < p.W; ++x) {
        const Tap tp = axis_tap(p.lin_x[x], b.x, b.z, S, p.align);
        if (tp.i0 == t) ax += (double)tp.w0; else if (tp.i0 + 1 == t) ax += (double)tp.w1;
      }
      for (int y = 0; y < p.H; ++y) {
        const Tap tp = axis_tap(p.lin_y[y], b.y, b.w, S, p.align);
        if (tp.i0 == t) ay += (double)tp.w0; else if (tp.i0 + 1 == t) ay += (double)tp.w1;
      }
      cx[warp][t] = ax; cy[warp][t] = ay;
    }
    __syncwarp();
    double ms = 0.0;
    const float* m = p.masks + (size_t)o * S * S;
    for (int i = lane; i < S * S; i += 32) ms += (double)m[i] * cy[warp][i / S] * cx[warp][i % S];
    ms = warp_sum_d(ms);
    double vs = 0.0;
    for (int d = lane; d < p.D; d += 32) vs += (double)p.vecs[(size_t)o * p.D + d];
    vs = warp_sum_d(vs);
    if (lane == 0) {
      double v = vs * ms;
      mass[o] = (v == v) ? v : INFINITY;
    }
    __syncwarp();
  }
  __syncthreads();
  for (int o = obeg + threadIdx.x; o < oend; o += blockDim.x) {
    const double mo = mass[o];
    int rank = 0;
    for (int q = obeg; q < oend; ++q) {
      const double mq = mass[q];
      rank += (mq < mo || (mq == mo && q < o)) ? 1 : 0;
    }
    order[obeg + rank] = o;
  }
  if (threadIdx.x == 0) img_flag[n] = s_flag;
}

// =====================================================================================================
// occlusion, pass 2: out[n, d, y, x] = vecs[j*, d] * S_j*(y, x),  j* = first object in `order` with S_j(y, x) > 0.5
// =====================================================================================================
namespace occ {
constexpr int TW = 64, TH = 8, NTHREADS = 128;

// T: canvas element type (float, __nv_bfloat16, __half); a 16-bit canvas is the fp32 one rounded once
template <typename T>
__global__ void __launch_bounds__(NTHREADS) layout_occlude_kernel(LayoutParams p, const int* __restrict__ order,
                                                                  const int* __restrict__ img_flag,
                                                                  T* __restrict__ out) {
  extern __shared__ __align__(16) float smem_raw[];
  __shared__ int s_cursor, s_count;
  float* cxs = smem_raw;                          // [lcap][TW] column sample coordinates
  float* cys = cxs + (size_t)p.lcap * TW;         // [lcap][TH]
  int* list = reinterpret_cast<int*>(cys + (size_t)p.lcap * TH);
  const int n = blockIdx.y;
  const int x0 = (blockIdx.x % p.tiles_x) * TW, y0 = (blockIdx.x / p.tiles_x) * TH;
  const int obeg = p.obj_off[n], oend = p.obj_off[n + 1];
  const int tid = threadIdx.x, lane = tid & 31;
  const int S = p.M;
  const int row = tid >> 4, col = (tid & 15) * 4;
  const int y = y0 + row, x = x0 + col;
  int win[4] = {-1, -1, -1, -1};
  float ww[4] = {0.f, 0.f, 0.f, 0.f};
  unsigned open = 0u;                             // pixels of this thread that have no owner yet
#pragma unroll
  for (int k = 0; k < 4; ++k) if (y < p.H && x + k < p.W) open |= 1u << k;
  const bool poisoned = img_flag[n] != 0;
  if (tid == 0) s_cursor = obeg;
  __syncthreads();
  while (!poisoned) {
    // objects, in compositing order, whose support may touch this tile
    if (tid < 32) {
      const float xlo = p.lin_x[x0], xhi = p.lin_x[min(x0 + TW, p.W) - 1];
      const float ylo = p.lin_y[y0], yhi = p.lin_y[min(y0 + TH, p.H) - 1];
      int cursor = s_cursor, count = 0;
      while (cursor < oend && count < p.lcap) {
        const int q = cursor + lane;
        bool keep = false;
        int o = -1;
        if (q < oend) {
          o = order[q];
          const float4 b = ld_f4(p.boxes + 4 * (size_t)o);
          keep = axis_may_touch(b.x, b.z, xlo, xhi, S, p.align) && axis_may_touch(b.y, b.w, ylo, yhi, S, p.align);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        const int pos = count + __popc(bal & ((1u << lane) - 1u));
        const int total = __popc(bal);
        if (total <= p.lcap - count) {
          if (keep) list[pos] = o;
          count += total;
          cursor += 32;
        } else {
          if (keep && pos < p.lcap) list[pos] = o;
          const unsigned last = __ballot_sync(0xffffffffu, keep && pos == p.lcap - 1);
          cursor += __ffs(last);
          count = p.lcap;
        }
      }
      if (lane == 0) { s_cursor = min(cursor, oend); s_count = count; }
    }
    __syncthreads();
    const int L = s_count;
    const bool more = s_cursor < oend;
    for (int i = tid; i < L * (TW + TH); i += NTHREADS) {
      const int c = i / (TW + TH);
      int r = i % (TW + TH);
      const float4 b = ld_f4(p.boxes + 4 * (size_t)list[c]);
      if (r < TW) {
        cxs[c * TW + r] = axis_coord(p.lin_x[min(x0 + r, p.W - 1)], b.x, b.z, S, p.align);
      } else {
        r -= TW;
        cys[c * TH + r] = axis_coord(p.lin_y[min(y0 + r, p.H - 1)], b.y, b.w, S, p.align);
      }
    }
    __syncthreads();
    for (int c = 0; c < L && open; ++c) {
      const int o = list[c];
      const Tap ty = coord_tap(cys[c * TH + row], S);
      if (ty.i0 < -1 || ty.i0 >= S) continue;
      const float* m = p.masks + (size_t)o * S * S;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (open & (1u << k)) {
          const float w = mask_weight(m, S, coord_tap(cxs[c * TW + col + k], S), ty);
          if (w > 0.5f) { win[k] = o; ww[k] = w; open &= ~(1u << k); }
        }
      }
    }
    __syncthreads();
    if (!more) break;
  }
  if (y >= p.H || x >= p.W) return;
  const bool vec4 = (p.W & 3) == 0;
  const float qnan = __int_as_float(0x7fc00000);
  for (int d0 = 0; d0 < p.D; d0 += 4) {
    float v[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (win[k] >= 0) t = ld_f4(p.vecs + (size_t)win[k] * p.D + d0);
      v[k][0] = t.x * ww[k]; v[k][1] = t.y * ww[k]; v[k][2] = t.z * ww[k]; v[k][3] = t.w * ww[k];
      if (poisoned) v[k][0] = v[k][1] = v[k][2] = v[k][3] = qnan;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      T* dst = out + (((size_t)n * p.D + d0 + j) * p.H + y) * p.W + x;
      if (vec4) {
        st4_stream(dst, v[0][j], v[1][j], v[2][j], v[3][j]);
      } else {
        for (int k = 0; k < 4 && x + k < p.W; ++k) dst[k] = from_f32<T>(v[k][j]);
      }
    }
  }
}

__host__ __device__ inline size_t smem_bytes(int lcap) { return (size_t)lcap * (TW + TH + 1) * 4; }
}  // namespace occ

// =====================================================================================================
// gradients wrt boxes and masks.  For object o of image n, with g(y, x) = sum_d dout[n, d, y, x] * vecs[o, d]:
//   dS/dix = (m_ne - m_nw) * wy0 + (m_se - m_sw) * wy1        (ATen grid_sampler_2d_backward, bilinear / zeros)
//   dS/diy = (m_sw - m_nw) * wx0 + (m_se - m_ne) * wx1
//   d ix / d gx = S / 2  (align_corners=False)  or  (S - 1) / 2;   gx = 2 u - 1;   u = (lin - x0) / w
//   dx0 = -(1/w) sum 2 k g dS/dix,   dw = -(1/w) sum 2 k g dS/dix * u           (and the same in y)
//   dmask[a, b] = sum_{y, x} g(y, x) * wy(y, a) * wx(x, b)
// m_* are the in-range mask values (1 inside the 8 x 8 constant image for boxes_to_layout).
// =====================================================================================================
namespace geom {
constexpr int NTHREADS = 256;
constexpr int RB = 8;      // canvas rows per pass

template <typename T>
struct Params {
  LayoutParams p;
  const T* dout;          // float, __nv_bfloat16 or __half: widened on load
  float* dboxes;    // [NO, 4]
  float* dmasks;    // [NO, M, M] or nullptr
  const int* obj_img;
  int NO;
};

struct Smem {
  float* cx;        // [W] column sample coordinate
  float* cy;        // [H]
  float* vec;       // [D]
  float* mask;      // [S*S] (boxes: unused)
  float* g;         // [RB][W]
  float* T;         // [RB][S]
  double* dm;       // [S*S]
  double* red;      // [NTHREADS/32][4]
  int* bx;          // [S][2] canvas-column range feeding mask column b
  int* rng;         // [4]
};

__host__ __device__ inline size_t smem_bytes(int D, int H, int W, int S) {
  size_t f = (size_t)W + H + D + (size_t)S * S + (size_t)RB * W + (size_t)RB * S;
  f = (f + 1) & ~(size_t)1;
  return f * 4 + ((size_t)S * S + (NTHREADS / 32) * 4) * 8 + ((size_t)2 * S + 4) * 4;
}

__device__ __forceinline__ Smem carve(float* base, int D, int H, int W, int S) {
  Smem s;
  s.cx = base; s.cy = s.cx + W; s.vec = s.cy + H; s.mask = s.vec + D;
  s.g = s.mask + (size_t)S * S; s.T = s.g + (size_t)RB * W;
  size_t f = (size_t)W + H + D + (size_t)S * S + (size_t)RB * W + (size_t)RB * S;
  f = (f + 1) & ~(size_t)1;
  s.dm = reinterpret_cast<double*>(base + f);
  s.red = s.dm + (size_t)S * S;
  s.bx = reinterpret_cast<int*>(s.red + (NTHREADS / 32) * 4);
  s.rng = s.bx + 2 * S;
  return s;
}

template <bool HAS_MASK, typename T>
__global__ void __launch_bounds__(NTHREADS) layout_bwd_geom_kernel(Params<T> q) {
  extern __shared__ __align__(16) float smem_raw[];
  const LayoutParams& p = q.p;
  const int S = HAS_MASK ? p.M : 8;
  const Smem s = carve(smem_raw, p.D, p.H, p.W, S);
  const int o = blockIdx.x, n = q.obj_img[o];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float4 b = ld_f4(p.boxes + 4 * (size_t)o);
  const bool poison = box_poison(b);
  const bool want_dm = HAS_MASK && q.dmasks != nullptr;

  for (int i = tid; i < p.D; i += NTHREADS) s.vec[i] = p.vecs[(size_t)o * p.D + i];
  if (HAS_MASK) for (int i = tid; i < S * S; i += NTHREADS) { s.mask[i] = p.masks[(size_t)o * S * S + i]; s.dm[i] = 0.0; }
  for (int i = tid; i < S; i += NTHREADS) { s.bx[2 * i] = p.W; s.bx[2 * i + 1] = -1; }
  if (tid == 0) { s.rng[0] = p.W; s.rng[1] = -1; s.rng[2] = p.H; s.rng[3] = -1; }
  __syncthreads();
  for (int i = tid; i < p.W + p.H; i += NTHREADS) {
    const bool isx = i < p.W;
    const int k = isx ? i : i - p.W;
    const float c = axis_coord((isx ? p.lin_x : p.lin_y)[k], isx ? b.x : b.y, isx ? b.z : b.w, S, p.align);
    (isx ? s.cx : s.cy)[k] = c;
    if (c >= -1.f && c < (float)S) {                     // some tap in range
      atomicMin(&s.rng[isx ? 0 : 2], k);
      atomicMax(&s.rng[isx ? 1 : 3], k);
      if (isx) {
        const Tap t = coord_tap(c, S);
        if (t.i0 >= 0 && t.i0 < S) { atomicMin(&s.bx[2 * t.i0], k); atomicMax(&s.bx[2 * t.i0 + 1], k); }
        if (t.i0 + 1 >= 0 && t.i0 + 1 < S) { atomicMin(&s.bx[2 * t.i0 + 2], k); atomicMax(&s.bx[2 * t.i0 + 3], k); }
      }
    }
  }
  __syncthreads();
  const int xlo = s.rng[0], xhi = s.rng[1], ylo = s.rng[2], yhi = s.rng[3];
  const int nx = xhi - xlo + 1;
  double ax0 = 0.0, axw = 0.0, ay0 = 0.0, ayh = 0.0;     // sums of g*dS/dix, g*dS/dix*u, g*dS/diy, g*dS/diy*v
  const size_t plane = (size_t)p.H * p.W;
  const T* dimg = q.dout + (size_t)n * p.D * plane;

  if (!poison && nx > 0) {
    for (int yb = ylo; yb <= yhi; yb += RB) {
      const int nr = min(RB, yhi - yb + 1);
      // g[r][x] = sum_d dout[n, d, yb + r, x] * vec[d]
      for (int i = tid; i < nr * nx; i += NTHREADS) {
        const int r = i / nx, xx = xlo + i % nx;
        const T* src = dimg + (size_t)(yb + r) * p.W + xx;
        float acc = 0.f;
        for (int d = 0; d < p.D; ++d) acc = fmaf(to_f32(__ldg(src + (size_t)d * plane)), s.vec[d], acc);
        s.g[r * p.W + xx] = acc;
      }
      __syncthreads();
      // coordinate gradients
      for (int i = tid; i < nr * nx; i += NTHREADS) {
        const int r = i / nx, xx = xlo + i % nx, yy = yb + r;
        const Tap tx = coord_tap(s.cx[xx], S), ty = coord_tap(s.cy[yy], S);
        const int ix = tx.i0, iy = ty.i0;
        const bool vx0 = ix >= 0 && ix < S, vx1 = ix >= -1 && ix < S - 1;
        const bool vy0 = iy >= 0 && iy < S, vy1 = iy >= -1 && iy < S - 1;
        float m00, m01, m10, m11;
        if (HAS_MASK) {
          m00 = (vy0 && vx0) ? s.mask[iy * S + ix] : 0.f;
          m01 = (vy0 && vx1) ? s.mask[iy * S + ix + 1] : 0.f;
          m10 = (vy1 && vx0) ? s.mask[(iy + 1) * S + ix] : 0.f;
          m11 = (vy1 && vx1) ? s.mask[(iy + 1) * S + ix + 1] : 0.f;
        } else {
          m00 = (vy0 && vx0) ? 1.f : 0.f; m01 = (vy0 && vx1) ? 1.f : 0.f;
          m10 = (vy1 && vx0) ? 1.f : 0.f; m11 = (vy1 && vx1) ? 1.f : 0.f;
        }
        const float gv = s.g[r * p.W + xx];
        const float sx = (m01 - m00) * ty.w0 + (m11 - m10) * ty.w1;
        const float sy = (m10 - m00) * tx.w0 + (m11 - m01) * tx.w1;
        const double gx = (double)gv * (double)sx, gy = (double)gv * (double)sy;
        const float u = __fdiv_rn(__fsub_rn(p.lin_x[xx], b.x), b.z), v = __fdiv_rn(__fsub_rn(p.lin_y[yy], b.y), b.w);
        ax0 += gx; axw += gx * (double)u; ay0 += gy; ayh += gy * (double)v;
      }
      if (want_dm) {
        // T[r][bcol] = sum_x g[r][x] * wx(x, bcol)
        for (int i = tid; i < nr * S; i += NTHREADS) {
          const int r = i / S, bc = i % S;
          float acc = 0.f;
          for (int xx = s.bx[2 * bc]; xx <= s.bx[2 * bc + 1]; ++xx) {
            const Tap tx = coord_tap(s.cx[xx], S);
            const float w = tx.i0 == bc ? tx.w0 : (tx.i0 + 1 == bc ? tx.w1 : 0.f);
            acc = fmaf(s.g[r * p.W + xx], w, acc);
          }
          s.T[r * S + bc] = acc;
        }
        __syncthreads();
        for (int i = tid; i < S * S; i += NTHREADS) {
          const int a = i / S, bc = i % S;
          double acc = 0.0;
          for (int r = 0; r < nr; ++r) {
            const Tap ty = coord_tap(s.cy[yb + r], S);
            const float w = ty.i0 == a ? ty.w0 : (ty.i0 + 1 == a ? ty.w1 : 0.f);
            acc += (double)w * (double)s.T[r * S + bc];
          }
          s.dm[i] += acc;
        }
      }
      __syncthreads();
    }
  }
  // block reduction of the four coordinate sums, fixed order
  ax0 = warp_sum_d(ax0); axw = warp_sum_d(axw); ay0 = warp_sum_d(ay0); ayh = warp_sum_d(ayh);
  if (lane == 0) { s.red[warp * 4] = ax0; s.red[warp * 4 + 1] = axw; s.red[warp * 4 + 2] = ay0; s.red[warp * 4 + 3] = ayh; }
  __syncthreads();
  if (tid < 4) {
    double t = 0.0;
    for (int w = 0; w < NTHREADS / 32; ++w) t += s.red[w * 4 + tid];
    const double mult = p.align ? (double)(S - 1) : (double)S;      // 2 * (d ix / d g)
    const double ext = (tid & 2) ? (double)b.w : (double)b.z;
    float r = (float)(-mult * t / ext);
    if (poison) r = __int_as_float(0x7fc00000);
    // order in memory: x0, y0, w, h
    const int slot = tid == 0 ? 0 : tid == 1 ? 2 : tid == 2 ? 1 : 3;
    q.dboxes[4 * (size_t)o + slot] = r;
  }
  if (want_dm)
    for (int i = tid; i < S * S; i += NTHREADS)
      q.dmasks[(size_t)o * S * S + i] = poison ? __int_as_float(0x7fc00000) : (float)s.dm[i];
}

__global__ void obj_img_kernel(const int* __restrict__ obj_off, int N, int* __restrict__ obj_img) {
  const int n = blockIdx.x;
  for (int o = obj_off[n] + threadIdx.x; o < obj_off[n + 1]; o += blockDim.x) obj_img[o] = n;
}
}  // namespace geom

int fill(LayoutParams& p, const float* vecs, const float* boxes, const float* masks, const int* obj_off,
         const float* lin_x, const float* lin_y, int N, int D, int H, int W, int M, int align) {
  CSG_REQUIRE(N >= 0 && D > 0 && H > 0 && W > 0, "layout: bad sizes N=%d D=%d H=%d W=%d", N, D, H, W);
  CSG_REQUIRE(masks == nullptr || (M > 0 && M <= MAX_M), "layout: mask size M=%d not in 1..%d", M, MAX_M);
  CSG_REQUIRE((D & 3) == 0, "layout: D=%d must be a multiple of 4", D);
  p.vecs = vecs; p.boxes = boxes; p.masks = masks; p.obj_off = obj_off; p.lin_x = lin_x; p.lin_y = lin_y;
  p.N = N; p.D = D; p.H = H; p.W = W; p.M = M; p.align = align;
  p.TW = occ::TW; p.TH = occ::TH; p.tiles_x = csg_div_up(W, occ::TW); p.tiles_y = csg_div_up(H, occ::TH);
  p.lcap = 0;
  return 0;
}

}  // namespace

// ----------------------------------------------------------------------------------------
// C ABI
// ----------------------------------------------------------------------------------------
CSG_API size_t csg_layout_occlude_workspace(int N, int NO) {
  return (size_t)NO * 8 + (size_t)NO * 4 + (size_t)(N + 1) * 4 + 64;
}

CSG_API size_t csg_layout_bwd_geom_workspace(int NO) { return (size_t)(NO + 1) * 4 + 64; }

namespace {
template <typename T>
int layout_occlude_fwd(const float* vecs, const float* boxes, const float* masks, const int* obj_off, const float* lin_x,
                       const float* lin_y, T* out, int N, int NO, int D, int H, int W, int M, int align_corners,
                       void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  LayoutParams p;
  if (int rc = fill(p, vecs, boxes, masks, obj_off, lin_x, lin_y, N, D, H, W, M, align_corners)) return rc;
  CSG_REQUIRE(masks != nullptr, "layout occlude: masks are required (test_mode is a masks_to_layout feature)");
  if (N == 0) return 0;
  CSG_REQUIRE(workspace_bytes >= csg_layout_occlude_workspace(N, NO), "layout occlude: workspace too small");
  CSG_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0,
              "layout occlude: out must be 16-byte and workspace 8-byte aligned");
  double* mass = reinterpret_cast<double*>(workspace);
  int* order = reinterpret_cast<int*>(mass + NO);
  int* flag = order + NO;
  occlude_order_kernel<<<N, ORD_WARPS * 32, 0, stream>>>(p, mass, order, flag);
  CSG_CHECK_LAUNCH("csg_layout_occlude_fwd order");
  p.lcap = 64;
  dim3 grid(p.tiles_x * p.tiles_y, N);
  occ::layout_occlude_kernel<T><<<grid, occ::NTHREADS, occ::smem_bytes(p.lcap), stream>>>(p, order, flag, out);
  CSG_CHECK_LAUNCH("csg_layout_occlude_fwd");
  return 0;
}

template <typename T>
int layout_bwd_geom(const T* dout, const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                    const float* lin_x, const float* lin_y, float* dboxes, float* dmasks, int N, int NO, int D, int H,
                    int W, int M, int align_corners, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  LayoutParams p;
  if (int rc = fill(p, vecs, boxes, masks, obj_off, lin_x, lin_y, N, D, H, W, M, align_corners)) return rc;
  if (N == 0 || NO == 0) return 0;
  CSG_REQUIRE(workspace_bytes >= csg_layout_bwd_geom_workspace(NO), "layout bwd geom: workspace too small");
  CSG_REQUIRE(dboxes != nullptr, "layout bwd geom: dboxes is required");
  geom::Params<T> q;
  q.p = p; q.dout = dout; q.dboxes = dboxes; q.dmasks = masks ? dmasks : nullptr; q.NO = NO;
  int* obj_img = reinterpret_cast<int*>(workspace);
  q.obj_img = obj_img;
  geom::obj_img_kernel<<<N, 64, 0, stream>>>(obj_off, N, obj_img);
  CSG_CHECK_LAUNCH("csg_layout_bwd_geom obj_img");
  const int S = masks ? M : 8;
  const size_t smem = geom::smem_bytes(D, H, W, S);
  CSG_REQUIRE(smem <= 220 * 1024, "layout bwd geom: D=%d H=%d W=%d M=%d need %zu bytes of shared memory", D, H, W, M, smem);
  if (masks) {
    CSG_CUDA(cudaFuncSetAttribute(geom::layout_bwd_geom_kernel<true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    geom::layout_bwd_geom_kernel<true, T><<<NO, geom::NTHREADS, smem, stream>>>(q);
  } else {
    CSG_CUDA(cudaFuncSetAttribute(geom::layout_bwd_geom_kernel<false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    geom::layout_bwd_geom_kernel<false, T><<<NO, geom::NTHREADS, smem, stream>>>(q);
  }
  CSG_CHECK_LAUNCH("csg_layout_bwd_geom");
  return 0;
}
}  // namespace

CSG_API int csg_layout_occlude_fwd(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                                   const float* lin_x, const float* lin_y, float* out, int N, int NO, int D, int H,
                                   int W, int M, int align_corners, void* workspace, size_t workspace_bytes,
                                   cudaStream_t stream) {
  return layout_occlude_fwd(vecs, boxes, masks, obj_off, lin_x, lin_y, out, N, NO, D, H, W, M, align_corners, workspace,
                            workspace_bytes, stream);
}

CSG_API int csg_layout_occlude_fwd_bf16(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                                        const float* lin_x, const float* lin_y, void* out, int N, int NO, int D, int H,
                                        int W, int M, int align_corners, int fp16, void* workspace,
                                        size_t workspace_bytes, cudaStream_t stream) {
  if (fp16)
    return layout_occlude_fwd(vecs, boxes, masks, obj_off, lin_x, lin_y, static_cast<__half*>(out), N, NO, D, H, W, M,
                              align_corners, workspace, workspace_bytes, stream);
  return layout_occlude_fwd(vecs, boxes, masks, obj_off, lin_x, lin_y, static_cast<__nv_bfloat16*>(out), N, NO, D, H, W,
                            M, align_corners, workspace, workspace_bytes, stream);
}

CSG_API int csg_layout_bwd_geom(const float* dout, const float* vecs, const float* boxes, const float* masks,
                                const int* obj_off, const float* lin_x, const float* lin_y, float* dboxes,
                                float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return layout_bwd_geom(dout, vecs, boxes, masks, obj_off, lin_x, lin_y, dboxes, dmasks, N, NO, D, H, W, M,
                         align_corners, workspace, workspace_bytes, stream);
}

CSG_API int csg_layout_bwd_geom_bf16(const void* dout, const float* vecs, const float* boxes, const float* masks,
                                     const int* obj_off, const float* lin_x, const float* lin_y, float* dboxes,
                                     float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                     int fp16, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (fp16)
    return layout_bwd_geom(static_cast<const __half*>(dout), vecs, boxes, masks, obj_off, lin_x, lin_y, dboxes, dmasks,
                           N, NO, D, H, W, M, align_corners, workspace, workspace_bytes, stream);
  return layout_bwd_geom(static_cast<const __nv_bfloat16*>(dout), vecs, boxes, masks, obj_off, lin_x, lin_y, dboxes,
                         dmasks, N, NO, D, H, W, M, align_corners, workspace, workspace_bytes, stream);
}
