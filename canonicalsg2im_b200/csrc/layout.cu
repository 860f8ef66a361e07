// Single-pass layout compositor (boxes_to_layout / masks_to_layout) for sm_100a.
//
// Replaces sg2im/layout.py:12-188 of the reference: instead of materialising the per-object
// [O, D, H, W] samples (grid_sample) and scatter-adding them,
//
//   forward   a CTA (4 warps) owns a 512-pixel tile (8 rows x 64 or 4 rows x 128) of one image's [D, H, W]
//             canvas and builds the ordered list of objects whose support intersects the tile; each warp owns a
//             128-pixel strip, compacts the list to the objects that touch ITS strip, every lane accumulates
//             4 pixels x 16 channels in registers (64 FMAs per weight quad + 4 broadcast vector loads from shared
//             memory) and writes each canvas element exactly once with 128-bit streaming stores;
//   backward  (d/dvecs) a CTA owns (image, 32 channels, a range of 256-pixel bands): a producer warp streams the
//             incoming gradient band by band into a shared-memory ring with cp.async.bulk (1 KB per channel, fully
//             coalesced, completion on an mbarrier), four consumer warps -- thread = (channel, 64-pixel sub-band)
//             -- walk the objects that touch their sub-band, so the pixel weights are warp-uniform broadcasts and
//             zero weights are skipped without divergence; per-(object, channel) sums live in shared memory and
//             the per-range partials are combined in a fixed order by a second kernel.
//   backward, boxes_to_layout (W = 64 / 128 / 256): the same gradient ring, but the contraction is summed by parts
//             along y (layout_bwd_colsum_kernel below): thread = (channel, strip of W / 8 columns) keeps running
//             column sums in registers and an object costs a short dot product only on the rows where its row
//             factor changes.
//   generic   the previous tile/butterfly backward is kept for shapes the ring cannot serve (W % 64, H*W % 256,
//             D % 32 or unaligned gradients).
//   backward, d masks with fixed boxes (the predicted-mask training step): band-tiled, one more read of the gradient per
//             chunk of objects (layout_bwd_dmasks_kernel below, csg_layout_bwd_vecs_masks).
//
// The pixel weight of object o is separable for boxes_to_layout, S_o(y, x) = ay_o(y) * ax_o(x), and a 4-tap
// bilinear read of the mask for masks_to_layout.
//
// Coordinate chain (kept operation-for-operation so that ramp pixels of small
// boxes agree with the reference, SURVEY.md §7 "layout coordinate fidelity"):
//   u  = (lin[x] - x0) / w            layout.py:101   (lin = torch.linspace(0,1,W), passed in)
//   g  = 2u - 1                       layout.py:110
//   ix = ((g + 1) * S - 1) / 2        ATen grid_sampler unnormalize, align_corners=False
//   ix = ((g + 1) / 2) * (S - 1)      align_corners=True (torch <= 1.2 behaviour)
// with S = 8 for boxes_to_layout (layout.py:34) and S = M for masks_to_layout.
#include "layout_common.cuh"
#include <stdlib.h>
#include <type_traits>

// tensor-core backward (layout_bwd_tc.cu)
bool csg_layout_bwd_tc_eligible(const float* dout, int N, int D, int H, int W, int max_objs);
size_t csg_layout_bwd_tc_partial_floats(int N, int NO, int D, int H, int W, int max_objs);
int csg_layout_bwd_tc_launch(const float* dout, const float* masks, const int* obj_off, const float* axg, const float* ayg,
                             float* partial, float* dvecs, int N, int NO, int D, int H, int W, int M, int max_objs,
                             cudaStream_t stream);
CSG_API size_t csg_layout_bwd_vecs_workspace(int N, int NO, int D, int H, int W);

namespace {

// Warp 0 appends, in ascending object order, the objects of [*cursor, oend) that may touch the pixel rectangle
// [x0, x0+TW) x [y0, y0+TH), until the list holds lcap entries.  Returns through shared memory.
__device__ void build_list(const LayoutParams& p, int* list, int oend, int x0, int y0, int* s_cursor, int* s_count) {
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    const int S = p.masks ? p.M : 8;
    const float xlo = p.lin_x[x0], xhi = p.lin_x[min(x0 + p.TW, p.W) - 1];
    const float ylo = p.lin_y[y0], yhi = p.lin_y[min(y0 + p.TH, p.H) - 1];
    int cursor = *s_cursor, count = 0;
    while (cursor < oend && count < p.lcap) {
      int o = cursor + lane;
      bool keep = false;
      if (o < oend) {
        float4 b = ld_f4(p.boxes + 4 * (size_t)o);
        keep = box_poison(b) ||
               (axis_may_touch(b.x, b.z, xlo, xhi, S, p.align) && axis_may_touch(b.y, b.w, ylo, yhi, S, p.align));
      }
      unsigned bal = __ballot_sync(0xffffffffu, keep);
      int pos = count + __popc(bal & ((1u << lane) - 1u));
      int room = p.lcap - count;
      int total = __popc(bal);
      if (total <= room) {
        if (keep) list[pos] = o;
        count += total;
        cursor += 32;
      } else {
        // take only the first `room` kept objects; resume after the last one taken
        if (keep && pos < p.lcap) list[pos] = o;
        unsigned taken_last = __ballot_sync(0xffffffffu, keep && pos == p.lcap - 1);
        int last_lane = __ffs(taken_last) - 1;
        cursor += last_lane + 1;
        count = p.lcap;
      }
    }
    if (lane == 0) { *s_cursor = min(cursor, oend); *s_count = count; }
  }
}

// ========================================================================================
// forward: out[n, d, y, x] = sum_o vecs[o, d] * S_o(y, x)
// ========================================================================================
namespace fw {

constexpr int NTHREADS = 128;          // 4 warps x 128-pixel strips
constexpr int STRIP_PX = 128;
constexpr int TILE_PX = 4 * STRIP_PX;  // 512 pixels per tile: 8 rows x 64 or 4 rows x 128
constexpr int ORDER_MAX_N = 512;       // batches up to this many images are served heaviest-first

struct Smem {
  float* wS;           // [lcap][TILE_PX]   S_o(y, x) for the tile (masks_to_layout only)
  float* vS;           // [lcap][D]         vecs of the listed objects
  float* ax;           // [lcap][TW]        boxes: column factor; masks: column sample coordinate
  float* ay;           // [lcap][TH]        boxes: row factor;    masks: row sample coordinate
  int* list;           // [lcap]            object ids (global) in ascending order
  int* flags;          // [lcap]            1 = poison (never skipped)
  unsigned* rowmask;   // [lcap]            rows of the tile where the weight can be non-zero
  int* nact;           // [4]
  unsigned char* act;  // [4][lcap]         per-warp compacted list
};

__host__ __device__ inline size_t smem_floats(int lcap, int D, int TW, int TH, bool mask) {
  return (size_t)lcap * ((mask ? TILE_PX : 0) + D + TW + TH + 3) + 4 + (size_t)lcap;   // act: 4*lcap bytes = lcap words
}

__device__ __forceinline__ Smem carve(float* base, int lcap, int D, int TW, int TH, bool mask) {
  Smem s;
  s.wS = base;                                  // 16B aligned: first
  s.vS = s.wS + (mask ? (size_t)lcap * TILE_PX : 0);
  s.ax = s.vS + (size_t)lcap * D;
  s.ay = s.ax + (size_t)lcap * TW;
  s.list = reinterpret_cast<int*>(s.ay + (size_t)lcap * TH);
  s.flags = s.list + lcap;
  s.rowmask = reinterpret_cast<unsigned*>(s.flags + lcap);
  s.nact = reinterpret_cast<int*>(s.rowmask + lcap);
  s.act = reinterpret_cast<unsigned char*>(s.nact + 4);
  return s;
}

// Per-object separable factors for the tile (and, with masks, the per-pixel weights), plus the mask of rows
// where the weight can be non-zero (anything not exactly 0, NaN included).
template <bool HAS_MASK>
__device__ void build_weights(const LayoutParams& p, const Smem& s, int L, int x0, int y0) {
  const int tid = threadIdx.x;
  const int S = HAS_MASK ? p.M : 8;
  const int TW = p.TW, TH = p.TH;
  for (int c = tid; c < L; c += NTHREADS) {
    s.flags[c] = box_poison(ld_f4(p.boxes + 4 * (size_t)s.list[c])) ? 1 : 0;
    s.rowmask[c] = 0u;
  }
  __syncthreads();
  for (int i = tid; i < L * (TW + TH); i += NTHREADS) {
    int c = i / (TW + TH), r = i % (TW + TH);
    float4 b = ld_f4(p.boxes + 4 * (size_t)s.list[c]);
    const bool isx = r < TW;
    if (!isx) r -= TW;
    const int pos = (isx ? x0 : y0) + r;
    const int lim = isx ? p.W : p.H;
    const float coord = axis_coord((isx ? p.lin_x : p.lin_y)[min(pos, lim - 1)], isx ? b.x : b.y, isx ? b.z : b.w, S, p.align);
    if (HAS_MASK) {
      (isx ? s.ax : s.ay)[c * (isx ? TW : TH) + r] = coord;
    } else {
      float a = tap_ones(coord_tap(coord, S), S);
      if (pos >= lim) a = 0.f;
      if (isx) {
        s.ax[c * TW + r] = a;
      } else {
        s.ay[c * TH + r] = a;
        if (!(a == 0.f)) atomicOr(&s.rowmask[c], 1u << r);
      }
    }
  }
  if (HAS_MASK) {
    __syncthreads();
    for (int i = tid; i < L * TILE_PX; i += NTHREADS) {
      const int c = i / TILE_PX, px = i % TILE_PX;
      const int row = px / TW, col = px % TW;
      float w = 0.f;
      if (x0 + col < p.W && y0 + row < p.H)
        w = mask_weight(p.masks + (size_t)s.list[c] * S * S, S, coord_tap(s.ax[c * TW + col], S),
                        coord_tap(s.ay[c * TH + row], S));
      s.wS[i] = w;
      if (!(w == 0.f)) atomicOr(&s.rowmask[c], 1u << row);
    }
  }
  __syncthreads();
}

// acc[j][k] = sum over this warp's compacted objects, in list order, of vecs[o, d0 + j] * S_o(pixel k of this lane)
template <bool HAS_MASK, int NC>
__device__ __forceinline__ void accumulate(const LayoutParams& p, const Smem& s, const unsigned char* myact, int na,
                                           int TW, int TH, int warp, int spx, int row, int col, int d0,
                                           float (&acc)[NC][4]) {
#pragma unroll
  for (int j = 0; j < NC; ++j)
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[j][k] = 0.f;
  for (int a = 0; a < na; ++a) {
    const int c = myact[a];
    float4 w;
    if (HAS_MASK) {
      w = ld_f4(s.wS + c * TILE_PX + warp * STRIP_PX + spx);
    } else {
      const float wy = s.ay[c * TH + row];
      w = ld_f4(s.ax + c * TW + col);
      w.x *= wy; w.y *= wy; w.z *= wy; w.w *= wy;
    }
    const float* vp = s.vS + c * p.D + d0;
#pragma unroll
    for (int j4 = 0; j4 < NC; j4 += 4) {
      const float4 v = ld_f4(vp + j4);
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[j4 + j][0] = fmaf(vv[j], w.x, acc[j4 + j][0]);
        acc[j4 + j][1] = fmaf(vv[j], w.y, acc[j4 + j][1]);
        acc[j4 + j][2] = fmaf(vv[j], w.z, acc[j4 + j][2]);
        acc[j4 + j][3] = fmaf(vv[j], w.w, acc[j4 + j][3]);
      }
    }
  }
}

// One pass over the tile's object list [*s_cursor, ...): list, weights, vectors and the per-warp compaction into
// myact.  Returns the number of objects of this warp; *L / *more describe the list.
template <bool HAS_MASK>
__device__ __forceinline__ int build_pass(const LayoutParams& p, const Smem& s, int oend, int x0, int y0, int* s_cursor,
                                          int* s_count, unsigned my_rows, unsigned char* myact, bool* more) {
  const int tid = threadIdx.x, lane = tid & 31;
  build_list(p, s.list, oend, x0, y0, s_cursor, s_count);
  __syncthreads();
  const int L = *s_count;
  *more = *s_cursor < oend;   // read before the next build_list may advance it
  build_weights<HAS_MASK>(p, s, L, x0, y0);
  for (int i = tid; i < L * (p.D >> 2); i += NTHREADS) {
    int c = i / (p.D >> 2), d4 = i % (p.D >> 2);
    st_f4(s.vS + c * p.D + d4 * 4, ld_f4(p.vecs + (size_t)s.list[c] * p.D + d4 * 4));
  }
  // per-warp compaction: objects that touch this warp's strip (poisoned objects always do)
  int na = 0;
  for (int c0 = 0; c0 < L; c0 += 32) {
    const int c = c0 + lane;
    const bool keep = c < L && ((s.rowmask[c] & my_rows) != 0u || (s.flags[c] & 1));
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (keep) myact[na + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)c;
    na += __popc(bal);
  }
  __syncthreads();
  return na;
}

// T = float: the fp32 canvas.  T = __nv_bfloat16 / __half: the fp32 canvas rounded once to T (Tensor.to(T)).
template <bool HAS_MASK, int CH, typename T>
__global__ void __launch_bounds__(NTHREADS) layout_fwd_kernel(LayoutParams p, T* __restrict__ out) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) float smem_raw[];
  __shared__ int s_cursor, s_count;
  const Smem s = carve(smem_raw, p.lcap, p.D, p.TW, p.TH, HAS_MASK);
  // Images are served heaviest first (most objects first; CTAs are dispatched in blockIdx.y order), so that the
  // partial last wave of CTAs consists of the cheapest tiles: blockIdx.y is a rank, not an image index.
  __shared__ int s_cnt[ORDER_MAX_N];
  __shared__ int s_img;
  int n = blockIdx.y;
  if (p.N <= ORDER_MAX_N) {
    for (int i = threadIdx.x; i < p.N; i += NTHREADS) s_cnt[i] = p.obj_off[i + 1] - p.obj_off[i];
    __syncthreads();
    for (int i = threadIdx.x; i < p.N; i += NTHREADS) {
      const int ci = s_cnt[i];
      int rank = 0;
      for (int j = 0; j < p.N; ++j) {
        const int cj = s_cnt[j];
        rank += (cj > ci || (cj == ci && j < i)) ? 1 : 0;
      }
      if (rank == (int)blockIdx.y) s_img = i;
    }
    __syncthreads();
    n = s_img;
  }
  const int TW = p.TW, TH = p.TH;
  const int x0 = (blockIdx.x % p.tiles_x) * TW, y0 = (blockIdx.x / p.tiles_x) * TH;
  const int oend = p.obj_off[n + 1];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) s_cursor = p.obj_off[n];
  __syncthreads();

  // this lane's 4 pixels: strip `warp` = rows [warp*SR, warp*SR + SR) of the tile, SR = 128 / TW
  const int SR = STRIP_PX / TW;
  const int spx = lane * 4;                         // pixel offset inside the strip
  const int row = warp * SR + spx / TW, col = spx % TW;
  const int y = y0 + row, x = x0 + col;
  const bool vec4 = (p.W & 3) == 0;
  const bool active = y < p.H && x < p.W;
  const unsigned my_rows = ((1u << SR) - 1u) << (warp * SR);
  unsigned char* myact = s.act + warp * p.lcap;
  if constexpr (sizeof(T) == 4) {
    // (the fp32 canvas keeps its own loop, written out, so that its code is exactly what it was before the 16-bit
    // canvases were added)
    bool first = true;
    while (true) {
      build_list(p, s.list, oend, x0, y0, &s_cursor, &s_count);
      __syncthreads();
      const int L = s_count;
      const bool more = s_cursor < oend;   // read before the next build_list may advance it
      build_weights<HAS_MASK>(p, s, L, x0, y0);
      for (int i = tid; i < L * (p.D >> 2); i += NTHREADS) {
        int c = i / (p.D >> 2), d4 = i % (p.D >> 2);
        st_f4(s.vS + c * p.D + d4 * 4, ld_f4(p.vecs + (size_t)s.list[c] * p.D + d4 * 4));
      }
      // per-warp compaction: objects that touch this warp's strip (poisoned objects always do)
      int na = 0;
      for (int c0 = 0; c0 < L; c0 += 32) {
        const int c = c0 + lane;
        const bool keep = c < L && ((s.rowmask[c] & my_rows) != 0u || (s.flags[c] & 1));
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) myact[na + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)c;
        na += __popc(bal);
      }
      __syncthreads();
      if (active) {
        const size_t plane = (size_t)p.H * p.W;
        float* dst = out + (size_t)n * p.D * plane + (size_t)y * p.W + x;      // channel 0 of this lane's pixels
        for (int d0 = 0; d0 < p.D; d0 += CH) {
          float acc[CH][4];
#pragma unroll
          for (int j = 0; j < CH; ++j)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[j][k] = 0.f;
          for (int a = 0; a < na; ++a) {
            const int c = myact[a];
            float4 w;
            if (HAS_MASK) {
              w = ld_f4(s.wS + c * TILE_PX + warp * STRIP_PX + spx);
            } else {
              const float wy = s.ay[c * TH + row];
              w = ld_f4(s.ax + c * TW + col);
              w.x *= wy; w.y *= wy; w.z *= wy; w.w *= wy;
            }
            const float* vp = s.vS + c * p.D + d0;
#pragma unroll
            for (int j4 = 0; j4 < CH; j4 += 4) {
              const float4 v = ld_f4(vp + j4);
              const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                acc[j4 + j][0] = fmaf(vv[j], w.x, acc[j4 + j][0]);
                acc[j4 + j][1] = fmaf(vv[j], w.y, acc[j4 + j][1]);
                acc[j4 + j][2] = fmaf(vv[j], w.z, acc[j4 + j][2]);
                acc[j4 + j][3] = fmaf(vv[j], w.w, acc[j4 + j][3]);
              }
            }
          }
          if (vec4 && first) {
            // the common case: every canvas element is written exactly once, 16 bytes per lane, 512 contiguous
            // bytes per warp and channel
#pragma unroll
            for (int j = 0; j < CH; ++j, dst += plane)
              st_f4_stream(dst, make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]));
          } else {
#pragma unroll
            for (int j = 0; j < CH; ++j, dst += plane) {
              if (vec4) {
                float4 r = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
                float4 o = ld_f4(dst);
                r.x += o.x; r.y += o.y; r.z += o.z; r.w += o.w;
                st_f4_stream(dst, r);
              } else {
                for (int k = 0; k < 4 && x + k < p.W; ++k) dst[k] = first ? acc[j][k] : dst[k] + acc[j][k];
              }
            }
          }
        }
      }
      first = false;
      __syncthreads();
      if (!more) break;
    }
  } else {
    // 16-bit canvas: every element is rounded once, from the same fp32 sum as the fp32 canvas.  A tile whose objects
    // fit one list (the common case) is written as the fp32 kernel writes it, 8 bytes per lane, 256 contiguous bytes
    // per warp and channel.  A tile that needs several passes keeps the running total tot = tot + acc_pass (the fp32
    // canvas's out = out + acc) in registers for 4 channels at a time and rebuilds its lists for every channel group.
    auto store = [&](T* dst, const float (&v)[4]) {
      if (vec4) st4_stream(dst, v[0], v[1], v[2], v[3]);
      else for (int k = 0; k < 4 && x + k < p.W; ++k) dst[k] = from_f32<T>(v[k]);
    };
    const size_t plane = (size_t)p.H * p.W;
    T* dst0 = out + (size_t)n * p.D * plane + (size_t)y * p.W + x;
    bool more;
    int na = build_pass<HAS_MASK>(p, s, oend, x0, y0, &s_cursor, &s_count, my_rows, myact, &more);
    if (!more) {
      if (active) {
        T* dst = dst0;
        for (int d0 = 0; d0 < p.D; d0 += CH) {
          float acc[CH][4];
          accumulate<HAS_MASK, CH>(p, s, myact, na, TW, TH, warp, spx, row, col, d0, acc);
#pragma unroll
          for (int j = 0; j < CH; ++j, dst += plane) store(dst, acc[j]);
        }
      }
      return;
    }
    constexpr int MC = 4;
    for (int d0 = 0; d0 < p.D; d0 += MC) {
      if (d0 > 0) {
        __syncthreads();
        if (tid == 0) s_cursor = p.obj_off[n];
        __syncthreads();
        na = build_pass<HAS_MASK>(p, s, oend, x0, y0, &s_cursor, &s_count, my_rows, myact, &more);
      }
      float tot[MC][4];
      accumulate<HAS_MASK, MC>(p, s, myact, na, TW, TH, warp, spx, row, col, d0, tot);
      while (more) {
        __syncthreads();
        na = build_pass<HAS_MASK>(p, s, oend, x0, y0, &s_cursor, &s_count, my_rows, myact, &more);
        float acc[MC][4];
        accumulate<HAS_MASK, MC>(p, s, myact, na, TW, TH, warp, spx, row, col, d0, acc);
#pragma unroll
        for (int j = 0; j < MC; ++j)
#pragma unroll
          for (int k = 0; k < 4; ++k) tot[j][k] = tot[j][k] + acc[j][k];
      }
      if (active) {
#pragma unroll
        for (int j = 0; j < MC; ++j) store(dst0 + (size_t)(d0 + j) * plane, tot[j]);
      }
    }
  }
}

}  // namespace fw

// ========================================================================================
// backward wrt vecs, ring version: dvecs[o, d] = sum_{y, x} dout[n, d, y, x] * S_o(y, x)
// ========================================================================================
namespace bw {

constexpr int DC = 32;                 // channels per CTA
constexpr int BAND = 256;              // pixels per band (1 KB per channel)
constexpr int SUBS = 8;                // consumer warps = 32-pixel sub-bands (8 + 1 warps per CTA, two CTAs per SM: the
                                       // per-object load -> FMA -> accumulate chains of one warp hide behind the others)
constexpr int SUB_PX = BAND / SUBS;
constexpr int STAGES = 2;
// A stage holds DC channels x one band of the gradient in its own element type T (fp32: 1 KB, 16-bit: 512 B per channel,
// one bulk copy each).  Channels are 16 B apart beyond the band, so that the 16-B loads of 8 consecutive lanes
// (= channels) land on distinct bank groups: 260 floats for fp32, 264 halves for 16-bit.
template <typename T>
struct Stage {
  static constexpr int CSTRIDE = BAND + 16 / (int)sizeof(T);        // elements between channels
  static constexpr int FLOATS = DC * CSTRIDE * (int)sizeof(T) / 4;  // size of one stage in 4-byte words
};
constexpr int STAGE_FLOATS = Stage<float>::FLOATS;
constexpr int NCONS = SUBS * 32;
constexpr int NTHREADS = NCONS + 32;   // + producer warp

struct Params {
  LayoutParams p;
  const void* dout;      // float, __nv_bfloat16 or __half (the kernel's T)
  float* partial;        // [splits][NO][D]
  const float* axg;      // [NO][W]  boxes: column factor; masks: column sample coordinate   (layout_tables_kernel)
  const float* ayg;      // [NO][H]
  const int* rng;        // [NO][4]  xmin, xmax, ymin, ymax: outside, the weight is exactly zero (max < min: nowhere)
  int NO, splits, bands_per_item, cblocks;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      printf("csg layout_bwd: mbarrier timeout (block %d thread %d parity %u)\n", blockIdx.x, threadIdx.x, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NCONS) : "memory"); }

struct Smem {
  float* stage;     // [STAGES][DC][CSTRIDE]
  float* acc;       // [lcap][SUBS][DC]
  float* ax;        // [lcap][W]   boxes: column factor; masks: column sample coordinate
  float* wS;        // [lcap][BAND] masks only: weights of the current band
  int* rng;         // [lcap][4]   xmin, xmax, ymin, ymax
  unsigned char* act;  // [SUBS][lcap]
  unsigned long long* bars;   // full[STAGES], empty[STAGES], tables
};

__host__ __device__ inline size_t smem_bytes(int lcap, int H, int W, bool mask, int stage_floats = STAGE_FLOATS) {
  (void)H;   // the per-row factors stay in global memory (one L1-resident float per object visit)
  size_t f = (size_t)STAGES * stage_floats + (size_t)lcap * SUBS * DC + (size_t)lcap * W +
             (mask ? (size_t)lcap * BAND : 0) + (size_t)lcap * 4 + (size_t)lcap * SUBS / 4 /* act: SUBS * lcap bytes */;
  return f * 4 + (2 * STAGES + 1) * 8 + 16;
}

__device__ __forceinline__ Smem carve(float* base, int lcap, int H, int W, bool mask, int stage_floats) {
  Smem s;
  s.stage = base;
  s.acc = s.stage + (size_t)STAGES * stage_floats;
  s.ax = s.acc + (size_t)lcap * SUBS * DC;
  s.wS = s.ax + (size_t)lcap * W;
  s.rng = reinterpret_cast<int*>(s.wS + (mask ? (size_t)lcap * BAND : 0));
  s.act = reinterpret_cast<unsigned char*>(s.rng + 4 * lcap);
  uintptr_t b = reinterpret_cast<uintptr_t>(s.act + (size_t)SUBS * lcap);
  s.bars = reinterpret_cast<unsigned long long*>((b + 7) & ~(uintptr_t)7);
  return s;
}

// One block per object: ax[o][W], ay[o][H] (boxes: separable weight factors; masks: sample coordinates) and the
// column / row intervals outside of which the weight of the object is exactly zero.
template <bool HAS_MASK>
__global__ void __launch_bounds__(128) layout_tables_kernel(LayoutParams p, int NO, float* __restrict__ axg,
                                                            float* __restrict__ ayg, int* __restrict__ rng) {
  CSG_PDL_WAIT();
  __shared__ int r[4];
  const int o = blockIdx.x;
  const int S = HAS_MASK ? p.M : 8;
  const float4 b = ld_f4(p.boxes + 4 * (size_t)o);
  const bool poison = box_poison(b);
  if (threadIdx.x == 0) {
    r[0] = poison ? 0 : p.W;  r[1] = poison ? p.W - 1 : -1;
    r[2] = poison ? 0 : p.H;  r[3] = poison ? p.H - 1 : -1;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < p.W + p.H; i += blockDim.x) {
    const bool isx = i < p.W;
    const int k = isx ? i : i - p.W;
    const float coord = axis_coord((isx ? p.lin_x : p.lin_y)[k], isx ? b.x : b.y, isx ? b.z : b.w, S, p.align);
    float val;
    bool touched;
    if (HAS_MASK) {
      val = coord;
      touched = !(coord <= -1.f) && !(coord >= (float)S);          // some tap in range (NaN counts as touched)
    } else {
      val = tap_ones(coord_tap(coord, S), S);
      touched = !(val == 0.f);
    }
    (isx ? axg + (size_t)o * p.W : ayg + (size_t)o * p.H)[k] = val;
    if (touched) {
      atomicMin(&r[isx ? 0 : 2], k);
      atomicMax(&r[isx ? 1 : 3], k);
    }
  }
  __syncthreads();
  if (threadIdx.x < 4) rng[4 * (size_t)o + threadIdx.x] = r[threadIdx.x];
}

// T: element type of the incoming gradient (float, __nv_bfloat16, __half); widened to fp32 as it leaves the stage, so the
// sums are those of the fp32 kernel given the widened gradient.
template <bool HAS_MASK, typename T>
__global__ void __launch_bounds__(NTHREADS) layout_bwd_ring_kernel(Params q) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) float smem_raw[];
  constexpr int CSTRIDE = Stage<T>::CSTRIDE;
  const LayoutParams& p = q.p;
  const Smem s = carve(smem_raw, p.lcap, p.H, p.W, HAS_MASK, Stage<T>::FLOATS);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = blockIdx.x % q.splits;
  const int cblk = (blockIdx.x / q.splits) % q.cblocks;
  const int n = blockIdx.x / (q.splits * q.cblocks);
  const int obeg = p.obj_off[n], oend = p.obj_off[n + 1];
  const int On = oend - obeg;
  const int b0 = split * q.bands_per_item, nb = q.bands_per_item;
  const int nchunks = (On + p.lcap - 1) / p.lcap;
  const int S = HAS_MASK ? p.M : 8;
  const size_t plane = (size_t)p.H * p.W;
  float* my_partial = q.partial + ((size_t)split * q.NO + obeg) * p.D + cblk * DC;   // [On][D] slice, DC wide

  const uint32_t full0 = smem_u32(s.bars), empty0 = smem_u32(s.bars + STAGES), tab = smem_u32(s.bars + 2 * STAGES);
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(full0 + 8 * i, 1);
      mbar_init(empty0 + 8 * i, NCONS);
    }
    mbar_init(tab, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == SUBS) {
    // ---------------- producer: one 1 KB bulk copy per channel per band
    const T* src0 = static_cast<const T*>(q.dout) + ((size_t)n * p.D + cblk * DC + lane) * plane + (size_t)b0 * BAND;
    int it = 0;
    for (int ch = 0; ch < nchunks; ++ch) {
      for (int b = 0; b < nb; ++b, ++it) {
        const int st = it % STAGES;
        if (it >= STAGES) mbar_wait(empty0 + 8 * st, ((it / STAGES) - 1) & 1);
        if (lane == 0) mbar_arrive_expect_tx(full0 + 8 * st, DC * BAND * sizeof(T));
        __syncwarp();
        bulk_load(smem_u32(reinterpret_cast<T*>(s.stage + (size_t)st * Stage<T>::FLOATS) + lane * CSTRIDE),
                  src0 + (size_t)b * BAND, BAND * sizeof(T), full0 + 8 * st);
      }
    }
    return;
  }

  // ---------------- consumers: thread = (channel lane, sub-band warp)
  // The 64 gradient values of (channel, sub-band) are copied to registers once per band and the stage is handed
  // back to the producer at once.  Weights are warp-uniform broadcasts; quarters of the sub-band outside an
  // object's columns are skipped without divergence.
  const int sub = warp;
  unsigned char* myact = s.act + sub * p.lcap;
  int it = 0;
  for (int ch = 0; ch < nchunks; ++ch) {
    const int cbeg = obeg + ch * p.lcap;
    const int L = min(p.lcap, oend - cbeg);
    // per-object tables of this chunk (separable factors / sample coordinates and the non-zero intervals),
    // precomputed by layout_tables_kernel: two bulk copies (row factors are read from global memory on use)
    if (tid == 0) {
      const uint32_t bx = L * p.W * 4, br = L * 16;
      mbar_arrive_expect_tx(tab, bx + br);
      bulk_load(smem_u32(s.ax), q.axg + (size_t)cbeg * p.W, bx, tab);
      bulk_load(smem_u32(s.rng), q.rng + (size_t)cbeg * 4, br, tab);
    }
    for (int i = tid; i < L * SUBS * DC; i += NCONS) s.acc[i] = 0.f;
    mbar_wait(tab, ch & 1);
    consumer_sync();

    for (int b = 0; b < nb; ++b, ++it) {
      const int st = it % STAGES;
      const int pix0 = (b0 + b) * BAND + sub * SUB_PX;      // first pixel of this warp's sub-band
      const int row = pix0 / p.W, col0 = pix0 % p.W;
      if (HAS_MASK) {
        // weights of this band for the objects that touch it (others are never read)
        const int bpix = (b0 + b) * BAND;
        for (int i = tid; i < L * BAND; i += NCONS) {
          const int c = i / BAND, px = i % BAND;
          const int y = (bpix + px) / p.W, x = (bpix + px) % p.W;
          float w = 0.f;
          const int4 r4 = *reinterpret_cast<const int4*>(s.rng + 4 * c);
          if (y >= r4.z && y <= r4.w && x >= r4.x && x <= r4.y)
            w = mask_weight(p.masks + (size_t)(cbeg + c) * S * S, S, coord_tap(s.ax[c * p.W + x], S),
                            coord_tap(__ldg(q.ayg + (size_t)(cbeg + c) * p.H + y), S));
          s.wS[i] = w;
        }
        consumer_sync();
      }
      // objects touching this sub-band, in ascending order
      int na = 0;
      for (int c0 = 0; c0 < L; c0 += 32) {
        const int c = c0 + lane;
        bool keep = false;
        if (c < L) {
          const int4 r4 = *reinterpret_cast<const int4*>(s.rng + 4 * c);
          keep = row >= r4.z && row <= r4.w && r4.x <= col0 + SUB_PX - 1 && r4.y >= col0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) myact[na + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)c;
        na += __popc(bal);
      }
      __syncwarp();
      mbar_wait(full0 + 8 * st, (it / STAGES) & 1);
      float4 g[SUB_PX / 4];
      {
        const T* gch = reinterpret_cast<const T*>(s.stage + (size_t)st * Stage<T>::FLOATS) + lane * CSTRIDE + sub * SUB_PX;
        if constexpr (sizeof(T) == 4) {
#pragma unroll
          for (int i = 0; i < SUB_PX / 4; ++i) g[i] = ld_f4(gch + 4 * i);
        } else {
#pragma unroll
          for (int i = 0; i < SUB_PX / 8; ++i) {
            float f[8];
            ld8_f32(gch + 8 * i, f);
            g[2 * i] = make_float4(f[0], f[1], f[2], f[3]);
            g[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
          }
        }
      }
      mbar_arrive(empty0 + 8 * st);          // the stage is free as soon as the registers hold it
      // Weights outside an object's column interval are exact zeros, so the dot product over the whole 32-pixel
      // sub-band needs no per-quarter test (adding 0 * g changes nothing), and two objects are walked per iteration:
      // their weight loads, FMA chains and accumulator updates are independent and overlap.
      // (the same dot product on the packed fp32 pipe -- fma.rn.f32x2, 16 FFMA2 per object in two 8-deep or four 4-deep
      // chains -- measured 89 us against 81 us for this scalar form on the cfg2 canvas: dropped)
      auto dot = [&](const float* wrow) {
        float sum = 0.f;
#pragma unroll
        for (int qd = 0; qd < SUB_PX / 16; ++qd) {
          const float4 w0 = ld_f4(wrow + 16 * qd), w1 = ld_f4(wrow + 16 * qd + 4);
          const float4 w2 = ld_f4(wrow + 16 * qd + 8), w3 = ld_f4(wrow + 16 * qd + 12);
          const float4 g0 = g[4 * qd], g1 = g[4 * qd + 1], g2 = g[4 * qd + 2], g3 = g[4 * qd + 3];
          float t0 = g0.x * w0.x, t1 = g1.x * w1.x, t2 = g2.x * w2.x, t3 = g3.x * w3.x;
          t0 = fmaf(g0.y, w0.y, t0); t1 = fmaf(g1.y, w1.y, t1); t2 = fmaf(g2.y, w2.y, t2); t3 = fmaf(g3.y, w3.y, t3);
          t0 = fmaf(g0.z, w0.z, t0); t1 = fmaf(g1.z, w1.z, t1); t2 = fmaf(g2.z, w2.z, t2); t3 = fmaf(g3.z, w3.z, t3);
          t0 = fmaf(g0.w, w0.w, t0); t1 = fmaf(g1.w, w1.w, t1); t2 = fmaf(g2.w, w2.w, t2); t3 = fmaf(g3.w, w3.w, t3);
          sum += (t0 + t1) + (t2 + t3);
        }
        return sum;
      };
      auto wrow_of = [&](int c) { return HAS_MASK ? s.wS + c * BAND + sub * SUB_PX : s.ax + c * p.W + col0; };
      int a = 0;
#pragma unroll 1
      for (; a + 1 < na; a += 2) {
        const int c0 = myact[a], c1 = myact[a + 1];                    // distinct objects: the two updates do not alias
        float wy0 = 1.f, wy1 = 1.f;
        if (!HAS_MASK) {
          wy0 = __ldg(q.ayg + (size_t)(cbeg + c0) * p.H + row);
          wy1 = __ldg(q.ayg + (size_t)(cbeg + c1) * p.H + row);
        }
        float* acc0 = s.acc + (c0 * SUBS + sub) * DC + lane;
        float* acc1 = s.acc + (c1 * SUBS + sub) * DC + lane;
        const float old0 = *acc0, old1 = *acc1;
        const float s0 = dot(wrow_of(c0)), s1 = dot(wrow_of(c1));
        *acc0 = old0 + s0 * wy0;
        *acc1 = old1 + s1 * wy1;
      }
      if (a < na) {
        const int c = myact[a];
        const float wy = HAS_MASK ? 1.f : __ldg(q.ayg + (size_t)(cbeg + c) * p.H + row);
        s.acc[(c * SUBS + sub) * DC + lane] += dot(wrow_of(c)) * wy;
      }
      if (HAS_MASK) consumer_sync();      // wS is rebuilt for the next band
    }
    consumer_sync();
    // combine the sub-band warps in a fixed order
    for (int i = tid; i < L * DC; i += NCONS) {
      const int c = i / DC, d = i % DC;
      float v = 0.f;
#pragma unroll
      for (int u = 0; u < SUBS; ++u) v += s.acc[(c * SUBS + u) * DC + d];
      my_partial[(size_t)(ch * p.lcap + c) * p.D + d] = v;
    }
    consumer_sync();
  }
}

// ----------------------------------------------------------------------------------------
// boxes_to_layout only: the same contraction through running COLUMN sums (summation by parts along y).
//
// The weight of a box is separable, S_o(y, x) = ay_o(y) * ax_o(x), and ay_o is a trapezoid: 0, a ramp of about h/8
// rows, 1 inside, a ramp, 0.  Over the rows y0 ... y1 of a CTA's range
//     sum_y ay(y) G(y)  =  sum_y [ay(y) - ay(y + 1)] * Cum(y)         (ay(y1 + 1) := 0),   Cum(y) = sum_{y' <= y} G(y'),
// and Cum(y) = sum_x ax(x) * C_y(x) with C_y(x) the running column sum of the incoming gradient.  So a thread
// (channel, strip of W / 8 columns) keeps C in registers (one FADD per gradient element, whatever the number of
// objects) and an object costs one short dot product only on the rows where ay CHANGES -- its two ramps and the last
// row of the range -- instead of on every row it covers: ~2.5x fewer object visits on the cfg2 canvas, each over 8
// columns instead of 32, and no per-band list building (the visit set of a row is rowmask[y] & stripmask, one AND).
// Rounding: C is a sum of at most 64 rows (pick_splits), so the result differs from the direct sum by a few ulp of
// max_y |Cum(y)| -- inside the 1e-5 (relative to the tensor scale) contract, tested against the golden vectors.
namespace cs {
constexpr int RR_MAX = 64;             // rows per CTA range (bounds the length of the running sums)
constexpr int LCAP_MAX = 32;           // objects per chunk: one bit each in a row's visit mask

struct Smem {
  float* stage;     // [STAGES][DC][CSTRIDE]
  float* acc;       // [lcap][SUBS][DC]
  float* ax;        // [lcap][W]
  float* day;       // [lcap][RR]   ay(y) - ay(y + 1) over the CTA's rows (last row: ay(y))
  int* rng;         // [lcap][4]
  unsigned* rowmask;   // [RR]      objects of the chunk whose factor changes behind row r
  unsigned long long* bars;
};
__host__ __device__ inline size_t smem_bytes(int lcap, int W, int RR, int stage_floats = STAGE_FLOATS) {
  size_t f = (size_t)STAGES * stage_floats + (size_t)lcap * SUBS * DC + (size_t)lcap * W + (size_t)lcap * RR +
             (size_t)lcap * 4 + (size_t)RR;
  return f * 4 + (2 * STAGES + 1) * 8 + 16;
}
__device__ __forceinline__ Smem carve(float* base, int lcap, int W, int RR, int stage_floats) {
  Smem s;
  s.stage = base;
  s.acc = s.stage + (size_t)STAGES * stage_floats;
  s.ax = s.acc + (size_t)lcap * SUBS * DC;
  s.day = s.ax + (size_t)lcap * W;
  s.rng = reinterpret_cast<int*>(s.day + (size_t)lcap * RR);
  s.rowmask = reinterpret_cast<unsigned*>(s.rng + 4 * lcap);
  uintptr_t b = reinterpret_cast<uintptr_t>(s.rowmask + RR);
  s.bars = reinterpret_cast<unsigned long long*>((b + 7) & ~(uintptr_t)7);
  return s;
}

// SW: strip width, W = 8 * SW columns, one strip per consumer warp.  T: gradient element type, widened on load.
template <int SW, typename T>
__global__ void __launch_bounds__(NTHREADS) layout_bwd_colsum_kernel(Params q) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) float smem_raw[];
  constexpr int CSTRIDE = Stage<T>::CSTRIDE;
  constexpr int W = SW * SUBS;
  constexpr int RPB = BAND / W;          // rows per band
  static_assert(RPB * SW == SUB_PX, "a thread holds 32 gradient values per band");
  const LayoutParams& p = q.p;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = blockIdx.x % q.splits;
  const int cblk = (blockIdx.x / q.splits) % q.cblocks;
  const int n = blockIdx.x / (q.splits * q.cblocks);
  const int obeg = p.obj_off[n], oend = p.obj_off[n + 1];
  const int On = oend - obeg;
  const int b0 = split * q.bands_per_item, nb = q.bands_per_item;
  const int RR = nb * RPB, row0 = b0 * RPB;
  const Smem s = carve(smem_raw, p.lcap, W, RR, Stage<T>::FLOATS);
  const int nchunks = (On + p.lcap - 1) / p.lcap;
  const size_t plane = (size_t)p.H * W;
  float* my_partial = q.partial + ((size_t)split * q.NO + obeg) * p.D + cblk * DC;

  const uint32_t full0 = smem_u32(s.bars), empty0 = smem_u32(s.bars + STAGES), tab = smem_u32(s.bars + 2 * STAGES);
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(full0 + 8 * i, 1);
      mbar_init(empty0 + 8 * i, NCONS);
    }
    mbar_init(tab, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == SUBS) {
    // ---------------- producer: one 1 KB bulk copy per channel per band (as in the ring kernel)
    const T* src0 = static_cast<const T*>(q.dout) + ((size_t)n * p.D + cblk * DC + lane) * plane + (size_t)b0 * BAND;
    int it = 0;
    for (int ch = 0; ch < nchunks; ++ch) {
      for (int b = 0; b < nb; ++b, ++it) {
        const int st = it % STAGES;
        if (it >= STAGES) mbar_wait(empty0 + 8 * st, ((it / STAGES) - 1) & 1);
        if (lane == 0) mbar_arrive_expect_tx(full0 + 8 * st, DC * BAND * sizeof(T));
        __syncwarp();
        bulk_load(smem_u32(reinterpret_cast<T*>(s.stage + (size_t)st * Stage<T>::FLOATS) + lane * CSTRIDE),
                  src0 + (size_t)b * BAND, BAND * sizeof(T), full0 + 8 * st);
      }
    }
    return;
  }

  // ---------------- consumers: thread = (channel lane, column strip warp)
  const int sx0 = warp * SW;
  int it = 0;
  for (int ch = 0; ch < nchunks; ++ch) {
    const int cbeg = obeg + ch * p.lcap;
    const int L = min(p.lcap, oend - cbeg);
    if (tid == 0) {
      const uint32_t bx = L * W * 4, br = L * 16;
      mbar_arrive_expect_tx(tab, bx + br);
      bulk_load(smem_u32(s.ax), q.axg + (size_t)cbeg * W, bx, tab);
      bulk_load(smem_u32(s.rng), q.rng + (size_t)cbeg * 4, br, tab);
    }
    for (int i = tid; i < L * SUBS * DC; i += NCONS) s.acc[i] = 0.f;
    for (int i = tid; i < L * RR; i += NCONS) {
      const int c = i / RR, r = i % RR;
      const float* ayo = q.ayg + (size_t)(cbeg + c) * p.H + row0 + r;
      const float a0 = __ldg(ayo), a1 = (r == RR - 1) ? 0.f : __ldg(ayo + 1);
      s.day[i] = a0 - a1;
    }
    mbar_wait(tab, ch & 1);
    consumer_sync();
    for (int r = warp; r < RR; r += SUBS) {
      const float v = lane < L ? s.day[lane * RR + r] : 0.f;
      const unsigned bal = __ballot_sync(0xffffffffu, !(v == 0.f));      // NaN counts as a change
      if (lane == 0) s.rowmask[r] = bal;
    }
    unsigned smask;
    {
      bool keep = false;
      if (lane < L) {
        const int4 r4 = *reinterpret_cast<const int4*>(s.rng + 4 * lane);
        keep = r4.x <= sx0 + SW - 1 && r4.y >= sx0;
      }
      smask = __ballot_sync(0xffffffffu, keep);
    }
    consumer_sync();

    float C[SW];
#pragma unroll
    for (int i = 0; i < SW; ++i) C[i] = 0.f;
    for (int b = 0; b < nb; ++b, ++it) {
      const int st = it % STAGES;
      unsigned rm[RPB];
#pragma unroll
      for (int k = 0; k < RPB; ++k) rm[k] = s.rowmask[b * RPB + k] & smask;
      mbar_wait(full0 + 8 * st, (it / STAGES) & 1);
      float4 g[SUB_PX / 4];
      {
        const T* gch = reinterpret_cast<const T*>(s.stage + (size_t)st * Stage<T>::FLOATS) + lane * CSTRIDE + sx0;
        if constexpr (sizeof(T) == 4) {
#pragma unroll
          for (int k = 0; k < RPB; ++k)
#pragma unroll
            for (int i = 0; i < SW / 4; ++i) g[k * (SW / 4) + i] = ld_f4(gch + k * W + 4 * i);
        } else {
#pragma unroll
          for (int k = 0; k < RPB; ++k)
#pragma unroll
            for (int i = 0; i < SW / 8; ++i) {
              float f[8];
              ld8_f32(gch + k * W + 8 * i, f);
              g[k * (SW / 4) + 2 * i] = make_float4(f[0], f[1], f[2], f[3]);
              g[k * (SW / 4) + 2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
            }
        }
      }
      mbar_arrive(empty0 + 8 * st);          // the stage is free as soon as the registers hold it
#pragma unroll
      for (int k = 0; k < RPB; ++k) {
#pragma unroll
        for (int i = 0; i < SW / 4; ++i) {
          const float4 v = g[k * (SW / 4) + i];
          C[4 * i] += v.x; C[4 * i + 1] += v.y; C[4 * i + 2] += v.z; C[4 * i + 3] += v.w;
        }
        unsigned m = rm[k];
        const int r = b * RPB + k;
        while (m) {
          const int c = __ffs(m) - 1;
          m &= m - 1;
          const float* wrow = s.ax + c * W + sx0;
          float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
          for (int i = 0; i < SW / 4; ++i) {
            const float4 w4 = ld_f4(wrow + 4 * i);
            t0 = fmaf(C[4 * i], w4.x, t0); t1 = fmaf(C[4 * i + 1], w4.y, t1);
            t2 = fmaf(C[4 * i + 2], w4.z, t2); t3 = fmaf(C[4 * i + 3], w4.w, t3);
          }
          const float d = s.day[c * RR + r];
          float* a = s.acc + (c * SUBS + warp) * DC + lane;
          *a = fmaf(d, (t0 + t1) + (t2 + t3), *a);
        }
      }
    }
    consumer_sync();
    // combine the strip warps in a fixed order
    for (int i = tid; i < L * DC; i += NCONS) {
      const int c = i / DC, d = i % DC;
      float v = 0.f;
#pragma unroll
      for (int u = 0; u < SUBS; ++u) v += s.acc[(c * SUBS + u) * DC + d];
      my_partial[(size_t)(ch * p.lcap + c) * p.D + d] = v;
    }
    consumer_sync();
  }
}

int pick_lcap(int max_objs, int W, int RR) {
  int lcap = max_objs > 0 ? max_objs : 16;
  lcap = (lcap + 3) & ~3;
  if (lcap < 4) lcap = 4;
  if (lcap > LCAP_MAX) lcap = LCAP_MAX;
  while (lcap > 4 && smem_bytes(lcap, W, RR) > 110 * 1024) lcap -= 4;   // two CTAs per SM
  return lcap;
}
bool shape_ok(int H, int W) { return W == 64 || W == 128 || W == 256; }
}  // namespace cs

__global__ void layout_bwd_sum_splits_kernel(const float* __restrict__ partial, float* __restrict__ dvecs,
                                             long long n, int splits) {
  CSG_PDL_WAIT();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += partial[(size_t)s * n + i];
  dvecs[i] = acc;
}

int pick_splits(int N, int D, int H, int W, bool colsum = false) {
  const int nbands = (H * W) / BAND;
  const long long base = (long long)N * (D / DC);
  // CTAs wanted: ~7 waves of two CTAs per SM for the ring kernel; the column-sum kernel has little to do per band and
  // pays ~2.9 us of set-up per CTA against 1.6 us per band, so it takes half as many CTAs of twice the length
  // (cfg2 canvas: 61.5 us with 1024 CTAs of 8 bands, 64 us with 2048 of 4, 75 us with 512 of 16)
  const long long want = (colsum ? 3LL : 6LL) * 2 * csg_num_sms();
  int s = 1;
  while (s * 2 <= nbands && nbands % (s * 2) == 0 && base * s < want) s *= 2;
  while (H / s > cs::RR_MAX && s * 2 <= nbands && nbands % (s * 2) == 0) s *= 2;   // column-sum kernel: short running sums
  { const char* e = getenv("CSG_LAYOUT_SPLITS"); if (e && atoi(e) > 0 && nbands % atoi(e) == 0) s = atoi(e); }   // scratch/bench_layout.py
  return s;
}

int pick_lcap(int max_objs, int H, int W, bool mask) {
  int lcap = max_objs > 0 ? max_objs : 16;
  lcap = (lcap + 3) & ~3;
  if (lcap < 4) lcap = 4;
  if (lcap > 64) lcap = 64;
  while (lcap > 4 && smem_bytes(lcap, H, W, mask) > 110 * 1024) lcap -= 4;   // two CTAs per SM
  return lcap;
}

bool shape_ok(int D, int H, int W) {
  return (W % 64) == 0 && (H % 4) == 0 && ((long long)H * W) % BAND == 0 && (D % DC) == 0 &&
         smem_bytes(4, H, W, true) <= 200 * 1024;
}
size_t workspace_bytes(int N, int NO, int D, int H, int W) {
  return ((size_t)pick_splits(N, D, H, W) * NO * D + (size_t)NO * (W + H) + (size_t)NO * 4) * 4 + 256;
}
bool eligible(const void* dout, int D, int H, int W) {
  return shape_ok(D, H, W) && (reinterpret_cast<uintptr_t>(dout) & 15) == 0;
}

}  // namespace bw

// ========================================================================================
// generic backward wrt vecs (any shape): per-tile partial[tile][o_local][d], then an ordered sum over tiles
// ========================================================================================
namespace gen {

constexpr int TILE_W = 64;
constexpr int TILE_H = 8;
constexpr int TILE_PX = TILE_W * TILE_H;
constexpr int NTHREADS = 256;

struct Smem {
  int* list;     // [lcap]            object ids (global) in ascending order
  int* ci;       // [lcap][TILE_W]    first column tap
  float* cw;     // [lcap][TILE_W][2] column tap weights
  int* ri;       // [lcap][TILE_H]
  float* rw;     // [lcap][TILE_H][2]
  float* wS;     // [lcap][TILE_PX]   S_o(y, x) for the tile
  float* vS;     // [lcap][D]         per-object accumulators
};

__device__ __forceinline__ Smem carve(float* base, int lcap, int D) {
  Smem s;
  s.wS = base;                                  // 16B aligned: first
  s.vS = s.wS + (size_t)lcap * TILE_PX;
  s.cw = s.vS + (size_t)lcap * D;
  s.rw = s.cw + (size_t)lcap * TILE_W * 2;
  s.ci = reinterpret_cast<int*>(s.rw + (size_t)lcap * TILE_H * 2);
  s.ri = s.ci + (size_t)lcap * TILE_W;
  s.list = s.ri + (size_t)lcap * TILE_H;
  return s;
}

size_t smem_bytes(int lcap, int D) {
  return sizeof(float) * ((size_t)lcap * TILE_PX + (size_t)lcap * D + (size_t)lcap * TILE_W * 2 +
                          (size_t)lcap * TILE_H * 2 + (size_t)lcap * TILE_W + (size_t)lcap * TILE_H + lcap);
}

template <bool HAS_MASK>
__device__ void build_weights(const LayoutParams& p, const Smem& s, int L, int x0, int y0) {
  const int tid = threadIdx.x;
  const int S = HAS_MASK ? p.M : 8;
  // separable taps: 64 column + 8 row evaluations per object
  for (int i = tid; i < L * (TILE_W + TILE_H); i += NTHREADS) {
    int c = i / (TILE_W + TILE_H), r = i % (TILE_W + TILE_H);
    float4 b = ld_f4(p.boxes + 4 * (size_t)s.list[c]);
    if (r < TILE_W) {
      int x = x0 + r;
      Tap t = axis_tap(p.lin_x[min(x, p.W - 1)], b.x, b.z, S, p.align);
      s.ci[c * TILE_W + r] = t.i0;
      s.cw[(c * TILE_W + r) * 2] = t.w0;
      s.cw[(c * TILE_W + r) * 2 + 1] = t.w1;
    } else {
      r -= TILE_W;
      int y = y0 + r;
      Tap t = axis_tap(p.lin_y[min(y, p.H - 1)], b.y, b.w, S, p.align);
      s.ri[c * TILE_H + r] = t.i0;
      s.rw[(c * TILE_H + r) * 2] = t.w0;
      s.rw[(c * TILE_H + r) * 2 + 1] = t.w1;
    }
  }
  __syncthreads();
  for (int i = tid; i < L * TILE_PX; i += NTHREADS) {
    int c = i / TILE_PX, px = i % TILE_PX;
    int row = px / TILE_W, col = px % TILE_W;
    Tap tx, ty;
    tx.i0 = s.ci[c * TILE_W + col]; tx.w0 = s.cw[(c * TILE_W + col) * 2]; tx.w1 = s.cw[(c * TILE_W + col) * 2 + 1];
    ty.i0 = s.ri[c * TILE_H + row]; ty.w0 = s.rw[(c * TILE_H + row) * 2]; ty.w1 = s.rw[(c * TILE_H + row) * 2 + 1];
    float w;
    if (HAS_MASK) w = mask_weight(p.masks + (size_t)s.list[c] * S * S, S, tx, ty);
    else w = tap_ones(tx, S) * tap_ones(ty, S);
    s.wS[i] = w;
  }
}

constexpr int BWD_CH = 8;   // objects whose 8 weights per pixel slice are kept in registers

// T: element type of the incoming gradient (float, __nv_bfloat16, __half), widened on load
template <bool HAS_MASK, typename T>
__global__ void __launch_bounds__(NTHREADS) layout_bwd_vecs_kernel(LayoutParams p, const T* __restrict__ dout,
                                                                  float* __restrict__ partial) {
  extern __shared__ __align__(16) float smem_raw[];
  __shared__ int s_cursor, s_count;
  const Smem s = carve(smem_raw, p.lcap, p.D);
  const int n = blockIdx.y;
  const int x0 = (blockIdx.x % p.tiles_x) * TILE_W, y0 = (blockIdx.x / p.tiles_x) * TILE_H;
  const int obeg = p.obj_off[n], oend = p.obj_off[n + 1];
  const int On = oend - obeg;
  const int tid = threadIdx.x, lane = tid & 31;
  const int tiles = p.tiles_x * p.tiles_y;
  float* my_partial = partial + ((size_t)tiles * obeg + (size_t)blockIdx.x * On) * p.D;
  for (int i = tid; i < On * p.D; i += NTHREADS) my_partial[i] = 0.f;
  if (tid == 0) s_cursor = obeg;
  __syncthreads();

  const int slice = tid & 63, cg = tid >> 6;       // 64 slices of 8 px, 4 channel groups
  const int row = slice >> 3, col8 = (slice & 7) * 8;
  const int y = y0 + row, x = x0 + col8;
  // 8 pixels per 16-B aligned load pair (fp32) or load (16-bit)
  const bool vec4 = (p.W & (16 / (int)sizeof(T) - 1)) == 0 && (reinterpret_cast<uintptr_t>(dout) & 15) == 0;
  const bool rowok = y < p.H;
  while (true) {
    build_list(p, s.list, oend, x0, y0, &s_cursor, &s_count);
    __syncthreads();
    const int L = s_count;
    const bool more = s_cursor < oend;
    build_weights<HAS_MASK>(p, s, L, x0, y0);
    for (int i = tid; i < L * p.D; i += NTHREADS) s.vS[i] = 0.f;
    __syncthreads();
    for (int cb = 0; cb < L; cb += BWD_CH) {
      float wr[BWD_CH][8];
#pragma unroll
      for (int c = 0; c < BWD_CH; ++c) {
        if (cb + c < L) {
          float4 a = ld_f4(s.wS + (cb + c) * TILE_PX + slice * 8);
          float4 b = ld_f4(s.wS + (cb + c) * TILE_PX + slice * 8 + 4);
          wr[c][0] = a.x; wr[c][1] = a.y; wr[c][2] = a.z; wr[c][3] = a.w;
          wr[c][4] = b.x; wr[c][5] = b.y; wr[c][6] = b.z; wr[c][7] = b.w;
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) wr[c][k] = 0.f;
        }
      }
      for (int d = cg; d < p.D; d += 4) {
        float g[8];
        const T* src = dout + (((size_t)n * p.D + d) * p.H + y) * p.W + x;
        if (rowok && vec4 && x + 7 < p.W) {
          if constexpr (sizeof(T) == 4) {
            float4 a = ld_f4_stream(src), b = ld_f4_stream(src + 4);
            g[0] = a.x; g[1] = a.y; g[2] = a.z; g[3] = a.w; g[4] = b.x; g[5] = b.y; g[6] = b.z; g[7] = b.w;
          } else {
            unpack8_16(__ldcs(reinterpret_cast<const uint4*>(src)), g, std::is_same<T, __half>::value);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) g[k] = (rowok && x + k < p.W) ? to_f32(src[k]) : 0.f;
        }
        float v[BWD_CH];
#pragma unroll
        for (int c = 0; c < BWD_CH; ++c) {
          float a = 0.f;
#pragma unroll
          for (int k = 0; k < 8; ++k) a = fmaf(g[k], wr[c][k], a);
          v[c] = a;
        }
        // transposing butterfly: 8 values x 32 lanes -> lane holds the warp sum of object
        // c = 4*bit4 + 2*bit3 + bit2 of its lane id (9 shuffles instead of 40)
        {
          const bool hi = lane & 16;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float send = hi ? v[i] : v[i + 4];
            float recv = __shfl_xor_sync(0xffffffffu, send, 16);
            v[i] = (hi ? v[i + 4] : v[i]) + recv;
          }
        }
        {
          const bool hi = lane & 8;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            float send = hi ? v[i] : v[i + 2];
            float recv = __shfl_xor_sync(0xffffffffu, send, 8);
            v[i] = (hi ? v[i + 2] : v[i]) + recv;
          }
        }
        {
          const bool hi = lane & 4;
          float send = hi ? v[0] : v[1];
          float recv = __shfl_xor_sync(0xffffffffu, send, 4);
          v[0] = (hi ? v[1] : v[0]) + recv;
        }
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 2);
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
        if ((lane & 3) == 0) {
          int c = cb + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
          // two warps (the two 256-pixel halves of the tile) add into each cell: a + b is order independent
          if (c < L) atomicAdd(&s.vS[c * p.D + d], v[0]);
        }
      }
    }
    __syncthreads();
    for (int i = tid; i < L * p.D; i += NTHREADS) {
      int c = i / p.D, d = i % p.D;
      my_partial[(size_t)(s.list[c] - obeg) * p.D + d] = s.vS[i];
    }
    __syncthreads();
    if (!more) break;
  }
}

__global__ void layout_bwd_reduce_kernel(const float* __restrict__ partial, const int* __restrict__ obj_off,
                                         const int* __restrict__ obj_img, float* __restrict__ dvecs,
                                         int NO, int D, int tiles) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)NO * D) return;
  int o = (int)(i / D), d = (int)(i % D);
  int n = obj_img[o];
  int obeg = obj_off[n], On = obj_off[n + 1] - obeg;
  const float* src = partial + ((size_t)tiles * obeg) * D + (size_t)(o - obeg) * D + d;
  float acc = 0.f;
  for (int t = 0; t < tiles; ++t) acc += src[(size_t)t * On * D];
  dvecs[i] = acc;
}

__global__ void obj_img_kernel(const int* __restrict__ obj_off, int N, int* __restrict__ obj_img) {
  int n = blockIdx.x;
  for (int o = obj_off[n] + threadIdx.x; o < obj_off[n + 1]; o += blockDim.x) obj_img[o] = n;
}

int pick_lcap(int max_objs, int D) {
  int lcap = max_objs > 0 ? max_objs : 16;
  if (lcap < 4) lcap = 4;
  if (lcap > 48) lcap = 48;
  while (lcap > 4 && smem_bytes(lcap, D) > 200 * 1024) lcap -= 4;
  return lcap;
}

size_t workspace_bytes(int NO, int D, int H, int W) {
  size_t tiles = (size_t)csg_div_up(W, TILE_W) * csg_div_up(H, TILE_H);
  return tiles * (size_t)NO * D * sizeof(float) + (size_t)(NO + 1) * sizeof(int) + 256;
}

}  // namespace gen

// ========================================================================================
// backward wrt float masks (masks_to_layout, the training step with predicted masks), band-tiled:
//   dmasks[o, a, b] = sum_{y, x} G_o(y, x) * wy_o(y, a) * wx_o(x, b),   G_o(y, x) = sum_d dout[n, d, y, x] * vecs[o, d]
// A CTA owns (image, range of 256-pixel bands) and reads the gradient of its range once per chunk of lcap objects
// (every channel of a pixel by the same thread), whatever the number of objects covering a pixel: thread = pixel,
// G of up to LC objects in registers, then per-row tap-column sums T[r][b] = sum_x G(y_r, x) wx(x, b) and their fold
// along y into per-(range, object) partials in shared memory, in a fixed order.  A second pass sums each object's
// partials over the ranges its rows meet, in ascending order.  No atomics on floats: runs are bitwise reproducible,
// and a 16-bit gradient gives exactly the result of its fp32 widening.  The weights of an object's taps come from
// the sample coordinates of bw::layout_tables_kernel (the ring kernel's tables).
// ========================================================================================
namespace dm {

constexpr int NTHREADS = bw::BAND;     // thread = pixel of the current band
constexpr int LC = 16;                 // objects whose G a thread holds in registers at a time
constexpr int M_MAX = 32;              // mask sizes served (the tables below grow as M^2)

struct Smem {
  float* vS;     // [lcap][D]      vecs of the chunk's objects
  float* G;      // [lcap][BAND]   G of the current band
  float* T;      // [lcap][RPB][M] per-row tap-column sums of the current band
  float* acc;    // [lcap][M * M]  partial of the CTA's range
  int* bx;       // [lcap][M][2]   canvas-column range feeding mask column b
  int* list;     // [lcap]         chunk-local -> global object id
  int* act;      // [lcap]         chunk-local ids of the objects that touch the current band
};

__host__ __device__ inline int rows_per_band(int W) { return W >= bw::BAND ? 1 : bw::BAND / W; }

__host__ __device__ inline size_t smem_bytes(int lcap, int D, int W, int M) {
  return 4 * ((size_t)lcap * (D + bw::BAND + rows_per_band(W) * M + M * M + 2 * M + 2)) + 16;
}

__device__ __forceinline__ Smem carve(float* base, int lcap, int D, int W, int M) {
  Smem s;
  s.vS = base;
  s.G = s.vS + (size_t)lcap * D;
  s.T = s.G + (size_t)lcap * bw::BAND;
  s.acc = s.T + (size_t)lcap * rows_per_band(W) * M;
  s.bx = reinterpret_cast<int*>(s.acc + (size_t)lcap * M * M);
  s.list = s.bx + (size_t)lcap * M * 2;
  s.act = s.list + lcap;
  return s;
}

struct Params {
  LayoutParams p;
  const void* dout;      // float, __nv_bfloat16 or __half (the kernel's T)
  float* partial;        // [splits][NO][M * M]
  const float* axg;      // [NO][W] column sample coordinates   (bw::layout_tables_kernel<true>)
  const float* ayg;      // [NO][H] row sample coordinates
  const int* rng;        // [NO][4] xmin, xmax, ymin, ymax of the non-zero weights
  int NO, splits, bands_per_item;
};

// Does object o (table row r4, not poisoned) take part in the rows [ylo, yhi]?  The same test picks the objects of a
// CTA and the ranges the sum pass reads, so every partial that is read was written.
__device__ __forceinline__ bool takes_part(int4 r4, int ylo, int yhi) {
  return r4.x <= r4.y && r4.z <= yhi && r4.w >= ylo;
}

template <typename T>
__global__ void __launch_bounds__(NTHREADS, 4) layout_bwd_dmasks_kernel(Params q) {
  CSG_PDL_WAIT();
  extern __shared__ __align__(16) float smem_raw[];
  __shared__ int s_cursor, s_count, s_na;
  const LayoutParams& p = q.p;
  const int S = p.M, MM = S * S;
  const Smem s = carve(smem_raw, p.lcap, p.D, p.W, S);
  const int tid = threadIdx.x, lane = tid & 31;
  const int split = blockIdx.x % q.splits, n = blockIdx.x / q.splits;
  const int obeg = p.obj_off[n], oend = p.obj_off[n + 1];
  const int ncols = min(p.W, bw::BAND), RPB = rows_per_band(p.W);
  const int b0 = split * q.bands_per_item;
  const int row0 = b0 * bw::BAND / p.W;
  const int row1 = ((b0 + q.bands_per_item) * bw::BAND - 1) / p.W;
  const size_t plane = (size_t)p.H * p.W;
  const T* dimg = static_cast<const T*>(q.dout) + (size_t)n * p.D * plane;
  if (tid == 0) s_cursor = obeg;
  __syncthreads();
  while (true) {
    // the next chunk of objects of image n that take part in the CTA's rows, in ascending order
    if (tid < 32) {
      int cursor = s_cursor, count = 0;
      while (cursor < oend && count < p.lcap) {
        const int o = cursor + lane;
        bool keep = false;
        if (o < oend)
          keep = !box_poison(ld_f4(p.boxes + 4 * (size_t)o)) &&
                 takes_part(*reinterpret_cast<const int4*>(q.rng + 4 * (size_t)o), row0, row1);
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        const int pos = count + __popc(bal & ((1u << lane) - 1u));
        if (__popc(bal) <= p.lcap - count) {
          if (keep) s.list[pos] = o;
          count += __popc(bal);
          cursor += 32;
        } else {
          if (keep && pos < p.lcap) s.list[pos] = o;
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
    if (L == 0) break;
    for (int i = tid; i < L * (p.D >> 2); i += NTHREADS) {
      const int c = i / (p.D >> 2), d4 = i % (p.D >> 2);
      st_f4(s.vS + c * p.D + d4 * 4, ld_f4(p.vecs + (size_t)s.list[c] * p.D + d4 * 4));
    }
    for (int i = tid; i < L * MM; i += NTHREADS) s.acc[i] = 0.f;
    for (int i = tid; i < L * S; i += NTHREADS) { s.bx[2 * i] = p.W; s.bx[2 * i + 1] = -1; }
    __syncthreads();
    for (int i = tid; i < L * p.W; i += NTHREADS) {
      const int c = i / p.W, x = i % p.W;
      const Tap t = coord_tap(__ldg(q.axg + (size_t)s.list[c] * p.W + x), S);
      if (t.i0 >= 0 && t.i0 < S) { atomicMin(&s.bx[(c * S + t.i0) * 2], x); atomicMax(&s.bx[(c * S + t.i0) * 2 + 1], x); }
      if (t.i0 + 1 >= 0 && t.i0 + 1 < S) {
        atomicMin(&s.bx[(c * S + t.i0 + 1) * 2], x); atomicMax(&s.bx[(c * S + t.i0 + 1) * 2 + 1], x);
      }
    }
    __syncthreads();

    for (int bb = b0; bb < b0 + q.bands_per_item; ++bb) {
      const int bpix = bb * bw::BAND;
      const int y0 = bpix / p.W, x0 = bpix % p.W;
      // objects of the chunk that touch this band
      if (tid < 32) {
        int na = 0;
        for (int c0 = 0; c0 < L; c0 += 32) {
          const int c = c0 + lane;
          bool keep = false;
          if (c < L) {
            const int4 r4 = *reinterpret_cast<const int4*>(q.rng + 4 * (size_t)s.list[c]);
            keep = r4.z <= y0 + RPB - 1 && r4.w >= y0 && r4.x <= x0 + ncols - 1 && r4.y >= x0;
          }
          const unsigned bal = __ballot_sync(0xffffffffu, keep);
          if (keep) s.act[na + __popc(bal & ((1u << lane) - 1u))] = c;
          na += __popc(bal);
        }
        if (lane == 0) s_na = na;
      }
      __syncthreads();
      const int na = s_na;
      // G of this thread's pixel for LC objects at a time: every channel of the pixel, read in ascending order
      const T* src = dimg + (size_t)bpix + tid;
      for (int k0 = 0; k0 < na; k0 += LC) {
        float g_acc[LC];
#pragma unroll
        for (int k = 0; k < LC; ++k) g_acc[k] = 0.f;
        // (unrolled: 16 gradient loads of the thread in flight, not 4)
#pragma unroll 4
        for (int d = 0; d < p.D; d += 4) {
          const float g0 = to_f32(src[(size_t)d * plane]), g1 = to_f32(src[(size_t)(d + 1) * plane]);
          const float g2 = to_f32(src[(size_t)(d + 2) * plane]), g3 = to_f32(src[(size_t)(d + 3) * plane]);
#pragma unroll
          for (int k = 0; k < LC; ++k) {
            if (k0 + k < na) {
              const float4 v = ld_f4(s.vS + s.act[k0 + k] * p.D + d);
              float a = g_acc[k];
              a = fmaf(g0, v.x, a); a = fmaf(g1, v.y, a); a = fmaf(g2, v.z, a); a = fmaf(g3, v.w, a);
              g_acc[k] = a;
            }
          }
        }
#pragma unroll
        for (int k = 0; k < LC; ++k)
          if (k0 + k < na) s.G[(k0 + k) * bw::BAND + tid] = g_acc[k];
      }
      __syncthreads();
      // per-row tap-column sums, (k, r, b) per thread item
      for (int i = tid; i < na * RPB * S; i += NTHREADS) {
        const int k = i / (RPB * S), r = (i / S) % RPB, b = i % S;
        const int c = s.act[k];
        const float* ax = q.axg + (size_t)s.list[c] * p.W;
        const float* gr = s.G + k * bw::BAND + r * ncols - x0;
        const int xlo = max(s.bx[(c * S + b) * 2], x0), xhi = min(s.bx[(c * S + b) * 2 + 1], x0 + ncols - 1);
        float sum = 0.f;
        for (int x = xlo; x <= xhi; ++x) {
          const Tap t = coord_tap(__ldg(ax + x), S);
          const float w = t.i0 == b ? t.w0 : (t.i0 + 1 == b ? t.w1 : 0.f);
          sum = fmaf(gr[x], w, sum);
        }
        s.T[(k * RPB + r) * S + b] = sum;
      }
      __syncthreads();
      // fold along y into the range's partial (rows in ascending order, bands in ascending order)
      for (int i = tid; i < na * MM; i += NTHREADS) {
        const int k = i / MM, a = (i / S) % S, b = i % S;
        const int c = s.act[k];
        const float* ay = q.ayg + (size_t)s.list[c] * p.H + y0;
        float sum = 0.f;
        for (int r = 0; r < RPB; ++r) {
          const Tap t = coord_tap(__ldg(ay + r), S);
          const float w = t.i0 == a ? t.w0 : (t.i0 + 1 == a ? t.w1 : 0.f);
          sum = fmaf(w, s.T[(k * RPB + r) * S + b], sum);
        }
        s.acc[c * MM + a * S + b] += sum;
      }
      __syncthreads();
    }
    for (int i = tid; i < L * MM; i += NTHREADS) {
      const int c = i / MM;
      q.partial[((size_t)split * q.NO + s.list[c]) * MM + i % MM] = s.acc[i];
    }
    __syncthreads();
    if (!more) break;
  }
}

// dmasks[o] = sum of o's partials over the ranges its rows meet, ascending; NaN for a poisoned box, exact zeros for an
// object that touches nothing (the __image__ dummy, box -1)
__global__ void layout_bwd_dmasks_sum_kernel(const float* __restrict__ partial, const int* __restrict__ rng,
                                             const float* __restrict__ boxes, float* __restrict__ dmasks, int NO, int MM,
                                             int splits, int rows_per_split) {
  CSG_PDL_WAIT();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)NO * MM) return;
  const int o = (int)(i / MM), j = (int)(i % MM);
  if (box_poison(ld_f4(boxes + 4 * (size_t)o))) { dmasks[i] = __int_as_float(0x7fc00000); return; }
  const int4 r4 = *reinterpret_cast<const int4*>(rng + 4 * (size_t)o);
  float acc = 0.f;
  if (r4.x <= r4.y && r4.z <= r4.w)
    for (int sp = r4.z / rows_per_split; sp <= min(r4.w / rows_per_split, splits - 1); ++sp)
      acc += partial[((size_t)sp * NO + o) * MM + j];
  dmasks[i] = acc;
}

int pick_lcap(int D, int W, int M) {
  int lcap = 16;
  while (lcap > 4 && smem_bytes(lcap, D, W, M) > 64 * 1024) lcap -= 4;
  return lcap;
}

// ranges per image: ~4 CTAs per SM in all, fewer when the partials would pass 64 MB
int pick_splits(int N, int NO, int H, int W, int M) {
  const int nbands = H * W / bw::BAND;
  int s = 1;
  // (a range is whole rows: W > 256 takes several bands per row)
  while (s * 2 <= nbands && nbands % (s * 2) == 0 && ((nbands / (s * 2)) * bw::BAND) % W == 0 &&
         (long long)N * s < 4LL * csg_num_sms())
    s *= 2;
  while (s > 1 && (size_t)s * NO * M * M * 4 > ((size_t)64 << 20)) s /= 2;
  return s;
}

bool shape_ok(int D, int H, int W, int M) {
  return bw::shape_ok(D, H, W) && (W == 64 || W == 128 || W % bw::BAND == 0) && M >= 1 && M <= M_MAX &&
         smem_bytes(4, D, W, M) <= 200 * 1024;
}

size_t partial_bytes(int N, int NO, int H, int W, int M) {
  return (size_t)pick_splits(N, NO, H, W, M) * NO * M * M * 4;
}

}  // namespace dm

int fill_params(LayoutParams& p, const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                const float* lin_x, const float* lin_y, int N, int D, int H, int W, int M, int align) {
  CSG_REQUIRE(N >= 0 && D > 0 && H > 0 && W > 0, "layout: bad sizes N=%d D=%d H=%d W=%d", N, D, H, W);
  CSG_REQUIRE(masks == nullptr || M > 0, "layout: masks given but M=%d", M);
  CSG_REQUIRE((D & 3) == 0, "layout: D=%d must be a multiple of 4", D);
  p.vecs = vecs; p.boxes = boxes; p.masks = masks; p.obj_off = obj_off; p.lin_x = lin_x; p.lin_y = lin_y;
  p.N = N; p.D = D; p.H = H; p.W = W; p.M = M; p.align = align;
  return 0;
}

template <typename K>
int set_smem(K kernel, size_t smem) {
  CSG_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return 0;
}

// csg_layout_fwd with a canvas of element type T
template <typename T>
int layout_fwd(const float* vecs, const float* boxes, const float* masks, const int* obj_off, const float* lin_x,
               const float* lin_y, T* out, int N, int D, int H, int W, int M, int align_corners, int max_objs_per_image,
               cudaStream_t stream) {
  LayoutParams p;
  if (int rc = fill_params(p, vecs, boxes, masks, obj_off, lin_x, lin_y, N, D, H, W, M, align_corners)) return rc;
  if (N == 0) return 0;
  CsgProfScope prof(CSG_PROF_LAYOUT_FWD, (double)sizeof(T) * N * D * H * W, stream);
  p.TW = W <= 64 ? 64 : 128;
  p.TH = fw::TILE_PX / p.TW;
  p.tiles_x = csg_div_up(W, p.TW); p.tiles_y = csg_div_up(H, p.TH);
  int lcap = max_objs_per_image > 0 ? max_objs_per_image : 16;
  lcap = (lcap + 3) & ~3;
  if (lcap < 4) lcap = 4;
  if (lcap > 64) lcap = 64;
  // keep at least three CTAs per SM resident
  while (lcap > 4 && fw::smem_floats(lcap, D, p.TW, p.TH, masks != nullptr) * 4 > 72 * 1024) lcap -= 4;
  p.lcap = lcap;
  const size_t smem = fw::smem_floats(lcap, D, p.TW, p.TH, masks != nullptr) * 4;
  CSG_REQUIRE(smem <= 220 * 1024, "layout fwd: D=%d needs %zu bytes of shared memory", D, smem);
  const bool vec_store = (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  CSG_REQUIRE(vec_store, "layout fwd: out must be 16-byte aligned");
  dim3 grid(p.tiles_x * p.tiles_y, N);
  const bool wide = (D % 16) == 0;
#define CSG_FWD_LAUNCH(MASK, CH)                                                          \
  do {                                                                                    \
    if (int rc = set_smem(fw::layout_fwd_kernel<MASK, CH, T>, smem)) return rc;           \
    CSG_CUDA(csg_launch_pdl(fw::layout_fwd_kernel<MASK, CH, T>, grid, dim3(fw::NTHREADS), smem, stream, p, out)); \
  } while (0)
  if (masks) { if (wide) CSG_FWD_LAUNCH(true, 16); else CSG_FWD_LAUNCH(true, 4); }
  else       { if (wide) CSG_FWD_LAUNCH(false, 16); else CSG_FWD_LAUNCH(false, 4); }
#undef CSG_FWD_LAUNCH
  CSG_CHECK_LAUNCH("csg_layout_fwd");
  return 0;
}

// csg_layout_bwd_vecs with an incoming gradient of element type T.  The kernel, its schedule (bands, splits, rows per
// CTA, object chunks) and its summation order are chosen from the shape alone, so a 16-bit gradient gives exactly the
// dvecs of its fp32 widening.  The tcgen05 contraction (CSG_LAYOUT_BWD=tc) takes fp32 gradients only.
template <typename T>
int layout_bwd_vecs(const T* dout, const float* boxes, const float* masks, const int* obj_off, const float* lin_x,
                    const float* lin_y, float* dvecs, int N, int NO, int D, int H, int W, int M, int align_corners,
                    int max_objs_per_image, void* workspace, size_t workspace_bytes, cudaStream_t stream,
                    const float** ring_tables = nullptr) {
  // ring_tables: set to the per-object tables (axg [NO][W], ayg [NO][H], rng [NO][4], contiguous) when the ring or
  // column-sum kernel ran, left alone otherwise
  LayoutParams p;
  if (int rc = fill_params(p, nullptr, boxes, masks, obj_off, lin_x, lin_y, N, D, H, W, M, align_corners)) return rc;
  if (N == 0 || NO == 0) return 0;
  CsgProfScope prof(CSG_PROF_LAYOUT_BWD, (double)sizeof(T) * N * D * H * W, stream);
  CSG_REQUIRE(workspace_bytes >= csg_layout_bwd_vecs_workspace(N, NO, D, H, W), "layout bwd: workspace too small");
  float* partial = reinterpret_cast<float*>(workspace);
  // CSG_LAYOUT_BWD = tc | ring | generic forces a path (benchmarks).  Default: the ring kernel.  The tcgen05 3xTF32
  // contraction (layout_bwd_tc.cu) is bit-compatible with the 1e-5 contract and streams the gradient at 4.9 TB/s when
  // its MMAs are switched off, but a kind::tf32 MMA of M = 128 with a narrow N costs ~180 cycles whatever N is, and
  // the 8 it needs per 32-pixel tile make it MMA-bound at 112 us on the cfg2 canvas (ring kernel: 81 us).
  static const char* force = getenv("CSG_LAYOUT_BWD");
  const bool want_tc = force && force[0] == 't';
  if constexpr (sizeof(T) == 4) {
    if (want_tc && csg_layout_bwd_tc_eligible(dout, N, D, H, W, max_objs_per_image)) {
      // tcgen05 path: dvecs = S * dout^T per image on the tensor cores (layout_bwd_tc.cu); tables as for the ring kernel
      LayoutParams tp = p;
      tp.TW = W; tp.TH = H; tp.tiles_x = tp.tiles_y = 1; tp.lcap = 0;
      float* axg = partial + csg_layout_bwd_tc_partial_floats(N, NO, D, H, W, max_objs_per_image);
      float* ayg = axg + (size_t)NO * W;
      int* rng = reinterpret_cast<int*>(ayg + (size_t)NO * H);
      if (masks) { CSG_CUDA(csg_launch_pdl(bw::layout_tables_kernel<true>, dim3(NO), dim3(128), 0, stream, tp, NO, axg, ayg, rng)); }
      else       { CSG_CUDA(csg_launch_pdl(bw::layout_tables_kernel<false>, dim3(NO), dim3(128), 0, stream, tp, NO, axg, ayg, rng)); }
      CSG_CHECK_LAUNCH("csg_layout_bwd_vecs tables");
      return csg_layout_bwd_tc_launch(dout, masks, obj_off, axg, ayg, partial, dvecs, N, NO, D, H, W, M, max_objs_per_image,
                                      stream);
    }
  }
  if ((!force || force[0] != 'g') && bw::eligible(dout, D, H, W)) {
    bw::Params q;
    q.p = p;
    q.p.TW = W; q.p.TH = H; q.p.tiles_x = q.p.tiles_y = 1;
    q.p.lcap = bw::pick_lcap(max_objs_per_image, H, W, masks != nullptr);
    q.dout = dout; q.partial = partial; q.NO = NO;
    const bool want_cs = !masks && !(force && force[0] == 'r') && bw::cs::shape_ok(H, W);
    q.splits = bw::pick_splits(N, D, H, W, want_cs);
    q.bands_per_item = (H * W) / bw::BAND / q.splits;
    q.cblocks = D / bw::DC;
    float* axg = partial + (size_t)q.splits * NO * D;
    float* ayg = axg + (size_t)NO * W;
    int* rng = reinterpret_cast<int*>(ayg + (size_t)NO * H);
    q.axg = axg; q.ayg = ayg; q.rng = rng;
    if (masks) { CSG_CUDA(csg_launch_pdl(bw::layout_tables_kernel<true>, dim3(NO), dim3(128), 0, stream, q.p, NO, axg, ayg, rng)); }
    else       { CSG_CUDA(csg_launch_pdl(bw::layout_tables_kernel<false>, dim3(NO), dim3(128), 0, stream, q.p, NO, axg, ayg, rng)); }
    CSG_CHECK_LAUNCH("csg_layout_bwd_vecs tables");
    if (ring_tables) *ring_tables = axg;
    const int grid = N * q.cblocks * q.splits;
    const int RR = q.bands_per_item * bw::BAND / W;       // rows per CTA
    if (want_cs && RR <= bw::cs::RR_MAX) {
      // boxes: running column sums + summation by parts along y (layout_bwd_colsum_kernel)
      q.p.lcap = bw::cs::pick_lcap(max_objs_per_image, W, RR);
      const size_t smem = bw::cs::smem_bytes(q.p.lcap, W, RR, bw::Stage<T>::FLOATS);
#define CSG_CS_LAUNCH(SW)                                                                                       \
      do {                                                                                                      \
        if (int rc = set_smem(bw::cs::layout_bwd_colsum_kernel<SW, T>, smem)) return rc;                        \
        CSG_CUDA(csg_launch_pdl(bw::cs::layout_bwd_colsum_kernel<SW, T>, dim3(grid), dim3(bw::NTHREADS), smem, stream, q)); \
      } while (0)
      if (W == 64) CSG_CS_LAUNCH(8); else if (W == 128) CSG_CS_LAUNCH(16); else CSG_CS_LAUNCH(32);
#undef CSG_CS_LAUNCH
      CSG_CHECK_LAUNCH("csg_layout_bwd_vecs colsum");
      const long long n = (long long)NO * D;
      CSG_CUDA(csg_launch_pdl(bw::layout_bwd_sum_splits_kernel, dim3(csg_div_up(n, 256)), dim3(256), 0, stream, partial, dvecs, n, q.splits));
      CSG_CHECK_LAUNCH("csg_layout_bwd_vecs sum");
      return 0;
    }
    const size_t smem = bw::smem_bytes(q.p.lcap, H, W, masks != nullptr, bw::Stage<T>::FLOATS);
    if (masks) {
      if (int rc = set_smem(bw::layout_bwd_ring_kernel<true, T>, smem)) return rc;
      CSG_CUDA(csg_launch_pdl(bw::layout_bwd_ring_kernel<true, T>, dim3(grid), dim3(bw::NTHREADS), smem, stream, q));
    } else {
      if (int rc = set_smem(bw::layout_bwd_ring_kernel<false, T>, smem)) return rc;
      CSG_CUDA(csg_launch_pdl(bw::layout_bwd_ring_kernel<false, T>, dim3(grid), dim3(bw::NTHREADS), smem, stream, q));
    }
    CSG_CHECK_LAUNCH("csg_layout_bwd_vecs ring");
    const long long n = (long long)NO * D;
    CSG_CUDA(csg_launch_pdl(bw::layout_bwd_sum_splits_kernel, dim3(csg_div_up(n, 256)), dim3(256), 0, stream, partial, dvecs, n, q.splits));
    CSG_CHECK_LAUNCH("csg_layout_bwd_vecs sum");
    return 0;
  }
  p.TW = gen::TILE_W; p.TH = gen::TILE_H;
  p.tiles_x = csg_div_up(W, gen::TILE_W); p.tiles_y = csg_div_up(H, gen::TILE_H);
  p.lcap = gen::pick_lcap(max_objs_per_image, D);
  const int tiles = p.tiles_x * p.tiles_y;
  int* obj_img = reinterpret_cast<int*>(partial + (size_t)tiles * NO * D);
  size_t smem = gen::smem_bytes(p.lcap, D);
  dim3 grid(tiles, N);
  gen::obj_img_kernel<<<N, 64, 0, stream>>>(obj_off, N, obj_img);
  if (masks) {
    if (int rc = set_smem(gen::layout_bwd_vecs_kernel<true, T>, smem)) return rc;
    gen::layout_bwd_vecs_kernel<true, T><<<grid, gen::NTHREADS, smem, stream>>>(p, dout, partial);
  } else {
    if (int rc = set_smem(gen::layout_bwd_vecs_kernel<false, T>, smem)) return rc;
    gen::layout_bwd_vecs_kernel<false, T><<<grid, gen::NTHREADS, smem, stream>>>(p, dout, partial);
  }
  CSG_CHECK_LAUNCH("csg_layout_bwd_vecs");
  gen::layout_bwd_reduce_kernel<<<csg_div_up((long long)NO * D, 256), 256, 0, stream>>>(partial, obj_off, obj_img, dvecs,
                                                                                       NO, D, tiles);
  CSG_CHECK_LAUNCH("csg_layout_bwd_reduce");
  return 0;
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

CSG_API size_t csg_layout_bwd_geom_workspace(int NO);
CSG_API int csg_layout_bwd_geom(const float* dout, const float* vecs, const float* boxes, const float* masks,
                                const int* obj_off, const float* lin_x, const float* lin_y, float* dboxes,
                                float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                void* workspace, size_t workspace_bytes, cudaStream_t stream);
CSG_API int csg_layout_bwd_geom_bf16(const void* dout, const float* vecs, const float* boxes, const float* masks,
                                     const int* obj_off, const float* lin_x, const float* lin_y, float* dboxes,
                                     float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                     int fp16, void* workspace, size_t workspace_bytes, cudaStream_t stream);

CSG_API size_t csg_layout_bwd_vecs_masks_workspace(int N, int NO, int D, int H, int W, int M) {
  const size_t vecs = align256(csg_layout_bwd_vecs_workspace(N, NO, D, H, W));
  size_t rest = align256((size_t)NO * 16) + csg_layout_bwd_geom_workspace(NO);       // shapes served by ring + geom
  if (dm::shape_ok(D, H, W, M)) {
    const size_t band = align256((size_t)NO * (W + H + 4) * 4) + dm::partial_bytes(N, NO, H, W, M);
    if (band > rest) rest = band;
  }
  return vecs + rest;
}

namespace {
// csg_layout_bwd_vecs_masks with an incoming gradient of element type T
template <typename T>
int layout_bwd_vecs_masks(const T* dout, const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                          const float* lin_x, const float* lin_y, float* dvecs, float* dmasks, int N, int NO, int D,
                          int H, int W, int M, int align_corners, int max_objs_per_image, void* workspace,
                          size_t workspace_bytes, cudaStream_t stream) {
  CSG_REQUIRE(masks != nullptr && M > 0, "layout bwd vecs+masks: float masks are required");
  CSG_REQUIRE(vecs != nullptr && dvecs != nullptr && dmasks != nullptr, "layout bwd vecs+masks: null vecs / dvecs / dmasks");
  CSG_REQUIRE(workspace_bytes >= csg_layout_bwd_vecs_masks_workspace(N, NO, D, H, W, M),
              "layout bwd vecs+masks: workspace too small");
  if (N == 0 || NO == 0) return 0;
  char* ws = static_cast<char*>(workspace);
  const size_t vb = align256(csg_layout_bwd_vecs_workspace(N, NO, D, H, W));
  const float* tables = nullptr;
  // d vecs: exactly csg_layout_bwd_vecs
  if (int rc = layout_bwd_vecs(dout, boxes, masks, obj_off, lin_x, lin_y, dvecs, N, NO, D, H, W, M, align_corners,
                               max_objs_per_image, ws, vb, stream, &tables))
    return rc;
  char* rest = ws + vb;
  if (!dm::shape_ok(D, H, W, M) || !bw::eligible(dout, D, H, W)) {
    // shapes the ring kernel does not serve: d masks from the per-object kernel (layout_geom.cu), as before
    float* dboxes = reinterpret_cast<float*>(rest);
    void* gws = rest + align256((size_t)NO * 16);
    const size_t gbytes = csg_layout_bwd_geom_workspace(NO);
    if constexpr (sizeof(T) == 4)
      return csg_layout_bwd_geom(dout, vecs, boxes, masks, obj_off, lin_x, lin_y, dboxes, dmasks, N, NO, D, H, W, M,
                                 align_corners, gws, gbytes, stream);
    else
      return csg_layout_bwd_geom_bf16(dout, vecs, boxes, masks, obj_off, lin_x, lin_y, dboxes, dmasks, N, NO, D, H, W,
                                      M, align_corners, (int)std::is_same<T, __half>::value, gws, gbytes, stream);
  }
  dm::Params q;
  if (int rc = fill_params(q.p, vecs, boxes, masks, obj_off, lin_x, lin_y, N, D, H, W, M, align_corners)) return rc;
  q.p.TW = W; q.p.TH = H; q.p.tiles_x = q.p.tiles_y = 1;
  float* own = reinterpret_cast<float*>(rest);
  if (!tables) {
    // the ring kernel did not run (CSG_LAYOUT_BWD forced another d vecs path): the same tables, here
    CSG_CUDA(csg_launch_pdl(bw::layout_tables_kernel<true>, dim3(NO), dim3(128), 0, stream, q.p, NO, own,
                            own + (size_t)NO * W, reinterpret_cast<int*>(own + (size_t)NO * (W + H))));
    CSG_CHECK_LAUNCH("csg_layout_bwd_vecs_masks tables");
    tables = own;
  }
  q.dout = dout;
  q.partial = reinterpret_cast<float*>(rest + align256((size_t)NO * (W + H + 4) * 4));
  q.axg = tables; q.ayg = tables + (size_t)NO * W; q.rng = reinterpret_cast<const int*>(tables + (size_t)NO * (W + H));
  q.NO = NO;
  q.splits = dm::pick_splits(N, NO, H, W, M);
  q.bands_per_item = H * W / bw::BAND / q.splits;
  q.p.lcap = dm::pick_lcap(D, W, M);
  const size_t smem = dm::smem_bytes(q.p.lcap, D, W, M);
  if (int rc = set_smem(dm::layout_bwd_dmasks_kernel<T>, smem)) return rc;
  CSG_CUDA(csg_launch_pdl(dm::layout_bwd_dmasks_kernel<T>, dim3(N * q.splits), dim3(dm::NTHREADS), smem, stream, q));
  CSG_CHECK_LAUNCH("csg_layout_bwd_vecs_masks dmasks");
  const long long n = (long long)NO * M * M;
  CSG_CUDA(csg_launch_pdl(dm::layout_bwd_dmasks_sum_kernel, dim3(csg_div_up(n, 256)), dim3(256), 0, stream,
                          (const float*)q.partial, q.rng, boxes, dmasks, NO, M * M, q.splits,
                          q.bands_per_item * bw::BAND / W));
  CSG_CHECK_LAUNCH("csg_layout_bwd_vecs_masks sum");
  return 0;
}
}  // namespace

// ----------------------------------------------------------------------------------------
// C ABI
// ----------------------------------------------------------------------------------------
CSG_API int csg_layout_fwd(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                           const float* lin_x, const float* lin_y, float* out, int N, int D, int H, int W,
                           int M, int align_corners, int max_objs_per_image, cudaStream_t stream) {
  return layout_fwd(vecs, boxes, masks, obj_off, lin_x, lin_y, out, N, D, H, W, M, align_corners, max_objs_per_image,
                    stream);
}

CSG_API int csg_layout_fwd_bf16(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                                const float* lin_x, const float* lin_y, void* out, int N, int D, int H, int W,
                                int M, int align_corners, int max_objs_per_image, int fp16, cudaStream_t stream) {
  if (fp16)
    return layout_fwd(vecs, boxes, masks, obj_off, lin_x, lin_y, static_cast<__half*>(out), N, D, H, W, M,
                      align_corners, max_objs_per_image, stream);
  return layout_fwd(vecs, boxes, masks, obj_off, lin_x, lin_y, static_cast<__nv_bfloat16*>(out), N, D, H, W, M,
                    align_corners, max_objs_per_image, stream);
}

CSG_API size_t csg_layout_bwd_vecs_workspace(int N, int NO, int D, int H, int W) {
  size_t need = gen::workspace_bytes(NO, D, H, W);
  if (bw::shape_ok(D, H, W)) {
    size_t ring = bw::workspace_bytes(N, NO, D, H, W);
    if (ring > need) need = ring;
  }
  if (N > 0 && (D % 128) == 0 && (W % 32) == 0) {
    size_t tc = (csg_layout_bwd_tc_partial_floats(N, NO, D, H, W, 16) + (size_t)NO * (W + H) + (size_t)NO * 4) * 4 + 256;
    if (tc > need) need = tc;
  }
  return need;
}

CSG_API int csg_layout_bwd_vecs(const float* dout, const float* boxes, const float* masks, const int* obj_off,
                                const float* lin_x, const float* lin_y, float* dvecs, int N, int NO, int D,
                                int H, int W, int M, int align_corners, int max_objs_per_image,
                                void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  return layout_bwd_vecs(dout, boxes, masks, obj_off, lin_x, lin_y, dvecs, N, NO, D, H, W, M, align_corners,
                         max_objs_per_image, workspace, workspace_bytes, stream);
}

CSG_API int csg_layout_bwd_vecs_bf16(const void* dout, const float* boxes, const float* masks, const int* obj_off,
                                     const float* lin_x, const float* lin_y, float* dvecs, int N, int NO, int D,
                                     int H, int W, int M, int align_corners, int max_objs_per_image, int fp16,
                                     void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (fp16)
    return layout_bwd_vecs(static_cast<const __half*>(dout), boxes, masks, obj_off, lin_x, lin_y, dvecs, N, NO, D, H, W,
                           M, align_corners, max_objs_per_image, workspace, workspace_bytes, stream);
  return layout_bwd_vecs(static_cast<const __nv_bfloat16*>(dout), boxes, masks, obj_off, lin_x, lin_y, dvecs, N, NO, D,
                         H, W, M, align_corners, max_objs_per_image, workspace, workspace_bytes, stream);
}

CSG_API int csg_layout_bwd_vecs_masks(const float* dout, const float* vecs, const float* boxes, const float* masks,
                                      const int* obj_off, const float* lin_x, const float* lin_y, float* dvecs,
                                      float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                      int max_objs_per_image, void* workspace, size_t workspace_bytes,
                                      cudaStream_t stream) {
  return layout_bwd_vecs_masks(dout, vecs, boxes, masks, obj_off, lin_x, lin_y, dvecs, dmasks, N, NO, D, H, W, M,
                               align_corners, max_objs_per_image, workspace, workspace_bytes, stream);
}

CSG_API int csg_layout_bwd_vecs_masks_bf16(const void* dout, const float* vecs, const float* boxes, const float* masks,
                                           const int* obj_off, const float* lin_x, const float* lin_y, float* dvecs,
                                           float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                           int max_objs_per_image, int fp16, void* workspace, size_t workspace_bytes,
                                           cudaStream_t stream) {
  if (fp16)
    return layout_bwd_vecs_masks(static_cast<const __half*>(dout), vecs, boxes, masks, obj_off, lin_x, lin_y, dvecs,
                                 dmasks, N, NO, D, H, W, M, align_corners, max_objs_per_image, workspace,
                                 workspace_bytes, stream);
  return layout_bwd_vecs_masks(static_cast<const __nv_bfloat16*>(dout), vecs, boxes, masks, obj_off, lin_x, lin_y,
                               dvecs, dmasks, N, NO, D, H, W, M, align_corners, max_objs_per_image, workspace,
                               workspace_bytes, stream);
}
