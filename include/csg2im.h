/* csg2im.h -- C ABI of libcsg2im.so: B200 (sm_100a) kernels for the scene-graph -> layout hot
 * path of roeiherz/CanonicalSg2Im.
 *
 * The reference has no FFI of its own: the path is plain Python/PyTorch
 * (sg2im/graph.py, sg2im/layout.py, sg2im/bilinear.py, sg2im/data/base_dataset.py,
 * scripts/graphs_utils.py).  These entry points are what a ctypes binding on the reference side
 * would call (see INTEGRATION.md); canonicalsg2im_b200/_lib.py is exactly such a binding.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless stated otherwise; the caller owns all inputs,
 *    outputs and workspaces, the library never allocates or frees device memory and keeps no
 *    state between calls (re-entrant; honours the current device and the stream passed in);
 *  - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *  - all functions return 0 on success; on failure a non-zero code, and csg_last_error()
 *    returns a thread-local message.  No exception crosses the ABI.  Kernel launch errors are
 *    reported by the call that launched (cudaGetLastError), never deferred;
 *  - batches are FLAT: objects [NO, .] and triples [NT, .] with per-graph ranges obj_off[B+1] /
 *    tri_off[B+1].  The reference's padded [B, O, .] / [B, T, .] tensors are the special case
 *    obj_off[b] = b*O, tri_off[b] = b*T;
 *  - boxes are [x0, y0, w, h] (sg2im/layout.py:95-96).
 */
#ifndef CSG2IM_H_
#define CSG2IM_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* csg_stream_t;

/* ---- library ---------------------------------------------------------------------------- */
const char* csg_last_error(void);
void csg_clear_error(void);
int csg_version(void);
int csg_device_sms(void);
long long csg_launch_count(void);   /* kernel-launch sites passed since the library was loaded */
/* Asynchronous index errors: kernels that use caller-supplied integers as offsets (triple subject / object /
 * predicate ids, embedding ids, canonicalization triplets) neutralise an out-of-range row and report it in a
 * pinned host record instead of reading out of bounds; the reference raises IndexError on the same inputs
 * (sg2im/graph.py:63-64,73,98-103, sg2im/model.py:108-109).  out4 (HOST, may be NULL) <- {code, row, value, limit};
 * returns the code (0 none, 1 triple subject/object, 2 triple predicate, 3 embedding id, 4 canonicalization
 * triplet) and clears the record.  Never synchronises: an error is visible once its kernel has run. */
int csg_async_error_poll(int* out4);
/* Live timing of kernel classes (measurement aid, off by default): while enabled, the instrumented entry points
 * record CUDA events on their stream.  csg_prof_collect fills a HOST array [8][3] = {work, seconds, calls} per
 * class (0 bf16 GEMMs: FLOP, 1 fp32 GEMMs: FLOP, 2 layout fwd: bytes, 3 layout bwd: bytes, 4 pooling: bytes,
 * 5 backward assemble: bytes) and clears the records; it synchronises on the recorded events. */
int csg_prof_enable(int on);
int csg_prof_collect(double* out);

/* ---- layout compositor: sg2im/layout.py:12-45 (boxes_to_layout), :48-77 (masks_to_layout),
 *      :80-112 (_boxes_to_grid), :156-188 (_pool_samples), batched over images as the caller
 *      loop spade/models/networks/generator.py:81-96 does ------------------------------------ */
/* out[n, d, y, x] = sum_{o in image n} vecs[o, d] * S_o(y, x);  masks == NULL selects boxes_to_layout.
 * lin_x[W], lin_y[H] = torch.linspace(0, 1, steps) in fp32 (layout.py:98-99).  out is fully written. */
int csg_layout_fwd(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                   const float* lin_x, const float* lin_y, float* out, int N, int D, int H, int W,
                   int M, int align_corners, int max_objs_per_image, csg_stream_t stream);
size_t csg_layout_bwd_vecs_workspace(int N, int NO, int D, int H, int W);
/* dvecs[o, d] = sum_{y, x} dout[n(o), d, y, x] * S_o(y, x)  (autograd of the above wrt vecs) */
int csg_layout_bwd_vecs(const float* dout, const float* boxes, const float* masks, const int* obj_off,
                        const float* lin_x, const float* lin_y, float* dvecs, int N, int NO, int D,
                        int H, int W, int M, int align_corners, int max_objs_per_image,
                        void* workspace, size_t workspace_bytes, csg_stream_t stream);

/* masks_to_layout(test_mode=True), sg2im/layout.py:72-76 + _pool_mask_samples :135-147: objects are visited in
 * ascending order of their total sampled mass; the first one whose clean mask sample is > 0.5 owns the pixel
 * (out = vecs[owner] * S_owner, 0 where nobody does).  Inference only; no host synchronisation. */
size_t csg_layout_occlude_workspace(int N, int NO);
int csg_layout_occlude_fwd(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                           const float* lin_x, const float* lin_y, float* out, int N, int NO, int D, int H,
                           int W, int M, int align_corners, void* workspace, size_t workspace_bytes,
                           csg_stream_t stream);
/* autograd of csg_layout_fwd wrt boxes [NO,4] (always) and wrt float masks [NO,M,M] (dmasks may be NULL):
 * F.grid_sample backward (bilinear, zero padding) chained through _boxes_to_grid, layout.py:80-112 */
size_t csg_layout_bwd_geom_workspace(int NO);
int csg_layout_bwd_geom(const float* dout, const float* vecs, const float* boxes, const float* masks,
                        const int* obj_off, const float* lin_x, const float* lin_y, float* dboxes,
                        float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                        void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* 16-bit canvases (fp16 = 0: bf16, 1: fp16).  Forward: `out` is the fp32 canvas of the entry point above rounded once
 * to nearest even (Tensor.to: fp16 overflow is +-inf, NaN stays NaN).  Backward: `dout` is widened on load; dvecs,
 * dboxes and dmasks are bitwise those of the fp32 entry points given the widened gradient.  vecs, boxes, masks and
 * all gradients stay fp32; the workspace queries above apply unchanged. */
int csg_layout_fwd_bf16(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                        const float* lin_x, const float* lin_y, void* out, int N, int D, int H, int W,
                        int M, int align_corners, int max_objs_per_image, int fp16, csg_stream_t stream);
int csg_layout_bwd_vecs_bf16(const void* dout, const float* boxes, const float* masks, const int* obj_off,
                             const float* lin_x, const float* lin_y, float* dvecs, int N, int NO, int D,
                             int H, int W, int M, int align_corners, int max_objs_per_image, int fp16,
                             void* workspace, size_t workspace_bytes, csg_stream_t stream);
int csg_layout_occlude_fwd_bf16(const float* vecs, const float* boxes, const float* masks, const int* obj_off,
                                const float* lin_x, const float* lin_y, void* out, int N, int NO, int D, int H,
                                int W, int M, int align_corners, int fp16, void* workspace, size_t workspace_bytes,
                                csg_stream_t stream);
int csg_layout_bwd_geom_bf16(const void* dout, const float* vecs, const float* boxes, const float* masks,
                             const int* obj_off, const float* lin_x, const float* lin_y, float* dboxes,
                             float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                             int fp16, void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* autograd of csg_layout_fwd wrt vecs and float masks [NO,M,M] together, boxes held fixed (the training step with
 * predicted masks on GT boxes).  dvecs is bitwise that of csg_layout_bwd_vecs.  On shapes the ring kernel serves
 * (W % 64 == 0 with W = 64, 128 or a multiple of 256, H*W % 256 == 0, D % 32 == 0, M <= 32, 16-byte aligned dout)
 * dmasks comes from a band-tiled kernel that reads dout once more per chunk of 16 objects (fp32 sums in a fixed
 * order, deterministic); on other shapes from csg_layout_bwd_geom.  Either way a poisoned box (zero / NaN extent,
 * non-finite origin) gives a NaN dmasks row and an object that touches no pixel an exact-zero row.  The _bf16 form
 * takes a bf16 (fp16 = 0) or fp16 (fp16 = 1) gradient, widened on load: results are bitwise those of its widening. */
size_t csg_layout_bwd_vecs_masks_workspace(int N, int NO, int D, int H, int W, int M);
int csg_layout_bwd_vecs_masks(const float* dout, const float* vecs, const float* boxes, const float* masks,
                              const int* obj_off, const float* lin_x, const float* lin_y, float* dvecs,
                              float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                              int max_objs_per_image, void* workspace, size_t workspace_bytes, csg_stream_t stream);
int csg_layout_bwd_vecs_masks_bf16(const void* dout, const float* vecs, const float* boxes, const float* masks,
                                   const int* obj_off, const float* lin_x, const float* lin_y, float* dvecs,
                                   float* dmasks, int N, int NO, int D, int H, int W, int M, int align_corners,
                                   int max_objs_per_image, int fp16, void* workspace, size_t workspace_bytes,
                                   csg_stream_t stream);

/* ---- box crops: sg2im/bilinear.py:65-94 (crop_bbox, backend 'cudnn'), :44-62 (crop_bbox_batch_cudnn).
 *      Crops crop_off[n]..crop_off[n+1] sample image n of feats [N,C,H,W] in place (the reference expands the
 *      image once per object); bbox [NC,4] xywh; swx/ewx [WW], swy/ewy [HH] = torch.linspace(1,0,.) / (0,1,.)
 *      in fp32 (tensor_linspace, bilinear.py:155-184).  crops [NC,C,HH,WW].  align_corners: 0 / 1 = the two
 *      F.grid_sample conventions of backend 'cudnn'; 2 = backend 'jj' (bilinear_sample, bilinear.py:97-152: [0, 1]
 *      coordinates scaled by the image size, taps clamped into the image). ------------------------------------ */
size_t csg_crop_bbox_workspace(int NC);
int csg_crop_bbox_fwd(const float* feats, const float* bbox, const int* crop_off, const float* swx,
                      const float* ewx, const float* swy, const float* ewy, float* crops, int N, int NC,
                      int C, int H, int W, int HH, int WW, int align_corners, void* workspace,
                      size_t workspace_bytes, csg_stream_t stream);
/* dfeats [N,C,H,W] (fully written) = autograd of the above wrt feats; deterministic gather */
int csg_crop_bbox_bwd(const float* dcrops, const float* bbox, const int* crop_off, const float* swx,
                      const float* ewx, const float* swy, const float* ewy, float* dfeats, int N, int NC,
                      int C, int H, int W, int HH, int WW, int align_corners, csg_stream_t stream);

/* ---- triple graph convolution: sg2im/graph.py:44-113 ---------------------------------------- */
int csg_offsets_uniform(int* off, int B, int stride, csg_stream_t stream);
/* model.py:104-107 + graph.py:60-61: split int64 triplets, globalise indices, valid = (p != padding).
 * Subject / object ids outside [0, n_g) and (when num_preds > 0) predicate ids outside [0, num_preds) -- where the
 * reference raises IndexError -- neutralise the row and are reported through csg_async_error_poll. */
int csg_triple_prep(const long long* triplets, const long long* triplet_type, const int* tri_off,
                    const int* obj_off, int B, int NT, int T_pad, int O_pad, int padding_id, int num_preds,
                    int* s_idx, int* o_idx, int* pred, int* type32, int* valid, csg_stream_t stream);
/* same, from GraphTripleConv.forward's argument layout (graph.py:44): edges [NT,2], predicate ids,
 * pred_indicators (uint8/bool, may be NULL = all valid) */
int csg_triple_prep_edges(const long long* edges, const long long* pred_ids, const unsigned char* indicators,
                          const long long* triplet_type, const int* tri_off, const int* obj_off, int B,
                          int NT, int T_pad, int O_pad, int num_preds, int* s_idx, int* o_idx, int* pred,
                          int* type32, int* valid, csg_stream_t stream);
/* stable CSR orderings by subject and by object (replace scatter_add, graph.py:98-103) */
size_t csg_csr_workspace(int NO);
int csg_csr_build(const int* keys_s, const int* keys_o, const int* tri_off, const int* obj_off, int B, int NT, int NO,
                  int* rowptr_s, int* perm_s, int* rowptr_o, int* perm_o,
                  void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* graph.py:69-74 */
int csg_triple_conf(const int* type32, const int* pred, const float* w_trans, int NT, float* conf,
                    csg_stream_t stream);
/* graph.py:85-107 (avg = 1) or a plain segmented sum (avg = 0, backward of the gathers graph.py:63-64) */
int csg_segpool_f32(const float* X, int ldx, int col_s, int col_o, int W,
                    const int* rowptr_s, const int* perm_s, const int* rowptr_o, const int* perm_o,
                    const int* valid, const float* conf, int NO, float* out, int ldo, float* cnt_out,
                    int avg, csg_stream_t stream);
int csg_pool_bwd_obj(const float* dpooled, const float* pooled, const float* cnt, int NO, int W,
                     float* dS, float* dcnt, csg_stream_t stream);
int csg_triple_bwd_assemble(const float* out, const float* dS, const float* d_newp, const float* dcnt,
                            const int* s_idx, const int* o_idx, const int* valid, const int* type32,
                            const float* conf, int NT, int H, int Dp, float* g, float* dconf,
                            csg_stream_t stream);
size_t csg_conf_bwd_workspace(int P);
int csg_conf_bwd(const float* dconf, const int* type32, const int* pred, const float* w_trans, int NT, int P,
                 float* dw, void* workspace, size_t workspace_bytes, csg_stream_t stream);

/* ---- MLPs (net1 / net2 / box_net: graph.py:33-41,67,110; model.py:58-60,115; layers.py:6-25) --- */
/* fp32 SIMT GEMM with fused gather / bias / ReLU / confidence / ReLU-mask epilogues.
 * amode: 0 A[m,k]  1 A[k,m]  2 gathered triple rows;  bmode: 0 B[n,k]  1 B[k,n]  2 gathered rows. */
size_t csg_gemm_f32_workspace(int M, int N, int K, int amode);
int csg_gemm_f32(int amode, int bmode, int M, int N, int K,
                 const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                 const float* bias, int relu, const float* rowscale,
                 const float* mask_aux, int ld_aux,
                 const float* g_obj, const float* g_pred, const int* g_sidx, const int* g_oidx,
                 int g_din, int g_dp, int g_ldp,
                 void* workspace, size_t workspace_bytes, csg_stream_t stream);
int csg_relu_mask_f32(const float* dy, const float* y, float* out, long long n, csg_stream_t stream);
size_t csg_colsum_f32_workspace(int M, int N);
int csg_colsum_f32(const float* X, int M, int N, int ld, float* out, void* workspace, size_t workspace_bytes,
                   csg_stream_t stream);

/* bf16 tensor-core GEMMs (tcgen05 + TMEM + TMA), fp32 accumulation.
 * mn_major = 0: C[M,N] = epi(A[M,K] B[N,K]^T), K contiguous; gather = 1 fuses the triple-input gather into A.
 * mn_major = 1: C[M,N] = A[K,M]^T B[K,N] (weight gradients, fp32 out, split-K); gather = 2 gathers B's rows.
 * The gathered operand is the virtual row [g_obj[g_sidx[t]] | g_pred[t] | g_obj[g_oidx[t]]] (graph.py:63-66);
 * g_obj is [g_nobj, g_din] contiguous, g_pred has row pitch g_ldp.  Object rows arrive by TMA tile::gather4.
 * g_pidx (may be NULL) [rows] int32: the predicate segment is gathered as well, g_pred then being a TABLE of g_npred
 * rows and the virtual row [g_obj[g_sidx[t]] | g_pred[g_pidx[t]] | g_obj[g_oidx[t]]] -- with g_obj the object
 * embedding table and g_sidx / g_oidx class ids this is layer 0 reading straight from the embedding tables
 * (sg2im/model.py:108-109), no [NT, Dp] / [NO, Din] rows materialised.
 * A, B, mask_aux, g_obj, g_pred are 16-bit floats; bias, rowscale fp32; C is 16-bit or (out_f32) fp32.
 * formats selects the 16-bit element formats per operand (tcgen05 kind::f16 takes fp16 and bf16, independently for A
 * and B): bit 0 = A (or the gathered rows when gather = 1) is fp16, bit 1 = B (or the gathered rows when gather = 2)
 * is fp16, bit 2 = a 16-bit C is written as fp16 (saturating at +-65504); a clear bit means bf16.  The engine keeps
 * FORWARD tensors (activations, weights) in fp16 -- 11 significant bits instead of bf16's 8 at the same tensor-pipe
 * rate -- and GRADIENT tensors in bf16 (fp16 cannot hold their range).  mask_aux is only tested for > 0. */
size_t csg_gemm_bf16_workspace(int M, int N, int K, int mn_major);
int csg_gemm_bf16(int mn_major, int gather, int M, int N, int K,
                  const void* A, int lda, const void* B, int ldb, void* C, int ldc, int out_f32,
                  const float* bias, int relu, const float* rowscale, const void* mask_aux, int ld_aux,
                  const void* g_obj, const void* g_pred, const int* g_sidx, const int* g_oidx,
                  int g_din, int g_dp, int g_ldp, int g_nobj, const int* g_pidx, int g_npred, int formats,
                  void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* CTA-pair policy of the K-major GEMMs (tcgen05.mma.cta_group::2, 256 x N pair tiles, each CTA stages half of B):
 * -1 automatic (default: pairs once M >= 2 * 128 * #SMs and K >= 1024), 0 never, 1 whenever the shape allows.
 * Process-wide. */
void csg_gemm_bf16_set_pair_mode(int mode);

/* bf16-activation twins of the pooling / assembly kernels (fp32 accumulation) + weight cast */
int csg_cast_bf16(const float* src, int rows, int cols, int ld_src, void* dst, int ld_dst, int transpose, int fp16,
                  csg_stream_t stream);
/* n <= 64 contiguous fp32 matrices -> contiguous 16-bit copies (transposed when transpose[i]; fp16 when fp16, else
 * bf16); HOST arrays */
int csg_cast_bf16_multi(int n, const void* const* src, void* const* dst, const int* rows, const int* cols,
                        const int* transpose, int fp16, csg_stream_t stream);
int csg_segpool_bf16(const void* X, int ldx, int col_s, int col_o, int W,
                     const int* rowptr_s, const int* perm_s, const int* rowptr_o, const int* perm_o,
                     const int* valid, const float* conf, int NO, float* out_f32, void* out_bf16, int ldo,
                     float* cnt_out, int avg, int fp16, csg_stream_t stream);   /* fp16: X and out_bf16 hold fp16 */
/* out[o, 0:W] = sum over the triples whose subject is o of X[t, 0:W]; out[o, W:2W] = the same over the triples whose
 * object is o (fixed order: ascending triple id).  The per-object sums of d hidden that give net1's first-layer weight /
 * bias / object-row gradients without a gathered GEMM over the triples (sg2im/graph.py:60-67 backward). */
int csg_segsum2_bf16(const void* X, int ldx, int W, const int* rowptr_s, const int* perm_s, const int* rowptr_o,
                     const int* perm_o, int NO, float* out_f32, void* out_bf16, int ldo, csg_stream_t stream);
/* fp32 accuracy on tcgen05: x = hi + mid + lo (three bf16 terms = the 24 significant bits of fp32) and a b ~= the six
 * products of parts down to 2^-24 |a b|, accumulated in fp32 -- as ONE bf16 GEMM with a 6x longer reduction: this writes an
 * operand with its parts concatenated along the reduction dimension (k_is_cols: out [R, 6 C], else out [6 R, C]; [R, C] = X or,
 * with `transpose`, X^T) in the order (mid, lo, hi, mid, hi, hi) for role 0 (A) / (mid, hi, lo, hi, mid, hi) for role 1 (B):
 * smallest products first, hi*hi last.  role 2 / 3: the hi block alone; role 4 / 5: the five correction blocks (out is then
 * [R, C] / [R, 5 C] resp. [R, C] / [5 R, C]).
 * The 1e-5 parity engine of sg2im/graph.py:33-41,67,110 on tensor cores instead of fp32 FMA pipes (ops.gemm_f32). */
int csg_split3_bf16(const float* X, int rows, int cols, int ld, int transpose, int k_is_cols, int role, void* out,
                    int ld_out, csg_stream_t stream);
int csg_relu_mask_bf16(const float* dy, const void* y, void* out, long long n, csg_stream_t stream);
size_t csg_colsum_bf16_workspace(int M, int N);
int csg_colsum_bf16(const void* X, int M, int N, int ld, float* out, void* workspace, size_t workspace_bytes,
                    csg_stream_t stream);
size_t csg_triple_bwd_assemble_bf16_workspace(int NT, int H, int Dp);
/* colsum_g (may be NULL): [2H+Dp] fp32 column sums of g = the bias gradient of net1's second Linear, fused */
int csg_triple_bwd_assemble_bf16(const void* out, const float* dS, const void* d_newp, int ld_newp,
                                 const float* dcnt, const int* s_idx, const int* o_idx, const int* valid,
                                 const int* type32, const float* conf, int NT, int H, int Dp, void* g,
                                 float* dconf, float* colsum_g, int out_fp16, void* workspace, size_t workspace_bytes,
                                 csg_stream_t stream);   /* out_fp16: `out` holds fp16; d_newp and g are bf16 */

/* ---- one GraphTripleConv layer (sg2im/graph.py:44-113) per call on the bf16 engine: the launch sequence of the
 *      stages above issued natively, out of caller-owned `saved` (activations kept for backward + bf16 weights)
 *      and `workspace` (scratch).  dims (HOST int[11]) = {NT, NO, Din, Dp, H, Dout, Dpo, P, fwd_fp16, n_gather, n_pred};
 *      all widths % 64 == 0; fwd_fp16 = 1 keeps the forward tensors (obj, pred, weights, hidden, net1 output, pooled,
 *      net2 hidden, new_obj) in fp16 instead of bf16 (inference only) -- gradient tensors are bf16 either way.
 *      n_gather > 0 / n_pred > 0 (layer 0 fused with the embedding lookups, sg2im/model.py:108-109): `obj` is the object
 *      embedding TABLE [n_gather, Din] gathered by the per-triple class ids index[9] (subjects) / index[10] (objects),
 *      `pred` the predicate embedding TABLE [n_pred, Dp] gathered by index[11]; dobj is still per object [NO, Din] (the
 *      caller folds it onto the table by class id) and dX's predicate columns per triple.
 *      params (HOST array of 9 device pointers, fp32): net1.0.weight [H, 2Din+Dp], net1.0.bias, net1.2.weight
 *      [2H+Dpo, H], net1.2.bias, net2.0.weight [H, H], net2.0.bias, net2.2.weight [Dout, H], net2.2.bias,
 *      predicates_transitive_weights [P].  index (HOST array of 9 device pointers, int32): s_idx, o_idx, pred_id,
 *      type32, valid [NT] (csg_triple_prep) and rowptr_s, perm_s, rowptr_o, perm_o (csg_csr_build); with the fused
 *      layer 0 three more: subject class ids, object class ids, predicate ids [NT] (index is then void*[12]). ---- */
size_t csg_gconv_bf16_saved_bytes(const int* dims, int need_bwd);
size_t csg_gconv_bf16_out_offset(const int* dims, int need_bwd);   /* byte offset in `saved` of net1's output [NT, 2H+Dpo] bf16 */
size_t csg_gconv_bf16_workspace(const int* dims);
int csg_gconv_bf16_dx_cols(const int* dims);   /* columns of the dX matrix csg_gconv_bf16_bwd writes: Dp, or 2Din+Dp (layer on the embedding tables, CSG_BWD_SEGSUM=0) */
/* obj [NO, Din] bf16 contiguous, pred [NT, Dp] bf16 rows of pitch ldp -> new_obj [NO, Dout] bf16; new_p_vecs are
 * columns H..H+Dpo of the [NT, 2H+Dpo] matrix at saved + csg_gconv_bf16_out_offset.  `saved` 256-byte aligned. */
int csg_gconv_bf16_fwd(const int* dims, const void* obj, const void* pred, int ldp,
                       const void* const* params, const void* const* index, int need_bwd, void* saved,
                       size_t saved_bytes, void* new_obj, const void* wbuf, const float* conf_ext, csg_stream_t stream);
/* d_new_obj [NO, Dout] fp32 or (d_new_obj_bf16) bf16, NULL = 0; d_new_p [NT, Dpo] bf16 rows of pitch ld_dnewp,
 * NULL = 0.  Writes dobj [NO, Din] fp32 or (dobj_bf16) bf16, dX [NT, csg_gconv_bf16_dx_cols] bf16 (d pred; on the gathered
 * dataflow the whole row [d obj[s] | d pred | d obj[o]])
 * and dparams: fp32, contiguous, 16-byte aligned, in the order of `params` (dw1, db1, dw2, db2, dw3, db3, dw4,
 * db4, dw_trans). */
int csg_gconv_bf16_bwd(const int* dims, const void* obj, const void* pred, int ldp,
                       const void* const* params, const void* const* index,
                       const void* d_new_obj, int d_new_obj_bf16, const void* d_new_p, int ld_dnewp,
                       const void* saved, const void* new_obj, void* dobj, int dobj_bf16, void* dX,
                       float* dparams, void* workspace, size_t workspace_bytes, const void* wbuf, const float* conf_ext,
                       csg_stream_t stream);
/* Optional hoisting of per-layer preparation out of the layer calls.  wbuf (may be NULL): the 16-bit weight copies of the
 * layer kept by the caller (csg_gconv_bf16_wbuf_bytes bytes, 256-byte aligned, filled by csg_gconv_bf16_cast_weights for up
 * to 6 layers in one launch -- once per optimizer step); NULL = the layer casts its weights itself into `saved`.  conf_ext
 * (may be NULL): the triple confidences [NT] (csg_triple_conf), computed once when all layers share w_trans as in
 * sg2im/model.py:47-55; NULL = computed by the layer.  The same pointers must be given to the backward call. */
size_t csg_gconv_bf16_wbuf_bytes(const int* dims);
int csg_gconv_bf16_cast_weights(int n, const int* dims, const void* const* params, void* const* wbufs, int need_bwd,
                                csg_stream_t stream);

/* out[i] = map[idx[i]] (int32): composes the per-triple class ids of the fused layer 0 from the triples' object indices
 * and the objects' class ids.  idx values outside [0, n_map) and (n_values > 0) map values outside [0, n_values) --
 * an embedding id nn.Embedding would raise on -- are reported through csg_async_error_poll. */
int csg_compose_index(const int* idx, const long long* map, long long map_stride, int n, int n_map, int n_values,
                      int* out, csg_stream_t stream);

/* ---- embeddings + box loss around the GCN: sg2im/model.py:108-109, sg2im/attribute_embed.py:38-48,
 *      sg2im/pix2pix_model.py:72-85 --------------------------------------------------------------- */
/* out[r, 0:E] = table[idx[r * idx_stride], :]  (rows with leading dimension ld_out; out_bf16: 0 fp32, 1 bf16, 2 fp16) */
int csg_embed_fwd(const float* table, const long long* idx, long long idx_stride, int n, int V, int E,
                  void* out, int ld_out, int out_bf16, csg_stream_t stream);
size_t csg_embed_bwd_workspace(int n, int V, int E);
/* dtable[v, :] = sum_{r: idx[r] = v} dout[r, :]  (deterministic; dout fp32 or bf16; dtable fully written) */
int csg_embed_bwd(const void* dout, int ld, int in_bf16, const long long* idx, long long idx_stride, int n,
                  int V, int E, float* dtable, void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* out[r, :] = one-hot(idx[r]) as bf16 rows of pitch ld (>= V, multiple of 8): operand of the tensor-core form of the
 * table gradient, dtable = onehot^T dout through csg_gemm_bf16(mn_major = 1). */
int csg_onehot_bf16(const long long* idx, long long idx_stride, int n, int V, void* out, int ld, csg_stream_t stream);
/* Geometric ("location") triplets (sg2im/data/base_dataset.py:35-87): for every ordered pair of real objects (class id
 * != image_id, graphs with a single object have none) the box predicates below / above / left of / right of / inside /
 * surrounding, each relation reduced to its minimal graph when it has >= 3 edges (graphs_utils.py:64-71), emitted
 * relation by relation in row-major order.  pred_ids: HOST array of the six predicate ids in that order.  Two passes
 * around csg_canon_offsets (pass a zero array as its cnt1): csg_location_count fills cnt[B], csg_location_emit writes
 * the [T, 3] int64 (s, p, o) rows (graph-local ids) at out_off[g].  max_objs >= the largest graph. */
int csg_location_count(const float* boxes, const float* centers, const long long* objs, long long objs_stride,
                       const int* obj_off, int B, long long image_id, const int* pred_ids, int max_objs, int* cnt,
                       csg_stream_t stream);
int csg_location_emit(const float* boxes, const float* centers, const long long* objs, long long objs_stride,
                      const int* obj_off, int B, long long image_id, const int* pred_ids, int max_objs,
                      const int* out_off, long long* out_triplets, csg_stream_t stream);

/* add_dummy_triplets (sg2im/data/base_dataset.py:141-150) on a flat batch: [i, __in_image__, image] for every object
 * i != image of a graph that holds an __image__ object, in ascending i.  count: cnt[g] = n_g - 1 (or 0); pass it as
 * cnt1 of csg_canon_offsets next to csg_location_count's cnt0, so that every graph's output range holds its location
 * triplets followed by its dummy triplets; emit: rows written at out_off[g] + skip[g] (skip = the location counts). */
int csg_dummy_triplets_count(const long long* objs, long long objs_stride, const int* obj_off, int B,
                             long long image_id, int* cnt, csg_stream_t stream);
int csg_dummy_triplets_emit(const long long* objs, long long objs_stride, const int* obj_off, int B,
                            long long image_id, int in_image_pred, const int* out_off, const int* skip,
                            long long* out_triplets, csg_stream_t stream);

/* Narrow output head (box_net's Linear(H, 4), model.py:58-60) of the bf16 engine: y = h w^T + b forward; backward
 * writes dh = (h > 0) * (dy w) as bf16 (the first layer's ReLU folded in), dw = dy^T h and db = colsum(dy) in fp32,
 * deterministically.  h / dh bf16 with pitches ldh / lddh, nout <= 8. */
int csg_head_fwd(const void* h, int ldh, const float* w, const float* b, int M, int K, int nout, float* y,
                 int h_fp16, csg_stream_t stream);
size_t csg_head_bwd_workspace(int M, int K, int nout);
int csg_head_bwd(const float* dy, const void* h, int ldh, const float* w, int M, int K, int nout, void* dh, int lddh,
                 float* dw, float* db, int h_fp16, void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* The same head for any element format of h / dh (fmt: 0 fp32, 1 bf16, 2 fp16) and with an optional sigmoid: the 1x1
 * output convolution of the mask head (model.py:62-75).  sigmoid = 1: y = sigmoid(h w^T + b); the backward then takes
 * those outputs as y (NULL: no sigmoid) and folds sigmoid' = y (1 - y) into dy.  relu = 1: h is a ReLU output and dh
 * takes its mask (h > 0); relu = 0: dh = dy w.  Reductions as above, in two ordered levels for many rows. */
int csg_head_fwd_ex(const void* h, int ldh, int h_fmt, const float* w, const float* b, int M, int K, int nout,
                    int sigmoid, float* y, csg_stream_t stream);
size_t csg_head_bwd_ex_workspace(int M, int K, int nout);
int csg_head_bwd_ex(const float* dy, const float* y, const void* h, int ldh, int h_fmt, const float* w, int M, int K,
                    int nout, void* dh, int lddh, int dh_fmt, int relu, float* dw, float* db, void* workspace,
                    size_t workspace_bytes, csg_stream_t stream);

/* ---- mask head of Sg2LayoutModel (sg2im/model.py:62-75, mask_size > 0): per stage Upsample(2) -> BatchNorm2d(C) ->
 *      Conv2d(C, C, 3, padding=1) -> ReLU, each convolution one GEMM (csg_gemm_bf16 / csg_gemm_f32) over a patch matrix.
 *      A stage input of side s is x [O*s*s, C] (NHWC rows, row (o*s + y)*s + x); fmt: 0 fp32, 1 bf16, 2 fp16.  BatchNorm
 *      runs at low resolution (nearest upsampling leaves the batch mean and biased variance unchanged). -------------- */
/* n = O*s*s rows.  training: batch statistics (deterministic), running_mean / running_var (may be NULL) updated with
 * `momentum` and the unbiased variance of the 4n upsampled elements, *num_batches_tracked += 1 (also for n = 0, which
 * leaves the running buffers unchanged).  eval: the running buffers.  Writes mean, invstd and scale = gamma * invstd
 * [C] (nothing for n = 0). */
size_t csg_mask_bn_fwd_workspace(int n, int C);
int csg_mask_bn_fwd(const void* x, int x_fmt, int n, int C, const float* gamma, float* running_mean, float* running_var,
                    long long* num_batches_tracked, double momentum, double eps, int training, float* scale, float* mean,
                    float* invstd, void* workspace, size_t workspace_bytes, csg_stream_t stream);
/* A [O*(2s)^2, 9C] (16-byte aligned) = patches of the upsampled, normalised, zero-padded input:
 * A[(o*S + Y)*S + X, c*9 + ky*3 + kx] = (x[o, (Y+ky-1)/2, (X+kx-1)/2, c] - mean[c]) * scale[c] + beta[c] inside the
 * S x S image (S = 2s), 0 outside.  conv.weight.view(C, 9C) is the matching GEMM operand.  C % 8 == 0. */
int csg_mask_patch(const void* x, int x_fmt, int O, int s, int C, const float* mean, const float* scale,
                   const float* beta, void* A, int a_fmt, csg_stream_t stream);
/* Backward of csg_mask_patch and of the BatchNorm in front of it: dA [O*(2s)^2, 9C] -> dx [O*s*s, C] (times (x > 0)
 * when relu_mask: x is then the previous stage's ReLU output), dgamma, dbeta [C].  mean / invstd from csg_mask_bn_fwd;
 * training selects the batch-statistics backward.  Deterministic. */
size_t csg_mask_bn_bwd_workspace(int n, int C);
int csg_mask_bn_bwd(const void* dA, int da_fmt, const void* x, int x_fmt, int O, int s, int C, const float* gamma,
                    const float* mean, const float* invstd, int training, int relu_mask, void* dx, int dx_fmt,
                    float* dgamma, float* dbeta, void* workspace, size_t workspace_bytes, csg_stream_t stream);

/* Multi-tensor Adam (torch.optim.Adam arithmetic, amsgrad off): updates `count` fp32 tensors in place in
 * ceil(count / 48) launches.  params / grads / exp_avg / exp_avg_sq / numel are HOST arrays (device pointers, element
 * counts); steps[i] >= 1 (HOST) is tensor i's own update index used for its bias corrections (torch.optim.Adam keeps
 * one step count per parameter).  The reference's training loop (scripts/train.py) calls torch.optim.Adam.step()
 * at this point. */
int csg_adam_multi(int count, void* const* params, const void* const* grads, void* const* exp_avg,
                   void* const* exp_avg_sq, const int* numel, double lr, double beta1, double beta2, double eps,
                   double weight_decay, const int* steps, csg_stream_t stream);

/* Box term of the generator loss, sg2im/pix2pix_model.py:72-85, on a flat batch: loss_all[b] ("bbox_pred_all") =
 * weight * sum over the real objects of image b of smooth_l1(pred - gt) / n_real(b); loss[0] ("bbox_pred") = mean_b;
 * dpred [NO, 4] = d loss[0] / d pred.  objs [NO, A] int64: a row is real iff its id (A == 1) / the sum of its ids
 * (A > 1) is non-zero.  An image without real objects yields NaN, as the reference's 0 / 0. */
int csg_box_loss(const float* pred, const float* gt, const long long* objs, int A, const int* obj_off, int B,
                 double weight, float* loss, float* loss_all, float* dpred, csg_stream_t stream);
/* Mask term of the generator loss (sg2im's compute_generator_loss): loss[0] = weight * F.binary_cross_entropy(pred,
 * target), the mean over all n elements, and dpred [n] = d loss[0] / d pred, in one pass.  pred fp32 [n]; target [n]
 * fp32 (target_fmt 0; soft targets in [0, 1]) or int64 (target_fmt 1).  torch's arithmetic: per element
 * -(t max(log p, -100) + (1 - t) max(log(1 - p), -100)), d/dp = weight (p - t) / max((1 - p) p, 1e-12) / n; a NaN in
 * pred gives a NaN loss and a NaN in its own dpred element; pred outside [0, 1] is not checked.  n == 0: loss[0] = NaN,
 * nothing is read.  Deterministic (block partials + one ordered final pass), no host synchronisation. */
size_t csg_mask_loss_workspace(long long n);
int csg_mask_loss(const float* pred, const void* target, int target_fmt, long long n, double weight, float* loss,
                  float* dpred, void* workspace, size_t workspace_bytes, csg_stream_t stream);

/* ---- canonicalization: sg2im/data/base_dataset.py:89-139, scripts/graphs_utils.py:15-155 ------ */
/* pass 1: per-graph output sizes (cnt0 = type-0 edges, cnt1 = transitive edges; cnt0 = -1 flags a
 * graph with more than max_objs_per_graph objects) and conv_counts [B, P, P+1] */
int csg_canon_count(const long long* triplets, const int* tri_off, const int* obj_off, int B,
                    const double* uniforms, const double* cdf, const int* vals, int ncand,
                    int P, int meta0, int meta1, int learned_converse, int learned_transitivity,
                    int max_objs_per_graph, int* cnt0, int* cnt1, int* conv_counts, csg_stream_t stream);
/* between the passes: out_off[B+1] = exclusive scan of cnt0 + cnt1; summary[0] = total rows, summary[1] = min(cnt0)
 * (the one host read of a canonicalization: it sizes the output allocation) */
int csg_canon_offsets(const int* cnt0, const int* cnt1, int B, int* out_off, int* summary, csg_stream_t stream);
/* pass 2: emit [s, p, o] int64 rows + edge types at out_off[g] (exclusive scan of cnt0 + cnt1) */
int csg_canon_emit(const long long* triplets, const int* tri_off, const int* obj_off, int B,
                   const double* uniforms, const double* cdf, const int* vals, int ncand,
                   int P, int meta0, int meta1, int learned_converse, int learned_transitivity,
                   int max_objs_per_graph, const int* out_off, long long* out_triplets, long long* out_type,
                   csg_stream_t stream);
/* graphs_utils.py:15-27 (reduce = 0) / :41-44 (reduce = 1) on G adjacency matrices [G, n, n] uint8 */
int csg_canon_closure(const unsigned char* adj, int G, int n, int reduce, unsigned char* out,
                      csg_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CSG2IM_H_ */
