"""Tensor-core (bf16 operands, fp32 accumulation) engine of the triple graph convolution.

Same dataflow as ``graph._TripleConvF32`` with every GEMM on tcgen05 (csrc/gemm_tc.cu), one native call per layer
and direction (csrc/gconv_engine.cu):

    forward   F1 (gather fused into A)  ->  F2 (+bias, ReLU, x confidence)  ->  CSR pooling  ->  net2
    backward  dW-type GEMMs are MN-major split-K GEMMs over the triples (dW1 re-gathers its B operand),
              dX-type GEMMs use per-call transposed bf16 copies of the weights so both operands are K-major;
              all final passes of a layer's ordered reductions (split-K, bias column sums, d w_trans) run in one launch

Activations between layers stay bf16; weight gradients, pooling sums and confidences are fp32.
Tolerance vs the fp32 reference: 1e-2 relative (north_star).
"""
import ctypes
import os

import torch

from . import _lib
from . import ops
from .ops import lib, ptr, f32c, workspace, _stream, Gather

BF = torch.bfloat16
F16 = torch.float16
INFERENCE_ONLY = ("precision='fp16' keeps the forward tensors in fp16 (11 significant bits instead of bf16's 8, same "
                  "tensor-core rate) and is inference-only: gradients need bf16's range and tcgen05.mma cannot mix an "
                  "fp16 operand with a bf16 one (scratch/probe_mixed_mma.py); run under torch.no_grad() or use 'bf16'")


def _fmt(dtype):
    """csg_embed_fwd's output selector: 0 fp32, 1 bf16, 2 fp16."""
    return {torch.float32: 0, BF: 1, F16: 2}[dtype]


def cast_bf16(w, transpose=False):
    """fp32 [rows, cols] -> bf16 copy (optionally transposed) in one kernel."""
    w = f32c(w)
    rows, cols = w.shape
    out = torch.empty((cols, rows) if transpose else (rows, cols), dtype=BF, device=w.device)
    _lib.check(lib().csg_cast_bf16(ptr(w), rows, cols, w.stride(0), ptr(out), out.stride(0), int(transpose), 0, _stream()),
               "csg_cast_bf16")
    return out


def cast_bf16_multi(jobs, dtype=BF, outs=None):
    """jobs: list of (fp32 matrix, transpose) -> list of bf16 (or fp16) copies, one launch.  ``outs``: cast into these
    tensors (contiguous, of the copies' shapes and ``dtype``) instead of new ones."""
    import ctypes
    srcs = [f32c(w) for w, _ in jobs]
    shapes = [(w.shape[1], w.shape[0]) if tr else tuple(w.shape) for w, (_, tr) in zip(srcs, jobs)]
    if outs is None:
        outs = [torch.empty(shp, dtype=dtype, device=w.device) for w, shp in zip(srcs, shapes)]
    elif any(tuple(o.shape) != tuple(shp) or o.dtype != dtype or not o.is_contiguous() for o, shp in zip(outs, shapes)):
        raise ValueError("cast_bf16_multi: outs do not match the copies' shapes / dtype")
    n = len(jobs)
    VP, IA = ctypes.c_void_p * n, ctypes.c_int * n
    rc = lib().csg_cast_bf16_multi(n, VP(*[w.data_ptr() for w in srcs]), VP(*[o.data_ptr() for o in outs]),
                                   IA(*[w.shape[0] for w in srcs]), IA(*[w.shape[1] for w in srcs]),
                                   IA(*[int(tr) for _, tr in jobs]), int(dtype == F16), _stream())
    _lib.check(rc, "csg_cast_bf16_multi")
    return outs


def as_bf16_rows(x, dtype=BF):
    """16-bit (bf16, or fp16 for the inference-only precision) 2-D tensor with unit inner stride and 16-byte aligned
    rows (views are kept)."""
    if x.dtype != dtype:
        if x.dtype == torch.float32 and x.is_contiguous() and dtype == BF:
            return cast_bf16(x)
        x = x.to(dtype)
    if x.stride(-1) != 1 or x.stride(0) % 8 != 0 or x.data_ptr() % 16 != 0:
        x = x.contiguous()
    return x


def segpool_bf16(X, col_s, col_o, W, batch, conf=None, avg=True, want_f32=True, want_bf16=True):
    dev = X.device
    out32 = torch.empty((batch.NO, W), dtype=torch.float32, device=dev) if want_f32 else None
    out16 = torch.empty((batch.NO, W), dtype=BF, device=dev) if want_bf16 else None
    cnt = torch.empty(batch.NO, dtype=torch.float32, device=dev) if avg else None
    rc = lib().csg_segpool_bf16(ptr(X), X.stride(0), col_s, col_o, W, ptr(batch.rowptr_s), ptr(batch.perm_s),
                                ptr(batch.rowptr_o), ptr(batch.perm_o), ptr(batch.valid) if avg else 0,
                                ptr(conf) if avg else 0, batch.NO, ptr(out32), ptr(out16), W, ptr(cnt), int(avg), 0, _stream())
    _lib.check(rc, "csg_segpool_bf16")
    return out32, out16, cnt


def colsum_bf16(X):
    M, N = X.shape
    out = torch.empty(N, dtype=torch.float32, device=X.device)
    L = lib()
    ws = workspace(L.csg_colsum_bf16_workspace(M, N), X.device)
    _lib.check(L.csg_colsum_bf16(ptr(X), M, N, X.stride(0), ptr(out), ptr(ws), ws.numel(), _stream()), "csg_colsum_bf16")
    return out


def relu_mask_bf16(dy, y):
    dy = f32c(dy)
    out = torch.empty(y.shape, dtype=BF, device=y.device)
    _lib.check(lib().csg_relu_mask_bf16(ptr(dy), ptr(y), ptr(out), y.numel(), _stream()), "csg_relu_mask_bf16")
    return out


# --------------------------------------------------------------------------------------------
# native layer executor (csrc/gconv_engine.cu): the launch sequence of a layer issued by ONE call per direction
# --------------------------------------------------------------------------------------------
_WS = {}      # device -> reusable scratch (dead once the call has returned on the stream)


def _scratch(nbytes, dev):
    buf = _WS.get(dev)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=dev)
        _WS[dev] = buf
    return buf


def _ptr_array(tensors):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


# --------------------------------------------------------------------------------------------
# caller-kept 16-bit weight copies: one cast launch for all layers per optimizer step instead of one per layer and
# forward (csg_gconv_bf16_cast_weights).  An entry is valid while the fp32 weights it was cast from are unchanged:
# autograd's version counters catch every in-place torch update (torch.optim, load_state_dict, init), and FusedAdam,
# which writes the parameters through raw pointers, invalidates the entries of its parameters itself (optim.py).
# --------------------------------------------------------------------------------------------
_WCOPIES = {}      # data_ptr of net1.0.weight -> dict(wbuf, versions, key, params)


def _wkey(params, act, dims):
    return (tuple(int(x) for x in list(dims)[2:9]), act, tuple(p.data_ptr() for p in params[:8]))


def invalidate_weight_copies(params=None):
    """Mark the cached weight copies stale (of the layers that own any of ``params``; all when None).  The buffers stay
    where they are -- a captured CUDA graph may hold their addresses -- and are refilled by refresh_weight_copies."""
    ptrs = None if params is None else {p.data_ptr() for p in params}
    for e in _WCOPIES.values():
        if ptrs is None or ptrs & {q.data_ptr() for q in e["params"]}:
            e["versions"] = None
    from . import mask_head       # the mask head's 3x3 convolution weights are cached on the same terms
    mask_head.invalidate_weight_copies(params)


def refresh_weight_copies(layers, act=BF):
    """Cast the weights of ``layers`` (``GraphTripleConv`` modules on the tensor-core engine) into their cached 16-bit
    copies, six layers per launch.  Call after every optimizer step; a layer without a valid copy casts its weights
    itself inside its forward call, so forgetting to call this costs time, never correctness."""
    L = lib()
    todo = []
    for layer in layers:
        params = tuple(layer.layer_params()) + (layer.predicates_transitive_weights,)
        if any(p.dtype != torch.float32 or not p.is_contiguous() or not p.is_cuda for p in params):
            continue
        din, dp = layer.obj_input_dim, layer.predicate_input_dim
        H, Dout, Dpo = layer.hidden_dim, params[6].shape[0], layer.predicate_output_dim
        if din % 64 or dp % 64 or H % 64 or Dout % 64 or Dpo % 64:
            continue                    # zero-padded on the fly (triple_conv): those layers cast per call
        dims = (ctypes.c_int * 11)(0, 0, din, dp, H, Dout, Dpo, max(params[8].numel(), 1), int(act == F16), 0, 0)
        todo.append((params, dims))
    for i in range(0, len(todo), 6):
        grp = todo[i:i + 6]
        ents = []
        for params, dims in grp:
            key, k = params[0].data_ptr(), _wkey(params, act, dims)
            e = _WCOPIES.get(key)
            if e is None or e["key"] != k:
                nb = L.csg_gconv_bf16_wbuf_bytes(dims)
                e = _WCOPIES[key] = {"wbuf": torch.empty(nb, dtype=torch.uint8, device=params[0].device), "key": k,
                                     "params": params[:8]}
            ents.append(e)
        n = len(grp)
        dims_flat = (ctypes.c_int * (11 * n))(*[x for _, d in grp for x in list(d)])
        pp = (ctypes.c_void_p * (9 * n))(*[p.data_ptr() for params, _ in grp for p in params])
        wb = (ctypes.c_void_p * n)(*[e["wbuf"].data_ptr() for e in ents])
        _lib.check(L.csg_gconv_bf16_cast_weights(n, dims_flat, pp, wb, 1, _stream()), "csg_gconv_bf16_cast_weights")
        for e, (params, _) in zip(ents, grp):
            e["versions"] = tuple(p._version for p in params[:8])


def _cached_wbuf(params, act, dims):
    e = _WCOPIES.get(params[0].data_ptr())
    if e is None or e["key"] != _wkey(params, act, dims) or e.get("versions") != tuple(p._version for p in params[:8]):
        return None
    return e["wbuf"]


class FusedTables:
    """Layer 0 reading straight from the embedding tables (sg2im/model.py:108-109 fused into the net1 producer): the
    layer's `obj` / `pred` arguments are then the fp32 TABLES, gathered per triple by class id / predicate id."""

    def __init__(self, batch, obj_ids, pred_ids, act):
        # obj_ids [NO] int64 (any stride): class id of every object; per-triple class ids = obj_ids[s_idx], obj_ids[o_idx]
        # pred_ids [NT] int64 (any stride): predicate id of every triple (the int32 copy batch.pred feeds the gather)
        self.obj_ids, self.pred_ids, self.act = obj_ids, pred_ids, act
        self.batch = batch

    def indices(self, n_classes):
        """(subject class ids, object class ids) [NT] int32, composed once per batch and table size."""
        cache = getattr(self.batch, "_class_idx", None)
        if cache is None or cache[0] != (self.obj_ids.data_ptr(), n_classes):
            b, L = self.batch, lib()
            out = torch.empty((2, max(b.NT, 1)), dtype=torch.int32, device=b.s_idx.device)
            for k, idx in enumerate((b.s_idx, b.o_idx)):
                _lib.check(L.csg_compose_index(ptr(idx), ptr(self.obj_ids), self.obj_ids.stride(0), b.NT, b.NO, n_classes,
                                               ptr(out[k]), _stream()), "csg_compose_index")
            cache = self.batch._class_idx = ((self.obj_ids.data_ptr(), n_classes), out, self.obj_ids)
        return cache[1][0], cache[1][1]


class _TripleConvEngine(torch.autograd.Function):
    """One GraphTripleConv layer through csg_gconv_bf16_fwd / csg_gconv_bf16_bwd."""

    @staticmethod
    def forward(ctx, grad_on, batch, H, Dpo, obj, pred, w1, b1, w2, b2, w3, b3, w4, b4, w_trans, fused=None):
        # grad_on: torch.is_grad_enabled() at call time (inside forward() autograd has it switched off)
        L = lib()
        dev = obj.device
        ctx.in_dtypes = (obj.dtype, pred.dtype)
        ctx.fused = fused
        act = fused.act if fused is not None else (F16 if obj.dtype == F16 else BF)   # fp16: inference-only format
        need_bwd = int(grad_on and any(ctx.needs_input_grad))
        if act == F16 and need_bwd:
            raise _lib.CsgError(INFERENCE_ONLY)
        n_gather = n_pred = 0
        if fused is not None:
            # obj [V, Din] / pred [P, Dp]: the fp32 embedding tables, cast once per step (a few hundred rows)
            obj_b, pred_b = cast_bf16_multi([(obj.detach(), False), (pred.detach(), False)], act)
            n_gather, n_pred = obj_b.shape[0], pred_b.shape[0]
            gs, go = fused.indices(n_gather)
        else:
            obj_b, pred_b = as_bf16_rows(obj, act), as_bf16_rows(pred, act)
            if not obj_b.is_contiguous():
                obj_b = obj_b.contiguous()
        params = [f32c(p.detach()) for p in (w1, b1, w2, b2, w3, b3, w4, b4, w_trans)]
        Dout, P = w4.shape[0], w_trans.numel()
        dims = (ctypes.c_int * 11)(batch.NT, batch.NO, obj_b.shape[1], pred_b.shape[1], H, Dout, Dpo, P, int(act == F16),
                                   n_gather, n_pred)
        nsaved = L.csg_gconv_bf16_saved_bytes(dims, need_bwd)
        saved = torch.empty(nsaved, dtype=torch.uint8, device=dev)
        # hoisted preparation (both optional): weight copies kept across calls, confidences shared by the layers of a model
        wbuf = _cached_wbuf(params, act, dims) if os.environ.get("CSG_WCOPIES", "1") != "0" else None
        shared = getattr(batch, "_conf_shared", None)
        conf_ext = shared[1] if shared is not None and shared[0] == (w_trans.data_ptr(), w_trans._version) else None
        ctx.wbuf, ctx.conf_ext = wbuf, conf_ext
        new_obj = torch.empty((batch.NO, Dout), dtype=act, device=dev)
        index = batch.index_array()
        if fused is not None:
            index = (ctypes.c_void_p * 12)(*(list(index) + [gs.data_ptr(), go.data_ptr(), batch.pred.data_ptr()]))
            ctx.gather_idx = (gs, go)
        ctx.index = index
        rc = L.csg_gconv_bf16_fwd(dims, ptr(obj_b), ptr(pred_b), pred_b.stride(0), _ptr_array(params), index, need_bwd,
                                  ptr(saved), nsaved, ptr(new_obj), ptr(wbuf), ptr(conf_ext), _stream())
        _lib.check(rc, "csg_gconv_bf16_fwd")
        Wd = 2 * H + Dpo
        off = L.csg_gconv_bf16_out_offset(dims, need_bwd)
        out = saved[off:off + batch.NT * Wd * 2].view(act).view(batch.NT, Wd)
        new_p = out[:, H:H + Dpo]
        ctx.batch, ctx.dims, ctx.params = batch, dims, params
        ctx.save_for_backward(obj_b, pred_b, saved, new_obj)
        ctx.set_materialize_grads(False)
        return new_obj, new_p

    @staticmethod
    def backward(ctx, d_obj_out, d_newp):
        obj, pred, saved, new_obj = ctx.saved_tensors
        batch, dims, params = ctx.batch, ctx.dims, ctx.params
        NT, NO, Din, Dp, H, Dout, Dpo, P = list(dims)[:8]
        fused = ctx.fused
        K1, Wd = 2 * Din + Dp, 2 * H + Dpo
        dev = obj.device
        L = lib()
        if d_obj_out is not None:
            if d_obj_out.dtype not in (torch.float32, BF):
                d_obj_out = d_obj_out.float()
            d_obj_out = d_obj_out.contiguous()
        if d_newp is not None and not (d_newp.dtype == BF and d_newp.stride(-1) == 1 and d_newp.stride(0) % 8 == 0
                                       and d_newp.data_ptr() % 16 == 0):
            d_newp = d_newp.to(BF).contiguous()
        obj_bf16 = ctx.in_dtypes[0] == BF and fused is None
        dobj = torch.empty((NO, Din), dtype=BF if obj_bf16 else torch.float32, device=dev)
        dxc = L.csg_gconv_bf16_dx_cols(dims)          # Dp (d pred only), or K1 on the gathered dataflow
        dX = torch.empty((NT, dxc), dtype=BF, device=dev)
        sizes = (H * K1, H, Wd * H, Wd, H * H, H, Dout * H, Dout, P)
        dparams = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
        nws = L.csg_gconv_bf16_workspace(dims)
        ws = _scratch(nws, dev)
        rc = L.csg_gconv_bf16_bwd(dims, ptr(obj), ptr(pred), pred.stride(0), _ptr_array(params), ctx.index,
                                  ptr(d_obj_out), int(d_obj_out is not None and d_obj_out.dtype == BF),
                                  ptr(d_newp), d_newp.stride(0) if d_newp is not None else 0,
                                  ptr(saved), ptr(new_obj), ptr(dobj), int(obj_bf16), ptr(dX), ptr(dparams),
                                  ptr(ws), ws.numel(), ptr(ctx.wbuf), ptr(ctx.conf_ext), _stream())
        _lib.check(rc, "csg_gconv_bf16_bwd")
        dw1, db1, dw2, db2, dw3, db3, dw4, db4, dwt = torch.split(dparams, sizes)
        dpred = dX[:, Din:Din + Dp] if dxc == K1 else dX
        if fused is not None:
            # the gradients of the gathered rows folded back onto the embedding tables (attribute_embed.py:38-48,
            # model.py:109): per-object rows by class id, per-triple predicate rows by predicate id (one-hot GEMM)
            dobj = ops.embed_table_grad(dobj, fused.obj_ids, obj.shape[0], Din)
            dpred = ops.embed_table_grad(dpred, fused.pred_ids, pred.shape[0], Dp)
        else:
            if not obj_bf16 and ctx.in_dtypes[0] != torch.float32:
                dobj = dobj.to(ctx.in_dtypes[0])
            if ctx.in_dtypes[1] != BF:
                dpred = dpred.to(ctx.in_dtypes[1])
        return (None, None, None, None, dobj, dpred, dw1.view(H, K1), db1, dw2.view(Wd, H), db2, dw3.view(H, H), db3,
                dw4.view(Dout, H), db4, dwt, None)


def triple_conv_tables(batch, obj_table, obj_ids, pred_table, pred_ids, params, w_trans, hidden_dim, pred_out_dim,
                       act=BF):
    """Layer 0 of ``Sg2LayoutModel`` with the embedding lookups (model.py:108-109) fused into the net1 producer: the
    object rows are gathered from ``obj_table [V, Din]`` by the class ids ``obj_ids [NO]`` of the triples' subjects /
    objects, the predicate rows from ``pred_table [P, Dp]`` by the triples' predicate ids (``batch.pred``) -- no
    ``[NO, Din]`` / ``[NT, Dp]`` rows are materialised; the table gradients come back through the same node.
    Needs Din, Dp multiples of 64 (single-attribute objects: COCO / VG)."""
    return _TripleConvEngine.apply(torch.is_grad_enabled(), batch, hidden_dim, pred_out_dim, obj_table, pred_table,
                                   *params, w_trans, FusedTables(batch, obj_ids, pred_ids, act))


def triple_conv(batch, obj, pred, params, w_trans, hidden_dim, pred_out_dim):
    din, dp = obj.shape[1], pred.shape[1]
    dout = params[6].shape[0]
    if dp % 64 and not (din % 64 or hidden_dim % 64 or pred_out_dim % 64 or dout % 64):
        # predicate rows narrower than one 128-byte operand chunk (CLEVR: embedding_dim 32, model.py:109 -> layer 0
        # only): zero-pad them and the matching columns of net1.0.weight to the next multiple of 64 -- the products
        # with the zero columns vanish, and autograd slices the gradients back (two tiny torch ops on [NT, 64] /
        # [H, 2 Din + 64] outside the kernels' hot loop)
        pad = (-dp) % 64
        w1 = params[0]
        pred = torch.nn.functional.pad(pred, (0, pad))
        w1 = torch.cat([w1[:, :din + dp], w1.new_zeros((w1.shape[0], pad)), w1[:, din + dp:]], dim=1)
        params = (w1,) + tuple(params[1:])
        dp += pad
    if din % 64 or dp % 64 or hidden_dim % 64 or pred_out_dim % 64 or dout % 64:
        raise _lib.CsgError("precision='bf16' needs feature widths that are multiples of 64 "
                            "(got Din=%d Dp=%d H=%d Dout=%d Dp_out=%d); use precision='fp32'"
                            % (din, dp, hidden_dim, dout, pred_out_dim))
    return _TripleConvEngine.apply(torch.is_grad_enabled(), batch, hidden_dim, pred_out_dim, obj, pred, *params, w_trans)


class _DenseMLP2BF16(torch.autograd.Function):
    """box_net (model.py:58-60) on the bf16 engine: Linear(D, H) + ReLU on tcgen05, the 4-wide Linear(H, 4) head as a
    row-dot kernel (csrc/head_bf16.cu); the backward head kernel folds the ReLU mask and writes dh in bf16."""

    @staticmethod
    def forward(ctx, grad_on, x, w0, b0, w1, b1):
        L = lib()
        act = F16 if x.dtype == F16 else BF
        need_bwd = grad_on and any(ctx.needs_input_grad)
        if act == F16 and need_bwd:
            raise _lib.CsgError(INFERENCE_ONLY)
        xb = as_bf16_rows(x, act)
        M, (H, D), nout = xb.shape[0], w0.shape, w1.shape[0]
        casts = cast_bf16_multi([(w0, False)] + ([(w0, True)] if need_bwd else []), act)
        h = ops.gemm_bf16(M, H, D, xb, casts[0], bias=f32c(b0), relu=True, out_dtype=act)
        y = torch.empty((M, nout), dtype=torch.float32, device=xb.device)
        w1c = f32c(w1.detach())
        _lib.check(L.csg_head_fwd(ptr(h), h.stride(0), ptr(w1c), ptr(f32c(b1.detach())), M, H, nout, ptr(y), int(act == F16), _stream()),
                   "csg_head_fwd")
        ctx.save_for_backward(xb, h, w1c)
        ctx.w0t = casts[1] if need_bwd else None
        ctx.x_dtype = x.dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        xb, h, w1c = ctx.saved_tensors
        L = lib()
        M, H = h.shape
        D, nout = xb.shape[1], w1c.shape[0]
        dev = xb.device
        dy = f32c(dy)
        dh = torch.empty((M, H), dtype=BF, device=dev)
        dw1 = torch.empty((nout, H), dtype=torch.float32, device=dev)
        db1 = torch.empty(nout, dtype=torch.float32, device=dev)
        ws = workspace(L.csg_head_bwd_workspace(M, H, nout), dev)
        _lib.check(L.csg_head_bwd(ptr(dy), ptr(h), h.stride(0), ptr(w1c), M, H, nout, ptr(dh), dh.stride(0), ptr(dw1),
                                  ptr(db1), 0, ptr(ws), ws.numel(), _stream()), "csg_head_bwd")
        dw0 = ops.gemm_bf16(H, D, M, dh, xb, mn_major=True)
        db0 = colsum_bf16(dh)
        dx = ops.gemm_bf16(M, D, H, dh, ctx.w0t)
        if ctx.x_dtype != BF:
            dx = dx.to(ctx.x_dtype)
        return None, dx, dw0, db0, dw1, db1


class _LinearBF16(torch.autograd.Function):
    """y = x W^T + b on tcgen05 (bf16 operands, fp32 accumulate, bf16 output): ``attribute_fc_gen`` of the
    multi-attribute object embedding (attribute_embed.py:24-25,46-47) in front of the bf16 GCN."""

    @staticmethod
    def forward(ctx, grad_on, x, w, b):
        act = F16 if x.dtype == F16 else BF
        need_bwd = grad_on and any(ctx.needs_input_grad)
        if act == F16 and need_bwd:
            raise _lib.CsgError(INFERENCE_ONLY)
        xb = as_bf16_rows(x, act)
        casts = cast_bf16_multi([(w, False)] + ([(w, True)] if need_bwd else []), act)
        N, K = w.shape
        y = ops.gemm_bf16(xb.shape[0], N, K, xb, casts[0], bias=f32c(b), out_dtype=act)
        ctx.save_for_backward(xb)
        ctx.wt = casts[1] if need_bwd else None
        ctx.x_dtype, ctx.shape = x.dtype, (N, K)
        return y

    @staticmethod
    def backward(ctx, dy):
        (xb,) = ctx.saved_tensors
        N, K = ctx.shape
        M = xb.shape[0]
        dyb = as_bf16_rows(dy)
        dw = ops.gemm_bf16(N, K, M, dyb, xb, mn_major=True)
        db = colsum_bf16(dyb)
        dx = None
        if ctx.needs_input_grad[1]:
            dx = ops.gemm_bf16(M, K, N, dyb, ctx.wt)
            if ctx.x_dtype != BF:
                dx = dx.to(ctx.x_dtype)
        return None, dx, dw, db


def dense_mlp2(x, w0, b0, w1, b1, final_relu):
    """box_net (model.py:58-60).  Feature widths that fit the tensor-core tiles and a head of <= 8 outputs run on
    ``_DenseMLP2BF16``; anything else on the fp32 engine."""
    if (not final_relu and w1.shape[0] <= 8 and w0.shape[0] % 64 == 0 and w0.shape[1] % 64 == 0
            and w0.shape[0] * w1.shape[0] * 4 <= 48 * 1024):
        return _DenseMLP2BF16.apply(torch.is_grad_enabled(), x, w0, b0, w1, b1)
    return _dense_mlp2_f32(x, w0, b0, w1, b1, final_relu)


def _dense_mlp2_f32(x, w0, b0, w1, b1, final_relu):
    """box_net (model.py:58-60): M = #objects, output width 4 -- too small to matter; it runs on the fp32 engine."""
    from .graph import _DenseMLP2F32
    return _DenseMLP2F32.apply(x.float() if x.dtype != torch.float32 else x, w0, b0, w1, b1, final_relu)
