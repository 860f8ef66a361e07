"""Scene-graph -> layout model: drop-in for ``sg2im/model.py::Sg2LayoutModel`` (reference
``sg2im/model.py:18-124``) built on the csg2im kernels.

State-dict keys equal the reference's (``attribute_embedding.att_emb_{k}.weight``,
``pred_embeddings.weight``, ``trans_candidates_weights``, ``converse_candidates_weights``,
``gconvs.{i}.net1.{0,2}.*``, ``gconvs.{i}.net2.{0,2}.*``, ``gconvs.{i}.predicates_transitive_weights``,
``box_net.{0,2}.*``, and with ``mask_size > 0`` the mask head's ``mask_net.{1,5,9,..}.*`` BatchNorm2d,
``mask_net.{2,6,10,..}.*`` Conv2d and ``mask_net.{4k}.*`` 1x1 Conv2d), so reference checkpoints load with ``strict=True``.
The mask head (``model.py:62-75``) runs on the csg2im kernels too (``mask_head.py``): its convolutions are GEMMs on the
same engines as the GCN, with BatchNorm, upsampling and the patch gathers as memory-bound kernels around them.
"""
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .graph import GraphTripleConv, TripleBatch, build_mlp, dense_mlp2, get_predicates_weights, linear
from .ops import lib, ptr, need_cuda, workspace, _stream


class _EmbedFn(torch.autograd.Function):
    """``nn.Embedding`` lookup (attribute_embed.py:38-48, model.py:109) on csg_embed_fwd / csg_embed_bwd:
    rows are written straight in the GCN's operand type and the table gradient is a deterministic segmented sum."""

    @staticmethod
    def forward(ctx, table, idx, out_dtype):
        need_cuda(table, idx)
        if idx.dtype != torch.int64:
            idx = idx.to(torch.int64)
        if idx.dim() != 1:
            raise ValueError("embedding index must be 1-D (got %s)" % (tuple(idx.shape),))
        if idx.numel() and idx.stride(0) < 1:
            idx = idx.contiguous()
        tab = table.detach()
        if tab.dtype != torch.float32 or not tab.is_contiguous():
            tab = tab.float().contiguous()
        n, (V, E) = idx.numel(), tab.shape
        out = torch.empty((n, E), dtype=out_dtype, device=tab.device)
        rc = lib().csg_embed_fwd(ptr(tab), ptr(idx), idx.stride(0) if n else 1, n, V, E, ptr(out), E,
                                 {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}[out_dtype], _stream())
        _lib.check(rc, "csg_embed_fwd")
        ctx.save_for_backward(idx)
        ctx.dims = (n, V, E)
        return out

    @staticmethod
    def backward(ctx, dout):
        (idx,) = ctx.saved_tensors
        n, V, E = ctx.dims
        from .ops import embed_table_grad
        return embed_table_grad(dout, idx, V, E), None, None


def embedding_lookup(weight, idx, out_dtype=torch.float32):
    """``weight[idx]`` for a 1-D int64 index (any stride); ids must lie in [0, weight.shape[0])."""
    return _EmbedFn.apply(weight, idx, out_dtype)


class _BoxLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, gt, objs, obj_off, weight):
        need_cuda(pred, gt, objs, obj_off)
        p, g = pred.detach().float().contiguous(), gt.float().contiguous()
        objs = objs.to(torch.int64).contiguous()
        B, A = obj_off.numel() - 1, objs.shape[1]
        loss = torch.empty(1, dtype=torch.float32, device=p.device)
        loss_all = torch.empty(B, dtype=torch.float32, device=p.device)
        dpred = torch.empty_like(p)
        _lib.check(lib().csg_box_loss(ptr(p), ptr(g), ptr(objs), A, ptr(obj_off), B, float(weight), ptr(loss),
                                      ptr(loss_all), ptr(dpred), _stream()), "csg_box_loss")
        ctx.save_for_backward(dpred)
        ctx.mark_non_differentiable(loss_all)
        return loss[0], loss_all

    @staticmethod
    def backward(ctx, dloss, _dall):
        (dpred,) = ctx.saved_tensors
        return dpred * dloss, None, None, None, None


def bbox_pred_loss_ragged(boxes_pred, boxes_gt, objs, obj_off, weight=10.0):
    """Box term of ``Pix2PixModel.compute_generator_loss`` (sg2im/pix2pix_model.py:72-85) on a flat batch:
    per image, the smooth-L1 of the real objects (``objs != 0``; ``objs.sum(1) != 0`` for multi-attribute objects)
    summed over boxes and coordinates, times ``bbox_pred_loss_weight`` (args.py:172, default 10), divided by the
    image's real-object count.  Returns ``(G_losses["bbox_pred"], G_losses["bbox_pred_all"])`` = (mean over images,
    per-image values).  One pass, no host sync; an image without real objects gives NaN as the reference's 0/0."""
    objs = objs if objs.dim() == 2 else objs.reshape(-1, 1)
    off = obj_off if obj_off.dtype == torch.int32 else obj_off.to(torch.int32)
    return _BoxLossFn.apply(boxes_pred.reshape(-1, 4), boxes_gt.reshape(-1, 4), objs, off.contiguous(), weight)


def bbox_pred_loss(boxes_pred, boxes, objs, weight=10.0):
    """Padded form, the reference's own tensors: boxes_pred / boxes [B, O, 4], objs [B, O, A]."""
    from .graph import TripleBatch
    B, O = boxes.shape[0], boxes.shape[1]
    off = TripleBatch._uniform_off(B, O, boxes.device)
    return bbox_pred_loss_ragged(boxes_pred, boxes, objs.reshape(B * O, -1), off, weight)


class _MaskLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, weight):
        p, n = pred.detach().contiguous(), pred.numel()
        target = target.contiguous()
        loss = torch.empty(1, dtype=torch.float32, device=p.device)
        dpred = torch.empty_like(p)
        L = lib()
        ws = workspace(L.csg_mask_loss_workspace(n), p.device)
        _lib.check(L.csg_mask_loss(ptr(p), ptr(target), int(target.dtype == torch.int64), n, float(weight), ptr(loss),
                                   ptr(dpred), ptr(ws), ws.numel(), _stream()), "csg_mask_loss")
        ctx.save_for_backward(dpred)
        return loss[0]

    @staticmethod
    def backward(ctx, dloss):
        (dpred,) = ctx.saved_tensors
        return dpred * dloss, None, None


def mask_pred_loss(masks_pred, masks_gt, weight=1.0):
    """Mask term of the generator loss on GT masks (sg2im's ``compute_generator_loss``):
    ``weight * F.binary_cross_entropy(masks_pred, masks_gt.float())``, the mean over every element, with torch's clamps
    (``log`` at -100, ``(1 - p) p`` at 1e-12 in the gradient).  ``masks_pred`` / ``masks_gt``: any matching shape, e.g.
    ragged ``[NO, M, M]`` or padded ``[B, O, M, M]``; ``masks_gt`` fp32 (soft targets in [0, 1] allowed) or int64 as the
    datasets carry them, read without a cast pass; bool, other integer and float dtypes are cast to one of the two.
    Returns a differentiable scalar; the target gets no gradient.  One pass, no host synchronisation; an empty input
    gives NaN, as torch's mean of an empty tensor.  Predictions outside [0, 1] are not checked (torch raises)."""
    need_cuda(masks_pred, masks_gt)
    if tuple(masks_pred.shape) != tuple(masks_gt.shape):
        raise ValueError("mask_pred_loss: masks_pred %s and masks_gt %s differ in shape"
                         % (tuple(masks_pred.shape), tuple(masks_gt.shape)))
    tgt = masks_gt.detach()
    if tgt.dtype == torch.bool or tgt.is_floating_point():
        tgt = tgt.float()
    else:
        tgt = tgt.to(torch.int64)
    return _MaskLossFn.apply(masks_pred.float().reshape(-1), tgt.reshape(-1), weight)


def get_conv_converse(model):
    """sg2im/model.py:8-15 — symmetrised converse weights (triu + triu^T)."""
    if isinstance(model, dict):
        base = model["sg_to_layout.module.converse_candidates_weights"]
    elif hasattr(model, "sg_to_layout"):
        base = model.sg_to_layout.module.converse_candidates_weights
    else:
        base = model.converse_candidates_weights
    triu = torch.triu(base, diagonal=0)
    return triu + triu.t()


class _MultiEmbedFn(torch.autograd.Function):
    """``torch.cat([att_emb_k(x[:, k]) for k], -1)`` (attribute_embed.py:38-45) without the concat pass: every
    lookup writes its column slice of the ``[n, A*E]`` result (``csg_embed_fwd`` with ``ld_out = A*E``); the backward
    reads the slices of the incoming gradient in place."""

    @staticmethod
    def forward(ctx, idx, out_dtype, *tables):
        need_cuda(idx, *tables)
        idx = idx.to(torch.int64).contiguous()
        n, A = idx.shape
        tabs = [t.detach() if (t.dtype == torch.float32 and t.is_contiguous()) else t.detach().float().contiguous()
                for t in tables]
        widths = [t.shape[1] for t in tabs]
        W = sum(widths)
        out = torch.empty((n, W), dtype=out_dtype, device=idx.device)
        esz, col = out.element_size(), 0
        for k, tab in enumerate(tabs):
            V, E = tab.shape
            rc = lib().csg_embed_fwd(ptr(tab), idx.data_ptr() + 8 * k, A, n, V, E, out.data_ptr() + col * esz, W,
                                     {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}[out_dtype], _stream())
            _lib.check(rc, "csg_embed_fwd")
            col += E
        ctx.save_for_backward(idx)
        ctx.shapes = [tuple(t.shape) for t in tabs]
        return out

    @staticmethod
    def backward(ctx, dout):
        (idx,) = ctx.saved_tensors
        n, A = idx.shape
        if dout.dtype not in (torch.float32, torch.bfloat16):
            dout = dout.float()
        if dout.stride(-1) != 1 or dout.stride(0) % 4 != 0 or dout.data_ptr() % 16 != 0:
            dout = dout.contiguous()
        L = lib()
        esz, col, grads = dout.element_size(), 0, []
        for k, (V, E) in enumerate(ctx.shapes):
            dtable = torch.empty((V, E), dtype=torch.float32, device=dout.device)
            ws = workspace(L.csg_embed_bwd_workspace(n, V, E), dout.device)
            rc = L.csg_embed_bwd(dout.data_ptr() + col * esz, dout.stride(0) if n else E,
                                 int(dout.dtype == torch.bfloat16), idx.data_ptr() + 8 * k, A, n, V, E, ptr(dtable),
                                 ptr(ws), ws.numel(), _stream())
            _lib.check(rc, "csg_embed_bwd")
            grads.append(dtable)
            col += E
        return (None, None) + tuple(grads)


class AttributeEmbeddings(nn.Module):
    """sg2im/attribute_embed.py:18-48: one lookup table per attribute, the rows concatenated and (for more than
    one attribute, or ``use_attr_fc_gen``) mixed by ``attribute_fc_gen``.  Lookups are ``csg_embed_fwd``, the
    Linear runs on the csg2im GEMMs (``graph.linear``); parameter names equal the reference's."""

    def __init__(self, attributes, embedding_dim, use_attr_fc_gen=False, precision="fp32"):
        super().__init__()
        num_attr = len(attributes)
        if num_attr > 1 or use_attr_fc_gen:
            # parameter container only (weight / bias under the reference's names); never called as a module
            self.attribute_fc_gen = nn.Linear(num_attr * embedding_dim, num_attr * embedding_dim)
        for i, name in enumerate(list(attributes)):
            self.add_module("att_emb_%d" % i, nn.Embedding(max(attributes[name].values()) + 1, embedding_dim))
        self.num_attr = num_attr
        self.precision = precision

    def forward(self, x, out_dtype=torch.float32):
        lead = x.shape[:-1]
        flat = x.reshape(-1, x.size(-1))
        fc = getattr(self, "attribute_fc_gen", None)
        if fc is None and flat.size(-1) == 1:
            # single attribute (COCO / VG): the rows go straight out in the GCN's operand type
            v = embedding_lookup(self._modules["att_emb_0"].weight, flat[:, 0], out_dtype)
            return v.view(*lead, -1)
        tables = [self._modules["att_emb_%d" % k].weight for k in range(flat.size(-1))]
        if fc is None:
            return _MultiEmbedFn.apply(flat, out_dtype, *tables).view(*lead, -1)
        tc = out_dtype in (torch.bfloat16, torch.float16) and fc.weight.shape[0] % 64 == 0
        v = _MultiEmbedFn.apply(flat, out_dtype if tc else torch.float32, *tables)
        v = linear(v, fc.weight, fc.bias, "bf16" if tc else "fp32")
        if v.dtype != out_dtype:
            v = v.to(out_dtype)
        return v.view(*lead, -1)


class Sg2LayoutModel(nn.Module):
    def __init__(self, opt, precision="fp32"):
        super().__init__()
        args = vars(opt) if not isinstance(opt, dict) else dict(opt)
        self.args = args
        self.vocab = args["vocab"]
        self.precision = precision
        # True (or CSG_FUSE_EMB=1): layer 0 gathers its rows straight from the embedding tables inside the net1 producer.
        # Default off: with materialised rows layer 0 differentiates net1's first Linear through per-object sums of
        # dhidden like every other layer (csrc/gconv_engine.cu), which is 0.15 ms per cfg2 step faster (4.55 vs 4.71 ms)
        self.fuse_embeddings = os.environ.get("CSG_FUSE_EMB", "0") != "0"
        emb = args["embedding_dim"]
        self.attribute_embedding = AttributeEmbeddings(self.vocab["attributes"], emb)
        num_preds = self.num_preds = len(self.vocab["pred_idx_to_name"])
        self.pred_embeddings = nn.Embedding(num_preds, emb)
        num_attributes = len(self.vocab["attributes"].keys())
        init = args.get("learned_init", "uniform")
        self.trans_candidates_weights = get_predicates_weights(num_preds, init)
        self.converse_candidates_weights = get_predicates_weights((num_preds, num_preds), init)
        gdim, hdim = args["gconv_dim"], args["gconv_hidden_dim"]
        self.gconvs = nn.ModuleList()
        d_obj, d_pred = num_attributes * emb, emb
        for _ in range(args["gconv_num_layers"]):
            self.gconvs.append(GraphTripleConv(d_obj, gdim, d_pred, gdim, hdim, num_attributes,
                                               pooling=args.get("gconv_pooling", "avg"),
                                               mlp_normalization=args.get("mlp_normalization", "none"),
                                               predicates_transitive_weights=self.trans_candidates_weights,
                                               precision=precision))
            d_obj, d_pred = gdim, gdim
        self.box_net = build_mlp([gdim, hdim, 4], final_nonlinearity=None)      # model.py:58-60
        self.mask_net = None
        mask_size = args.get("mask_size") or 0
        if mask_size > 0:
            from .mask_head import build_mask_net
            self.mask_net = build_mask_net(gdim, mask_size)       # model.py:62-75
        self.padding_id = self.vocab["pred_name_to_idx"]["__padding__"]

    def _act_dtype(self):
        return {"bf16": torch.bfloat16, "fp16": torch.float16}.get(self.precision, torch.float32)

    def _fusable(self, objs_flat):
        """Layer 0 can gather its rows straight from the embedding tables (model.py:108-109 fused into the net1
        producer, csrc/gemm_tc.cu) on the tensor-core engine for single-attribute objects (COCO / VG)."""
        emb = self.pred_embeddings.weight.shape[1]
        return (self.precision in ("bf16", "fp16") and objs_flat.shape[1] == 1 and emb % 64 == 0
                and not hasattr(self.attribute_embedding, "attribute_fc_gen") and self.fuse_embeddings)

    def _embed_and_run(self, batch, objs_flat, pred_ids):
        """objs_flat [NO, A] int64, pred_ids [NT] int64 (any stride) -> (obj_vecs [NO, D], boxes [NO, 4])."""
        if self._fusable(objs_flat):
            from . import graph_tc
            l0 = self.gconvs[0]
            obj_vecs, pred_vecs = graph_tc.triple_conv_tables(
                batch, self.attribute_embedding.att_emb_0.weight, objs_flat[:, 0], self.pred_embeddings.weight, pred_ids,
                l0.layer_params(), l0.predicates_transitive_weights, l0.hidden_dim, l0.predicate_output_dim,
                self._act_dtype())
            if not l0.return_new_p_vecs:
                raise ValueError("fused layer 0 needs return_new_p_vecs")
            return self._run(batch, obj_vecs, pred_vecs, first=1)
        obj_vecs = self.attribute_embedding(objs_flat, self._act_dtype())
        pred_vecs = embedding_lookup(self.pred_embeddings.weight, pred_ids, self._act_dtype())
        return self._run(batch, obj_vecs, pred_vecs)

    def refresh_weight_copies(self):
        """Tensor-core engine: refresh the cached 16-bit copies of all layers' weights in one launch (call after every
        optimizer step; ``pipeline.SgToLayoutStep`` does).  Without it every layer casts its weights inside its call."""
        if self.precision in ("bf16", "fp16"):
            from . import graph_tc
            graph_tc.refresh_weight_copies(list(self.gconvs), self._act_dtype())
            if self.mask_net is not None:
                from . import mask_head
                mask_head.refresh_weight_copies(self.mask_net, self._act_dtype())

    def _run(self, batch, obj_vecs, pred_vecs, first=0):
        layers = list(self.gconvs)[first:]
        w = self.trans_candidates_weights
        if self.precision in ("bf16", "fp16") and batch.NT > 0 and all(l.predicates_transitive_weights is w for l in layers):
            # the triple confidences (graph.py:69-74) depend on the batch and on w_trans only: once for all layers
            from .graph import triple_confidence
            batch._conf_shared = ((w.data_ptr(), w._version), triple_confidence(batch, w))
        try:
            for layer in layers:
                obj_vecs, pred_vecs = layer.forward_flat(batch, obj_vecs, pred_vecs)
        finally:
            batch._conf_shared = None
        boxes = dense_mlp2(obj_vecs, self.box_net[0].weight, self.box_net[0].bias,
                           self.box_net[2].weight, self.box_net[2].bias, False, self.precision)
        return obj_vecs, boxes

    def masks_from_vecs(self, obj_vecs):
        """The mask head (model.py:62-75,121-123) on object vectors [NO, D] (the GCN's output) -> masks_pred [NO, M, M]
        fp32 in (0, 1).  BatchNorm uses the batch statistics of exactly these rows in training mode (and updates the
        running buffers), the running buffers in eval mode.  Needs ``mask_size > 0``."""
        if self.mask_net is None:
            raise ValueError("masks_from_vecs needs a model built with mask_size > 0")
        from .mask_head import mask_head
        return mask_head(self.mask_net, obj_vecs, self.precision)

    def forward(self, objs, triplets, triplet_type, boxes_gt=None, masks_gt=None):
        """Padded interface (model.py:90-124): objs [B,O,A] i64, triplets [B,T,3] i64, triplet_type [B,T] i64
        -> (obj_vecs [B,O,D], boxes_pred [B,O,4], masks_pred [B,O,M,M] or None when mask_size == 0).  The mask head
        sees every row of the padded batch, padded objects included, as the box head does."""
        B, O, T = objs.size(0), objs.size(1), triplets.size(1)
        batch = TripleBatch.from_padded_triplets(triplets, triplet_type, self.padding_id, O, self.num_preds)
        obj_vecs, boxes = self._embed_and_run(batch, objs.reshape(B * O, -1), triplets.reshape(B * T, 3)[:, 1])
        masks = None
        if self.mask_net is not None:
            masks = self.masks_from_vecs(obj_vecs)
            masks = masks.view(B, O, masks.shape[1], masks.shape[2])
        return obj_vecs.view(B, O, -1), boxes.view(B, O, 4), masks

    def forward_ragged(self, objs, triplets, triplet_type, tri_off, obj_off):
        """Flat interface: objs [NO,A], triplets [NT,3] (graph-local ids), triplet_type [NT], offsets [B+1] i32
        -> (obj_vecs [NO,D], boxes_pred [NO,4])."""
        batch = TripleBatch.from_ragged(triplets, triplet_type, tri_off, obj_off, objs.size(0), self.padding_id,
                                        self.num_preds)
        return self._embed_and_run(batch, objs, triplets[:, 1])
