"""Mask head of ``Sg2LayoutModel`` (sg2im/model.py:62-75, ``mask_size > 0``): a soft ``M x M`` mask per object.

``build_mask_net`` is the reference's ``_build_mask_net`` module for module, so the state-dict keys are the reference's
(``mask_net.{1,5,9,13}.*`` BatchNorm2d, ``mask_net.{2,6,10,14}.*`` 3x3 Conv2d, ``mask_net.16.*`` 1x1 Conv2d for
``mask_size = 16``).  It is a parameter container only; ``mask_head`` runs it on the csg2im kernels:

    stage (s -> 2s)   BatchNorm at low resolution (csg_mask_bn_fwd) -> patch matrix A [O (2s)^2, 9C] of the upsampled,
                      normalised, zero-padded input (csg_mask_patch) -> GEMM with conv.weight.view(C, 9C) + bias + ReLU
    head              1x1 convolution + sigmoid as a row-dot (csg_head_fwd_ex)
    backward          head (sigmoid' and the last ReLU folded into dZ), then per stage dW = dZ^T A (MN-major split-K GEMM),
                      db = column sums, dA = dZ W, and csg_mask_bn_bwd (nine-tap / 2x2 adjoint + BatchNorm backward with
                      the previous ReLU folded in)

Engines follow the model's precision: ``'fp32'`` on the parity GEMMs (``csg_gemm_f32``), ``'bf16'`` on tcgen05 with bf16
activations, ``'fp16'`` the same with fp16 forward tensors, inference only.  The patch matrices are not kept for the
backward: each stage rebuilds its own from the saved low-resolution input (the same kernel, bitwise the same matrix), so
only one stage's A and dA are alive at a time -- at 2.2 k objects and M = 16 the four bf16 patch matrices come to 1.75 GB,
the largest alone to 1.3 GB.  No host synchronisation anywhere.
"""
import os

import torch
import torch.nn as nn

from . import _lib
from . import ops
from .ops import lib, ptr, f32c, workspace, need_cuda, _stream

BF, F16 = torch.bfloat16, torch.float16
_FMT = {torch.float32: 0, BF: 1, F16: 2}


def build_mask_net(dim, mask_size):
    """sg2im/model.py:62-75 (``_build_mask_net``): [Upsample, BatchNorm2d, Conv2d 3x3, ReLU] per doubling, then a 1x1
    Conv2d to one channel.  Raises the reference's ValueError when ``mask_size`` is not a power of two."""
    output_dim = 1
    layers, cur_size = [], 1
    while cur_size < mask_size:
        layers.append(nn.Upsample(scale_factor=2, mode="nearest"))
        layers.append(nn.BatchNorm2d(dim))
        layers.append(nn.Conv2d(dim, dim, kernel_size=3, padding=1))
        layers.append(nn.ReLU())
        cur_size *= 2
    if cur_size != mask_size:
        raise ValueError("Mask size must be a power of 2")
    layers.append(nn.Conv2d(dim, output_dim, kernel_size=1))
    return nn.Sequential(*layers)


def _stages(net):
    """[(BatchNorm2d, Conv2d 3x3)] per stage and the final 1x1 Conv2d."""
    mods = list(net)
    return [(mods[i + 1], mods[i + 2]) for i in range(0, len(mods) - 1, 4)], mods[-1]


# ---------------------------------------------------------------------------------------------------------------
# 16-bit weight copies of the tensor-core engine: W [C, 9C] (forward B operand) and W^T [9C, C] (dA's B operand), kept
# across calls on the terms of graph_tc's copies.  An entry holds its weight tensors (so their storage cannot be freed
# and reused by another net while the entry exists) and is valid while those same tensors have the versions it was cast
# from: autograd's version counters catch every in-place torch update, and FusedAdam, which writes the parameters
# through raw pointers, marks the entries of its parameters stale (graph_tc.invalidate_weight_copies calls
# invalidate_weight_copies below).  A stale or missing entry makes the call cast its weights itself: forgetting
# refresh_weight_copies costs time, never correctness.
# ---------------------------------------------------------------------------------------------------------------
_WCOPIES = {}      # data_ptr of the first 3x3 conv weight -> dict(act, params, shapes, versions, copies)


def _conv_weights(net):
    return [conv.weight for _, conv in _stages(net)[0]]


def _cast(weights, act, outs=None):
    from .graph_tc import cast_bf16_multi
    jobs = []
    for w in weights:
        m = w.detach().reshape(w.shape[0], -1)
        jobs += [(m, False), (m, True)]
    return cast_bf16_multi(jobs, act, outs)


def refresh_weight_copies(net, act=BF):
    """Cast the 3x3 convolution weights of ``net`` into their cached 16-bit copies (one launch).  The copies are
    allocated on first use (or when the weights, their shapes or ``act`` change) and refilled in place afterwards: a
    captured CUDA graph holds their addresses, so its replays read the copies of the current weights."""
    weights = _conv_weights(net)
    if not weights or any(not w.is_cuda or w.dtype != torch.float32 for w in weights):
        return
    e = _WCOPIES.get(weights[0].data_ptr())
    if (e is not None and e["act"] == act and len(e["params"]) == len(weights)
            and all(a is b for a, b in zip(e["params"], weights))
            and all(tuple(a.shape) == tuple(b) for a, b in zip(weights, e["shapes"]))):
        _cast(weights, act, e["copies"])
        e["versions"] = tuple(w._version for w in weights)
        return
    _WCOPIES[weights[0].data_ptr()] = {"act": act, "params": tuple(weights), "shapes": [tuple(w.shape) for w in weights],
                                       "versions": tuple(w._version for w in weights), "copies": _cast(weights, act)}


def invalidate_weight_copies(params=None):
    """Mark the cached copies stale (the entries holding any of ``params``; all when None)."""
    ptrs = None if params is None else {p.data_ptr() for p in params}
    for e in _WCOPIES.values():
        if ptrs is None or ptrs & {q.data_ptr() for q in e["params"]}:
            e["versions"] = None


def _weight_copies(weights, act):
    e = _WCOPIES.get(weights[0].data_ptr()) if os.environ.get("CSG_WCOPIES", "1") != "0" else None
    if (e is not None and e["act"] == act and len(e["params"]) == len(weights)
            and all(a is b for a, b in zip(e["params"], weights))
            and e["versions"] == tuple(w._version for w in weights)):
        return e["copies"]
    return _cast(weights, act)


# ---------------------------------------------------------------------------------------------------------------
# one autograd node for the whole head
# ---------------------------------------------------------------------------------------------------------------
def _bn_fwd(x, n, C, bn, training, momentum):
    dev = x.device
    st = torch.empty((4, C), dtype=torch.float32, device=dev)        # mean, scale, beta, invstd
    L = lib()
    ws = workspace(L.csg_mask_bn_fwd_workspace(n, C), dev)
    rm, rv, nbt = bn.running_mean, bn.running_var, bn.num_batches_tracked
    _lib.check(L.csg_mask_bn_fwd(ptr(x), _FMT[x.dtype], n, C, ptr(f32c(bn.weight.detach())), ptr(rm), ptr(rv), ptr(nbt),
                                 float(momentum), float(bn.eps), int(training), ptr(st[1]), ptr(st[0]), ptr(st[3]),
                                 ptr(ws), ws.numel(), _stream()), "csg_mask_bn_fwd")
    st[2] = bn.bias.detach()
    return st


def _patch(x, O, s, C, st, dtype):
    A = torch.empty((O * 4 * s * s, 9 * C), dtype=dtype, device=x.device)
    _lib.check(lib().csg_mask_patch(ptr(x), _FMT[x.dtype], O, s, C, ptr(st[0]), ptr(st[1]), ptr(st[2]), ptr(A),
                                    _FMT[dtype], _stream()), "csg_mask_patch")
    return A


def _conv_fwd(A, w, b, wcopy, act):
    M, K = A.shape
    C = w.shape[0]
    if act == torch.float32:
        return ops.gemm_f32(ops.A_ROW, ops.B_NK, M, C, K, A, f32c(w.detach()).view(C, K), bias=f32c(b.detach()), relu=True)
    return ops.gemm_bf16(M, C, K, A, wcopy, bias=f32c(b.detach()), relu=True, out_dtype=act)


class _MaskHeadFn(torch.autograd.Function):
    """masks [O, M, M] fp32 = sigmoid(mask_net(x.view(O, C, 1, 1))).  Inputs: (engine, net, training, grad_on, x,
    then gamma, beta, conv weight, conv bias per stage, then the 1x1 weight and bias).  engine: 'fp32' or 'tc'."""

    @staticmethod
    def forward(ctx, engine, net, training, grad_on, x, *params):
        stages, head = _stages(net)
        O, C = x.shape
        nst = len(stages)
        act = torch.float32 if engine == "fp32" else (F16 if x.dtype == F16 else BF)
        need_bwd = grad_on and any(ctx.needs_input_grad[4:])
        if act == F16 and need_bwd:
            from .graph_tc import INFERENCE_ONLY
            raise _lib.CsgError(INFERENCE_ONLY)
        M = 2 ** nst
        dev = x.device
        xin = x.detach()
        if xin.dtype != act:
            xin = xin.to(act)
        xin = xin.contiguous()
        ctx.engine, ctx.training, ctx.act, ctx.dims = engine, training, act, (O, C, nst)
        ctx.set_materialize_grads(False)
        if O == 0:
            # BatchNorm2d on an empty batch (torch 2.11): empty output, num_batches_tracked += 1, running buffers kept
            for bn, _ in stages:
                _bn_fwd(xin, 0, C, bn, training, bn.momentum)
            ctx.x_dtype = x.dtype
            ctx.param_shapes = [tuple(p.shape) for p in params]
            return torch.empty((0, M, M), dtype=torch.float32, device=dev)
        convs = [conv for _, conv in stages]
        wcopies = _weight_copies([c.weight for c in convs], act) if act != torch.float32 and convs else None
        xs, sts, cur = [], [], xin
        for i, (bn, conv) in enumerate(stages):
            s = 2 ** i
            if bn.momentum is None:
                raise ValueError("mask_net BatchNorm2d with momentum=None (cumulative average) is not supported")
            st = _bn_fwd(cur, O * s * s, C, bn, training, bn.momentum)
            A = _patch(cur, O, s, C, st, act)
            z = _conv_fwd(A, conv.weight, conv.bias, wcopies[2 * i] if wcopies else None, act)
            del A
            xs.append(cur)
            sts.append(st)
            cur = z
        hw, hb = f32c(head.weight.detach()).view(1, C), f32c(head.bias.detach())
        masks = torch.empty((O * M * M,), dtype=torch.float32, device=dev)
        _lib.check(lib().csg_head_fwd_ex(ptr(cur), C, _FMT[act], ptr(hw), ptr(hb), O * M * M, C, 1, 1, ptr(masks),
                                         _stream()), "csg_head_fwd_ex")
        if need_bwd:
            ctx.wt = [wcopies[2 * i + 1] for i in range(nst)] if wcopies else None
            ctx.sts = sts
            ctx.save_for_backward(*xs, cur, masks, hw, *[f32c(c.weight.detach()) for c in convs],
                                  *[f32c(bn.weight.detach()) for bn, _ in stages])
        ctx.x_dtype = x.dtype
        return masks.view(O, M, M)

    @staticmethod
    def backward(ctx, dmasks):
        O, C, nst = ctx.dims
        act = ctx.act
        if dmasks is None:
            return (None,) * (5 + 4 * nst + 2)
        if O == 0:
            # an empty batch: zero gradients, no kernel reads an empty tensor
            dev = dmasks.device
            return (None, None, None, None, torch.zeros((0, C), dtype=ctx.x_dtype, device=dev)) + tuple(
                torch.zeros(shp, dtype=torch.float32, device=dev) for shp in ctx.param_shapes)
        saved = ctx.saved_tensors
        xs, z_last, masks, hw = saved[:nst], saved[nst], saved[nst + 1], saved[nst + 2]
        ws_conv, gammas = saved[nst + 3:2 * nst + 3], saved[2 * nst + 3:]
        dev = masks.device
        L = lib()
        R = masks.numel()
        dmasks = f32c(dmasks).view(-1)
        # head: dZ = (Z > 0) * sigmoid'(.) * dmask * w, dw / db of the 1x1 convolution; with no stage (mask_size = 1)
        # the head reads obj_vecs directly and there is no ReLU to fold
        x_out = ctx.x_dtype if ctx.x_dtype in _FMT else torch.float32       # dtype of d obj_vecs
        dz = torch.empty((R, C), dtype=act if nst else x_out, device=dev)
        dhw = torch.empty((1, C), dtype=torch.float32, device=dev)
        dhb = torch.empty(1, dtype=torch.float32, device=dev)
        ws = workspace(L.csg_head_bwd_ex_workspace(R, C, 1), dev)
        _lib.check(L.csg_head_bwd_ex(ptr(dmasks), ptr(masks), ptr(z_last), C, _FMT[act], ptr(hw), R, C, 1, ptr(dz), C,
                                     _FMT[dz.dtype], int(nst > 0), ptr(dhw), ptr(dhb), ptr(ws), ws.numel(), _stream()),
                   "csg_head_bwd_ex")
        grads = [None] * (4 * nst)
        for i in reversed(range(nst)):
            s = 2 ** i
            x, st, w = xs[i], ctx.sts[i], ws_conv[i]
            rows = O * 4 * s * s
            A = _patch(x, O, s, C, st, act)
            if act == torch.float32:
                dw = ops.gemm_f32(ops.A_COL, ops.B_KN, C, 9 * C, rows, dz, A)
                db = ops.colsum_f32(dz)
                del A
                dA = ops.gemm_f32(ops.A_ROW, ops.B_KN, rows, 9 * C, C, dz, w.view(C, 9 * C))
            else:
                from .graph_tc import colsum_bf16
                dw = ops.gemm_bf16(C, 9 * C, rows, dz, A, mn_major=True)
                db = colsum_bf16(dz)
                del A
                dA = ops.gemm_bf16(rows, 9 * C, C, dz, ctx.wt[i])
            n = O * s * s
            out_dtype = act if i > 0 else x_out
            dx = torch.empty((n, C), dtype=out_dtype, device=dev)
            dgb = torch.empty((2, C), dtype=torch.float32, device=dev)
            wsb = workspace(L.csg_mask_bn_bwd_workspace(n, C), dev)
            _lib.check(L.csg_mask_bn_bwd(ptr(dA), _FMT[dA.dtype], ptr(x), _FMT[x.dtype], O, s, C, ptr(gammas[i]),
                                         ptr(st[0]), ptr(st[3]), int(ctx.training), int(i > 0), ptr(dx), _FMT[out_dtype],
                                         ptr(dgb[0]), ptr(dgb[1]), ptr(wsb), wsb.numel(), _stream()), "csg_mask_bn_bwd")
            del dA
            grads[4 * i:4 * i + 4] = [dgb[0], dgb[1], dw.view(C, C, 3, 3), db]
            dz = dx
        return (None, None, None, None, dz) + tuple(grads) + (dhw.view(1, C, 1, 1), dhb)


def mask_head(net, obj_vecs, precision="fp32"):
    """``mask_net(obj_vecs.view(O, -1, 1, 1)).squeeze(1).sigmoid()`` (sg2im/model.py:62-75,115-124) on the csg2im kernels:
    obj_vecs [O, C] -> masks [O, M, M] fp32.  BatchNorm follows ``net.training`` (batch statistics and running-buffer
    update in training mode, running buffers in eval mode)."""
    need_cuda(obj_vecs)
    if obj_vecs.dim() != 2:
        raise ValueError("mask_head expects obj_vecs [O, C] (got %s)" % (tuple(obj_vecs.shape),))
    stages, head = _stages(net)
    C = obj_vecs.shape[1]
    engine = "fp32" if precision == "fp32" else "tc"
    if engine == "tc" and C % 64:
        raise _lib.CsgError("precision='%s' needs gconv_dim to be a multiple of 64 (got %d); use precision='fp32'"
                            % (precision, C))
    if engine == "fp32" and C % 8:
        raise _lib.CsgError("mask head: gconv_dim must be a multiple of 8 (got %d)" % C)
    if engine == "tc" and obj_vecs.dtype == torch.float32:
        obj_vecs = obj_vecs.to(F16 if precision == "fp16" else BF)
    params = [p for bn, conv in stages for p in (bn.weight, bn.bias, conv.weight, conv.bias)] + [head.weight, head.bias]
    return _MaskHeadFn.apply(engine, net, bool(net.training), torch.is_grad_enabled(), obj_vecs, *params)
