"""Layout compositor: drop-in for ``sg2im/layout.py`` of the reference.

``boxes_to_layout`` / ``masks_to_layout`` keep the reference's signatures
(``sg2im/layout.py:12,48``: one image per call, boxes ``[x0, y0, w, h]``) and
add ``align_corners`` (the reference relies on the torch default, which flipped
from True to False in torch 1.3; SURVEY.md §7).  ``layout_batched`` is the
ragged form (flat objects + ``obj_offsets``), one launch for all images, whose
result equals ``torch.cat`` of the per-image reference calls
(``spade/models/networks/generator.py:81-96``).

``out_dtype`` (``torch.float32`` default, ``torch.bfloat16`` or ``torch.float16``)
selects the element type of the canvas: a 16-bit canvas is the fp32 canvas
rounded once (``canvas.to(out_dtype)``, written directly by the kernels), and a
16-bit gradient of it is read directly by the backward kernels, whose results
are those of the fp32 path given ``grad.float()``.  Inputs and their gradients
stay fp32.

All arithmetic runs in ``csg_layout_*`` (csrc/layout.cu); a missing library or
CPU tensors raise.
"""
import torch

from . import _lib
from .ops import lib, ptr, need_cuda, f32c, workspace, _stream

_LIN = {}
_CANVAS_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


def _check_dtype(out_dtype):
    if out_dtype not in _CANVAS_DTYPES:
        raise ValueError("out_dtype must be torch.float32, torch.bfloat16 or torch.float16 (got %s)" % (out_dtype,))
    return out_dtype


def _fp16_flag(dtype):
    """``None`` for an fp32 tensor, else the ``fp16`` argument of the ``*_bf16`` entry points."""
    return None if dtype == torch.float32 else int(dtype == torch.float16)


def _linspace(steps, device):
    """fp32 ``torch.linspace(0, 1, steps)`` built on the CPU and moved, exactly like
    ``sg2im/layout.py:98-99`` (``torch.linspace(...).to(boxes)``)."""
    key = (int(steps), str(device))
    t = _LIN.get(key)
    if t is None:
        t = torch.linspace(0, 1, steps=int(steps)).to(device)
        _LIN[key] = t
    return t


def _offsets(obj_offsets, device):
    if obj_offsets.dtype != torch.int32:
        obj_offsets = obj_offsets.to(torch.int32)
    return obj_offsets.to(device).contiguous()


class _LayoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vecs, boxes, masks, obj_off, H, W, align_corners, max_objs, lin_x=None, lin_y=None,
                out_dtype=torch.float32):
        need_cuda(vecs, boxes, masks, obj_off)
        vecs_c, boxes_c = f32c(vecs), f32c(boxes)
        masks_c = f32c(masks) if masks is not None else None
        NO, D = vecs_c.shape
        N = obj_off.numel() - 1
        M = masks_c.shape[1] if masks_c is not None else 0
        # the canvas coordinates of the pixel columns / rows: torch.linspace(0, 1, W) / (0, 1, H) unless the caller
        # samples a sub-lattice of a finer canvas (layout_pyramid)
        lin_x = _linspace(W, vecs.device) if lin_x is None else lin_x
        lin_y = _linspace(H, vecs.device) if lin_y is None else lin_y
        ctx.lin = (lin_x, lin_y)
        out = torch.empty((N, D, H, W), dtype=out_dtype, device=vecs.device)
        args = (ptr(vecs_c), ptr(boxes_c), ptr(masks_c), ptr(obj_off), ptr(lin_x), ptr(lin_y), ptr(out), N, D, H, W, M,
                int(align_corners), int(max_objs))
        fp16 = _fp16_flag(out_dtype)
        if fp16 is None:
            _lib.check(lib().csg_layout_fwd(*args, _stream()), "csg_layout_fwd")
        else:
            _lib.check(lib().csg_layout_fwd_bf16(*args, fp16, _stream()), "csg_layout_fwd_bf16")
        ctx.save_for_backward(vecs_c, boxes_c, masks_c, obj_off)
        ctx.dims = (N, NO, D, H, W, M, int(align_corners), int(max_objs))
        ctx.masks_float = masks is not None and masks.is_floating_point()
        return out

    @staticmethod
    def backward(ctx, dout):
        vecs, boxes, masks, obj_off = ctx.saved_tensors
        N, NO, D, H, W, M, align, max_objs = ctx.dims
        # a 16-bit gradient goes to the kernels as it is: they widen it on load
        dout = dout.contiguous() if dout.dtype in (torch.bfloat16, torch.float16) else f32c(dout)
        fp16 = _fp16_flag(dout.dtype)
        dvecs = dboxes = dmasks = None
        L = lib()
        lin_x, lin_y = ctx.lin
        want_dm = ctx.needs_input_grad[2] and ctx.masks_float
        if ctx.needs_input_grad[0] and want_dm and not ctx.needs_input_grad[1]:
            # predicted masks on fixed boxes (the training step with a mask head): d vecs and d masks from one entry
            # point, d masks band-tiled instead of one pass over the gradient per object
            dvecs = torch.empty((NO, D), dtype=torch.float32, device=dout.device)
            dmasks = torch.empty_like(masks)
            ws = workspace(L.csg_layout_bwd_vecs_masks_workspace(N, NO, D, H, W, M), dout.device)
            args = (ptr(dout), ptr(vecs), ptr(boxes), ptr(masks), ptr(obj_off), ptr(lin_x), ptr(lin_y), ptr(dvecs),
                    ptr(dmasks), N, NO, D, H, W, M, align, max_objs)
            if fp16 is None:
                rc = L.csg_layout_bwd_vecs_masks(*args, ptr(ws), ws.numel(), _stream())
            else:
                rc = L.csg_layout_bwd_vecs_masks_bf16(*args, fp16, ptr(ws), ws.numel(), _stream())
            _lib.check(rc, "csg_layout_bwd_vecs_masks")
            return dvecs, None, dmasks, None, None, None, None, None, None, None, None
        if ctx.needs_input_grad[0]:
            dvecs = torch.empty((NO, D), dtype=torch.float32, device=dout.device)
            ws = workspace(L.csg_layout_bwd_vecs_workspace(N, NO, D, H, W), dout.device)
            args = (ptr(dout), ptr(boxes), ptr(masks), ptr(obj_off), ptr(lin_x), ptr(lin_y), ptr(dvecs), N, NO, D, H, W,
                    M, align, max_objs)
            if fp16 is None:
                rc = L.csg_layout_bwd_vecs(*args, ptr(ws), ws.numel(), _stream())
            else:
                rc = L.csg_layout_bwd_vecs_bf16(*args, fp16, ptr(ws), ws.numel(), _stream())
            _lib.check(rc, "csg_layout_bwd_vecs")
        need_geom = ctx.needs_input_grad[1] or (ctx.needs_input_grad[2] and ctx.masks_float)
        if need_geom:
            dboxes = torch.empty((NO, 4), dtype=torch.float32, device=dout.device)
            want_dm = ctx.needs_input_grad[2] and ctx.masks_float
            dmasks = torch.empty_like(masks) if want_dm else None
            ws = workspace(L.csg_layout_bwd_geom_workspace(NO), dout.device)
            args = (ptr(dout), ptr(vecs), ptr(boxes), ptr(masks), ptr(obj_off), ptr(lin_x), ptr(lin_y), ptr(dboxes),
                    ptr(dmasks), N, NO, D, H, W, M, align)
            if fp16 is None:
                rc = L.csg_layout_bwd_geom(*args, ptr(ws), ws.numel(), _stream())
            else:
                rc = L.csg_layout_bwd_geom_bf16(*args, fp16, ptr(ws), ws.numel(), _stream())
            _lib.check(rc, "csg_layout_bwd_geom")
            if not ctx.needs_input_grad[1]:
                dboxes = None
        return dvecs, dboxes, dmasks, None, None, None, None, None, None, None, None


def nearest_source_index(out_size, in_size, device):
    """Source index of every output index of ``F.interpolate(mode='nearest')`` (ATen nearest_neighbor_compute_source_index:
    ``min(floor(dst * in / out), in - 1)`` with the scale evaluated in float32)."""
    scale = torch.tensor(float(in_size) / float(out_size), dtype=torch.float32)
    idx = torch.floor(torch.arange(out_size, dtype=torch.float32) * scale).to(torch.int64).clamp_(max=in_size - 1)
    return idx.to(device)


def layout_pyramid(vecs, boxes, obj_offsets, H, W=None, sizes=(), masks=None, align_corners=False,
                   max_objs_per_image=0, out_dtype=torch.float32):
    """The canvas together with the nearest-neighbour resizes of it that the SPADE consumers compute from it:
    ``F.interpolate(seg, size=(sh, sw))`` of the generator head (spade/models/networks/generator.py:99) and
    ``F.interpolate(segmap, size=x.size()[2:], mode='nearest')`` of every SPADE block (normalization.py:102), which
    re-read the 268-512 MiB canvas about seven times per forward.

    A nearest resize only selects pixels, and a canvas pixel depends on nothing but its own coordinates
    (layout.py:98-101), so level (h, w) IS the compositor evaluated on the sub-lattice ``lin_y[src_y], lin_x[src_x]``:
    every level is written directly by the compositor kernels (bit-identical to slicing the full canvas), the big
    canvas is never re-read, and the backward pass adds the levels' gradients into d vecs / d boxes with the same
    kernels on the same sub-lattices.  Returns ``(canvas [N, D, H, W], [level [N, D, h, w] for (h, w) in sizes])``, all of dtype ``out_dtype``."""
    _check_dtype(out_dtype)
    W = H if W is None else W
    need_cuda(vecs, boxes, masks)
    off = _offsets(obj_offsets, vecs.device)
    canvas = _LayoutFn.apply(vecs, boxes, masks, off, int(H), int(W), bool(align_corners), int(max_objs_per_image),
                             None, None, out_dtype)
    lin_x, lin_y = _linspace(W, vecs.device), _linspace(H, vecs.device)
    levels = []
    for size in sizes:
        h, w = (size, size) if isinstance(size, int) else size
        ly = lin_y[nearest_source_index(h, H, vecs.device)].contiguous()
        lx = lin_x[nearest_source_index(w, W, vecs.device)].contiguous()
        levels.append(_LayoutFn.apply(vecs, boxes, masks, off, int(h), int(w), bool(align_corners),
                                      int(max_objs_per_image), lx, ly, out_dtype))
    return canvas, levels


def layout_batched(vecs, boxes, obj_offsets, H, W=None, masks=None, pooling="sum", test_mode=False,
                   align_corners=False, max_objs_per_image=0, out_dtype=torch.float32):
    """Ragged compositor: ``vecs [NO, D]``, ``boxes [NO, 4]`` (xywh), optional ``masks [NO, M, M]``,
    ``obj_offsets [N+1]`` (objects of image n are ``obj_offsets[n]:obj_offsets[n+1]``)
    -> ``[N, D, H, W]`` of dtype ``out_dtype``.  ``max_objs_per_image`` is a sizing hint (0 = unknown)."""
    _check_dtype(out_dtype)
    if pooling not in ("sum", "avg"):
        raise ValueError('Invalid pooling "%s"' % pooling)
    W = H if W is None else W
    need_cuda(vecs, boxes, masks)
    off = _offsets(obj_offsets, vecs.device)
    if masks is not None:
        O, M = masks.shape[0], masks.shape[1]
        assert tuple(masks.shape) == (vecs.shape[0], M, M)            # layout.py:63
    if test_mode:
        if masks is None:
            raise ValueError("test_mode needs masks")
        return _occlude(vecs, boxes, masks, off, H, W, align_corners, out_dtype)
    out = _LayoutFn.apply(vecs, boxes, masks, off, int(H), int(W), bool(align_corners), int(max_objs_per_image),
                          None, None, out_dtype)
    if pooling == "avg":                                              # layout.py:176-184 (in the canvas dtype)
        cnt = (off[1:] - off[:-1]).clamp(min=1).to(out.dtype)
        out = out / cnt.view(-1, 1, 1, 1)
    return out


def _occlude(vecs, boxes, masks, off, H, W, align_corners, out_dtype=torch.float32):
    L = lib()
    vecs_c, boxes_c, masks_c = f32c(vecs), f32c(boxes), f32c(masks)
    NO, D = vecs_c.shape
    N, M = off.numel() - 1, masks_c.shape[1]
    out = torch.empty((N, D, H, W), dtype=out_dtype, device=vecs.device)
    ws = workspace(L.csg_layout_occlude_workspace(N, NO), vecs.device)
    lin_x, lin_y = _linspace(W, vecs.device), _linspace(H, vecs.device)
    args = (ptr(vecs_c), ptr(boxes_c), ptr(masks_c), ptr(off), ptr(lin_x), ptr(lin_y), ptr(out), N, NO, D, H, W, M,
            int(align_corners))
    fp16 = _fp16_flag(out_dtype)
    if fp16 is None:
        rc = L.csg_layout_occlude_fwd(*args, ptr(ws), ws.numel(), _stream())
    else:
        rc = L.csg_layout_occlude_fwd_bf16(*args, fp16, ptr(ws), ws.numel(), _stream())
    _lib.check(rc, "csg_layout_occlude_fwd")
    return out


def _boxes_to_grid(boxes, H, W):
    """``sg2im/layout.py:80-112``: boxes [O, 4] xywh -> sampling grid [O, H, W, 2] in [-1, 1].  The
    compositor kernels evaluate this chain per pixel and never materialise the grid; the function is
    kept for callers that feed ``F.grid_sample`` themselves (elementwise torch ops on the caller's device)."""
    need_cuda(boxes)
    O = boxes.size(0)
    b = boxes.view(O, 4, 1, 1)
    X = (_linspace(W, boxes.device).view(1, 1, W).to(boxes) - b[:, 0]) / b[:, 2]
    Y = (_linspace(H, boxes.device).view(1, H, 1).to(boxes) - b[:, 1]) / b[:, 3]
    return torch.stack([X.expand(O, H, W), Y.expand(O, H, W)], dim=3).mul(2).sub(1)


def _pool_samples(samples, pooling="sum"):
    """``sg2im/layout.py:156-188``: samples [O, D, H, W] of ONE image -> [1, D, H, W].  Only used by callers
    that already hold materialised samples; ``boxes_to_layout`` / ``masks_to_layout`` never build them."""
    need_cuda(samples)
    O = samples.size(0)
    out = samples.sum(dim=0, keepdim=True)
    if pooling == "avg":
        out = out / max(O, 1)
    elif pooling != "sum":
        raise ValueError('Invalid pooling "%s"' % pooling)
    return out


def _single_offsets(O, device):
    return torch.tensor([0, O], dtype=torch.int32, device=device)


def boxes_to_layout(vecs, boxes, H, W=None, pooling="sum", align_corners=False, out_dtype=torch.float32):
    """``sg2im/layout.py:12-45``: vecs [O, D], boxes [O, 4] xywh -> [1, D, H, W]."""
    _check_dtype(out_dtype)
    O = vecs.size(0)
    return layout_batched(vecs, boxes, _single_offsets(O, vecs.device), H, W, None, pooling,
                          align_corners=align_corners, max_objs_per_image=O, out_dtype=out_dtype)


def masks_to_layout(vecs, boxes, masks, H, W=None, pooling="sum", test_mode=False, align_corners=False,
                    out_dtype=torch.float32):
    """``sg2im/layout.py:48-77``: + masks [O, M, M] (int 0/1 or float)."""
    _check_dtype(out_dtype)
    O = vecs.size(0)
    if pooling != "sum":                                              # layout.py:150-151
        raise ValueError('Invalid pooling "%s"' % pooling)
    return layout_batched(vecs, boxes, _single_offsets(O, vecs.device), H, W, masks, pooling, test_mode=test_mode,
                          align_corners=align_corners, max_objs_per_image=O, out_dtype=out_dtype)
