"""Backward of masks_to_layout wrt vecs and float masks together, boxes held fixed (csg_layout_bwd_vecs_masks, the
request of the training step with predicted masks): d vecs is bitwise csg_layout_bwd_vecs's, d masks agrees with the
float64 autograd of the reference compositor (F.grid_sample) and with the per-object kernel of csg_layout_bwd_geom
within 1e-5 of the tensor scale, 16-bit gradients give the results of their fp32 widening bit for bit, runs repeat bit
for bit, and a request that includes d boxes keeps today's kernels."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from canonicalsg2im_b200 import synth
from canonicalsg2im_b200.layout import layout_batched
from oracle.layout import boxes_to_grid
from tests.util import t, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _objs(seed, n_img, n_min, n_max, D, M=16, dummies=True):
    vocab = synth.Vocab(0)
    vecs, boxes, masks, off = [], [], [], [0]
    for i in range(n_img):
        g = synth.make_graph(seed * 100 + i, n_min, n_max, vocab, include_dummies=dummies, mask_size=M)
        n = len(g.boxes)
        vecs.append(synth.det_tensor((n, D), seed * 1000 + i, 1.0))
        boxes.append(g.boxes)
        masks.append(synth.det_uniform(n * M * M, seed * 1000 + i + 7).reshape(n, M, M).astype(np.float32))
        off.append(off[-1] + n)
    return t(np.concatenate(vecs)), t(np.concatenate(boxes)), t(np.concatenate(masks)), t(np.array(off, np.int32))


def _grad(N, D, H, W, seed, dtype=torch.float32):
    return t(synth.det_tensor((N, D, H, W), seed, 1.0)).to(dtype)


def _run(v, b, m, off, H, W, g, wrt=("vecs", "masks")):
    """Autograd of layout_batched wrt the inputs named in `wrt`: (d vecs, d boxes, d masks), None where not asked."""
    v = v.clone().requires_grad_("vecs" in wrt)
    b = b.clone().requires_grad_("boxes" in wrt)
    m = m.clone().requires_grad_("masks" in wrt)
    out = layout_batched(v, b, off, H, W, masks=m, out_dtype=g.dtype)
    out.backward(g)
    torch.cuda.synchronize()
    return v.grad, b.grad, m.grad


def _oracle_dmasks(v, b, m, off, H, W, g):
    """float64 autograd of masks_to_layout (sg2im/layout.py:48-77) per image on the GPU."""
    out = []
    offs = off.tolist()
    for n in range(len(offs) - 1):
        lo, hi = offs[n], offs[n + 1]
        O, D, M = hi - lo, v.shape[1], m.shape[1]
        mm = m[lo:hi].double().clone().requires_grad_(True)
        grid = boxes_to_grid(b[lo:hi].double(), H, W)
        img = v[lo:hi].double().view(O, D, 1, 1) * mm.view(O, 1, M, M)
        s = F.grid_sample(img, grid, mode="bilinear", padding_mode="zeros", align_corners=False).sum(0)
        s.backward(g[n].double())
        out.append(mm.grad)
    return torch.cat(out)


def _same_bits(a, b):
    """Bitwise equality that also holds for NaN entries (the rows of a poisoned box)."""
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def _check(v, b, m, off, H, W, seed, oracle=True):
    g = _grad(off.numel() - 1, v.shape[1], H, W, seed)
    dv_new, db_new, dm_new = _run(v, b, m, off, H, W, g)
    assert db_new is None
    dv_ref, _, _ = _run(v, b, m, off, H, W, g, wrt=("vecs",))
    assert _same_bits(dv_new, dv_ref), "d vecs differs from csg_layout_bwd_vecs"
    _, _, dm_geom = _run(v, b, m, off, H, W, g, wrt=("vecs", "boxes", "masks"))
    fin = torch.isfinite(dm_geom)
    assert torch.equal(fin, torch.isfinite(dm_new)), "non-finite rows differ from the per-object kernel"
    assert rel_err(dm_new[fin], dm_geom[fin]) <= TOL, rel_err(dm_new[fin], dm_geom[fin])
    if oracle:
        dm_o = _oracle_dmasks(v, b, m, off, H, W, g)
        assert rel_err(dm_new[fin], dm_o[fin]) <= TOL
    return dm_new


def test_cfg2_batch():
    """128 images of 3-30 objects plus the __image__ dummy (box -1), D = 128, 64 x 64, M = 16."""
    v, b, m, off = _objs(1, 128, 3, 30, 128)
    dm = _check(v, b, m, off, 64, 64, 11)
    dummy = (b[:, 0] == -1)
    assert dummy.any() and torch.equal(dm[dummy], torch.zeros_like(dm[dummy])), "the dummy rows must be exact zeros"


def test_canvas_256():
    """The cfg3 shape: 16 images, 256 x 256, D = 128 (a band is one row)."""
    v, b, m, off = _objs(2, 16, 3, 8, 128, dummies=False)
    _check(v, b, m, off, 256, 256, 12)


def test_chunking_many_objects():
    """70 objects in one 32 x 64 image and 40 in a second: several 16-object chunks per CTA and per band."""
    n1, n2 = 70, 40
    n = n1 + n2
    boxes = np.stack([synth.det_uniform(n, 1) * 0.3, synth.det_uniform(n, 2) * 0.3,
                      0.5 + 0.2 * synth.det_uniform(n, 3), 0.5 + 0.2 * synth.det_uniform(n, 4)], 1).astype(np.float32)
    v, b = t(synth.det_tensor((n, 32), 5, 1.0)), t(boxes)
    m = t(synth.det_uniform(n * 64, 6).reshape(n, 8, 8).astype(np.float32))
    off = torch.tensor([0, n1, n], dtype=torch.int32, device="cuda")
    _check(v, b, m, off, 32, 64, 13)


def test_edge_boxes():
    """Boxes partly and wholly outside the canvas, negative extents, the box -1 dummy, a NaN box and an image without
    objects: the NaN box gives a NaN row, objects that touch nothing exact-zero rows."""
    boxes = np.array([[-0.3, 0.2, 0.5, 0.4],      # partly left of the canvas
                      [0.8, 0.7, 0.5, 0.6],       # partly right / below
                      [1.5, 0.2, 0.3, 0.3],       # wholly right
                      [0.1, -2.0, 0.3, 0.5],      # wholly above
                      [0.6, 0.6, -0.3, -0.2],     # negative extents
                      [-1, -1, -1, -1],           # __image__ dummy
                      [0.2, 0.3, 0.4, 0.3],
                      [0.1, 0.1, float("nan"), 0.3],   # poisoned
                      [0.3, 0.1, 0.2, 0.7]], np.float32)
    n = len(boxes)
    v, b = t(synth.det_tensor((n, 64), 21, 1.0)), t(boxes)
    m = t(synth.det_uniform(n * 256, 22).reshape(n, 16, 16).astype(np.float32))
    off = torch.tensor([0, 7, 7, n], dtype=torch.int32, device="cuda")
    g = _grad(3, 64, 64, 128, 23)
    dv, _, dm = _run(v, b, m, off, 64, 128, g)
    assert torch.isnan(dm[7]).all()
    for o in (2, 3, 5):
        assert torch.equal(dm[o], torch.zeros_like(dm[o])), o
    dm_o = _oracle_dmasks(v[:7], b[:7], m[:7], off[:2], 64, 128, g[:1])
    assert rel_err(dm[:7], dm_o) <= TOL
    _check(v, b, m, off, 64, 128, 23, oracle=False)


@pytest.mark.parametrize("dtype", [pytest.param(torch.bfloat16, id="bf16"), pytest.param(torch.float16, id="fp16")])
@pytest.mark.parametrize("shape", [pytest.param((64, 64), id="64"), pytest.param((256, 256), id="256")])
def test_16bit_gradient_is_its_widening(dtype, shape):
    H, W = shape
    v, b, m, off = _objs(3, 16 if H == 256 else 64, 3, 30, 128)
    g16 = _grad(off.numel() - 1, 128, H, W, 31, dtype)
    dv16, _, dm16 = _run(v, b, m, off, H, W, g16)
    dv32, _, dm32 = _run(v, b, m, off, H, W, g16.float())
    assert _same_bits(dv16, dv32) and _same_bits(dm16, dm32)


def test_deterministic():
    v, b, m, off = _objs(4, 64, 3, 30, 128)
    g = _grad(64, 128, 64, 64, 41)
    a = _run(v, b, m, off, 64, 64, g)
    c = _run(v, b, m, off, 64, 64, g)
    assert _same_bits(a[0], c[0]) and _same_bits(a[2], c[2])


def test_dboxes_request_keeps_todays_kernels():
    """With boxes.requires_grad the per-object kernel still computes d boxes and d masks: equal to a direct
    csg_layout_bwd_geom call."""
    from canonicalsg2im_b200 import _lib
    from canonicalsg2im_b200.layout import _linspace
    from canonicalsg2im_b200.ops import lib, ptr, workspace, _stream
    v, b, m, off = _objs(5, 32, 3, 30, 128)
    N, NO, D, H, W, M = 32, v.shape[0], 128, 64, 64, 16
    g = _grad(N, D, H, W, 51)
    _, db, dm = _run(v, b, m, off, H, W, g, wrt=("vecs", "boxes", "masks"))
    dboxes = torch.empty((NO, 4), dtype=torch.float32, device="cuda")
    dmasks = torch.empty_like(m)
    ws = workspace(lib().csg_layout_bwd_geom_workspace(NO), "cuda")
    _lib.check(lib().csg_layout_bwd_geom(ptr(g), ptr(v), ptr(b), ptr(m), ptr(off), ptr(_linspace(W, "cuda")),
                                         ptr(_linspace(H, "cuda")), ptr(dboxes), ptr(dmasks), N, NO, D, H, W, M, 0,
                                         ptr(ws), ws.numel(), _stream()), "csg_layout_bwd_geom")
    torch.cuda.synchronize()
    assert _same_bits(db, dboxes) and _same_bits(dm, dmasks)
