"""16-bit layout canvases (``out_dtype`` = bf16 / fp16): the canvas is the fp32 canvas rounded once, bit for bit
(NaN where the fp32 canvas is NaN), and a 16-bit gradient gives exactly the fp32 path's gradients of ``g.float()``.
The backward shapes are chosen from the dispatch rules of ``csg_layout_bwd_vecs`` so that every kernel variant runs:
column sums (boxes, W = 64 / 128 / 256, H * W / 256 bands split 1 / 2 / 4 ways), the ring (masks, or boxes at a width
the column-sum kernel does not take) and the generic tile kernel (W % 64 != 0)."""
import numpy as np
import pytest
import torch

from canonicalsg2im_b200 import synth
from tests.util import t

pytestmark = pytest.mark.gpu
DTYPES = [pytest.param(torch.bfloat16, id="bf16"), pytest.param(torch.float16, id="fp16")]


@pytest.fixture(scope="module")
def L():
    from canonicalsg2im_b200 import layout
    return layout


def _objs(seed, n_img, n_min, n_max, D, M=4, box_mode="coco"):
    vocab = synth.Vocab(0)
    vecs, boxes, masks, off = [], [], [], [0]
    for i in range(n_img):
        g = synth.make_graph(seed * 100 + i, n_min, n_max, vocab, include_dummies=False, mask_size=M, box_mode=box_mode)
        n = len(g.boxes)
        vecs.append(synth.det_tensor((n, D), seed * 1000 + i, 1.0))
        boxes.append(g.boxes)
        masks.append(g.masks)
        off.append(off[-1] + n)
    return t(np.concatenate(vecs)), t(np.concatenate(boxes)), t(np.concatenate(masks)), t(np.array(off, np.int32))


def assert_rounded(x16, x32, dtype, what=""):
    """x16 == x32.to(dtype) bit for bit, NaN exactly where x32 is NaN (NaN payloads may differ)."""
    assert x16.dtype == dtype and x16.shape == x32.shape, what
    ref = x32.to(dtype)
    nan = torch.isnan(x32)
    assert torch.equal(torch.isnan(x16), nan), what + ": NaN positions differ"
    a, b = x16[~nan].view(torch.int16), ref[~nan].view(torch.int16)
    bad = (a != b).sum().item()
    assert bad == 0, "%s: %d of %d elements differ from the rounded fp32 canvas" % (what, bad, a.numel())


def _fwd_pair(L, dtype, *args, **kw):
    return L.layout_batched(*args, out_dtype=dtype, **kw), L.layout_batched(*args, **kw)


# ------------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("hint", [pytest.param(31, id="hint31"), pytest.param(0, id="hint0-multipass")])
def test_fwd_cfg2_boxes(L, dtype, hint):
    v, b, _, off = _objs(1, 128, 3, 31, 128)
    y16, y32 = _fwd_pair(L, dtype, v, b, off, 64, 64, max_objs_per_image=hint)
    assert_rounded(y16, y32, dtype, "cfg2 boxes")


@pytest.mark.parametrize("dtype", DTYPES)
def test_fwd_many_objects_multipass(L, dtype):
    """70 objects in one 32 x 64 canvas, hint 0 (a 16-entry list): every tile needs several passes."""
    n = 70
    boxes = np.stack([synth.det_uniform(n, 1) * 0.3, synth.det_uniform(n, 2) * 0.3,
                      0.5 + 0.2 * synth.det_uniform(n, 3), 0.5 + 0.2 * synth.det_uniform(n, 4)], 1).astype(np.float32)
    v, b = t(synth.det_tensor((n, 8), 5, 1.0)), t(boxes)
    off = torch.tensor([0, n], dtype=torch.int32, device="cuda")
    y16, y32 = _fwd_pair(L, dtype, v, b, off, 32, 64)
    assert_rounded(y16, y32, dtype, "70 objects")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("H,W,D", [pytest.param(48, 64, 8, id="CH4-D8"), pytest.param(40, 37, 16, id="scalar-W37"),
                                   pytest.param(24, 37, 8, id="scalar-W37-CH4")])
def test_fwd_narrow_shapes(L, dtype, H, W, D):
    v, b, _, off = _objs(2, 6, 1, 24, D)
    off = torch.cat([off[:2], off[1:]])                                   # an image without objects
    for hint in (0, 24):
        y16, y32 = _fwd_pair(L, dtype, v, b, off, H, W, max_objs_per_image=hint)
        assert_rounded(y16, y32, dtype, "H=%d W=%d D=%d hint %d" % (H, W, D, hint))
        assert (y16[1] == 0).all()


@pytest.mark.parametrize("dtype", DTYPES)
def test_fwd_nan_and_empty_images(L, dtype):
    v = torch.ones(3, 8, device="cuda")
    b = torch.tensor([[0.1, 0.1, 0.5, 0.5], [0.2, 0.2, 0.0, 0.3], [0.3, 0.3, 0.4, 0.4]], device="cuda")
    off = torch.tensor([0, 2, 2, 3], dtype=torch.int32, device="cuda")      # image 0 holds the w = 0 box, image 1 is empty
    y16, y32 = _fwd_pair(L, dtype, v, b, off, 16, 16)
    assert torch.isnan(y16[0]).all() and (y16[1] == 0).all() and torch.isfinite(y16[2]).all()
    assert_rounded(y16, y32, dtype, "NaN / empty")


def test_fwd_fp16_overflow_is_inf(L):
    v, b, _, off = _objs(3, 8, 3, 12, 16)
    y16, y32 = _fwd_pair(L, torch.float16, v * 3e5, b, off, 32, 32)
    assert (y32.abs() > 65520).any() and torch.isinf(y16).any()
    assert_rounded(y16, y32, torch.float16, "fp16 overflow")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("float_masks", [pytest.param(False, id="int-masks"), pytest.param(True, id="float-masks")])
def test_fwd_masks_256(L, dtype, float_masks):
    v, b, m, off = _objs(4, 4, 3, 20, 32, M=16)
    m = m.float() * (0.25 + 0.75 * torch.rand(m.shape, device="cuda", generator=torch.Generator("cuda").manual_seed(1))) \
        if float_masks else m
    y16, y32 = _fwd_pair(L, dtype, v, b, off, 256, 256, masks=m, max_objs_per_image=20)
    assert_rounded(y16, y32, dtype, "masks 256")


@pytest.mark.parametrize("dtype", DTYPES)
def test_pyramid_levels_and_grads(L, dtype):
    v, b, m, off = _objs(5, 3, 2, 7, 16, M=8)
    sizes = (32, 16, (8, 12))
    outs, grads = {}, {}
    for dt in (dtype, torch.float32):
        vg, bg = v.clone().requires_grad_(True), b.clone().requires_grad_(True)
        canvas, levels = L.layout_pyramid(vg, bg, off, 64, 64, sizes=sizes, masks=m, max_objs_per_image=7, out_dtype=dt)
        outs[dt] = [canvas] + levels
        gs = [torch.from_numpy(synth.det_tensor(tuple(x.shape), 300 + i, 1.0)).cuda().to(dtype) for i, x in enumerate(outs[dt])]
        torch.autograd.backward(outs[dt], [g.to(dt) for g in gs])
        grads[dt] = (vg.grad, bg.grad)
    for a, r in zip(outs[dtype], outs[torch.float32]):
        assert_rounded(a, r, dtype, "pyramid level %s" % (tuple(r.shape[2:]),))
    assert torch.equal(grads[dtype][0], grads[torch.float32][0]) and torch.equal(grads[dtype][1], grads[torch.float32][1])


@pytest.mark.parametrize("dtype", DTYPES)
def test_occlusion_single_and_cfg4(L, dtype):
    v, b, m, off = _objs(6, 1, 5, 9, 16, M=16)
    assert_rounded(L.masks_to_layout(v, b, m, 64, test_mode=True, out_dtype=dtype),
                   L.masks_to_layout(v, b, m, 64, test_mode=True), dtype, "masks_to_layout(test_mode=True)")
    v, b, m, off = _objs(21, 10, 32, 64, 128, M=16, box_mode="clevr")
    y16, y32 = _fwd_pair(L, dtype, v, b, off, 256, 256, masks=m, test_mode=True)
    assert_rounded(y16, y32, dtype, "occlusion cfg4")


def test_bad_dtype_raises(L):
    v = torch.ones(1, 8, device="cuda")
    b = torch.tensor([[0.1, 0.1, 0.5, 0.5]], device="cuda")
    for fn in (lambda: L.boxes_to_layout(v, b, 16, out_dtype=torch.float64),
               lambda: L.layout_pyramid(v, b, torch.tensor([0, 1], device="cuda"), 16, out_dtype=torch.float64)):
        with pytest.raises(ValueError):
            fn()


# ------------------------------------------------------------------------------------------------------ backward
def _grads(L, dtype, g16, v, b, off, H, W, masks=None, hint=0):
    """dvecs, dboxes, dmasks of the canvas in `dtype` given g16 (fp32 canvas: g16.float())."""
    vg, bg = v.clone().requires_grad_(True), b.clone().requires_grad_(True)
    mg = masks.clone().requires_grad_(True) if masks is not None and masks.is_floating_point() else masks
    y = L.layout_batched(vg, bg, off, H, W, masks=mg, max_objs_per_image=hint, out_dtype=dtype)
    y.backward(g16 if dtype != torch.float32 else g16.float())
    return vg.grad, bg.grad, (mg.grad if mg is not None and mg.requires_grad else None)


def _check_bwd(L, dtype, v, b, off, H, W, masks=None, hint=0, seed=7):
    N, D = off.numel() - 1, v.shape[1]
    g = torch.randn((N, D, H, W), device="cuda", generator=torch.Generator("cuda").manual_seed(seed)).to(dtype)
    a = _grads(L, dtype, g, v, b, off, H, W, masks, hint)
    r = _grads(L, torch.float32, g, v, b, off, H, W, masks, hint)
    for name, x, y in zip(("dvecs", "dboxes", "dmasks"), a, r):
        assert (x is None) == (y is None), name
        if x is not None:
            assert x.dtype == torch.float32 and torch.equal(x, y), name


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("W", [64, 128, 256])
@pytest.mark.parametrize("splits", [1, 2, 4])
def test_bwd_colsum(L, monkeypatch, dtype, W, splits):
    monkeypatch.setenv("CSG_LAYOUT_SPLITS", str(splits))
    v, b, _, off = _objs(11, 3, 3, 40, 64)
    off = torch.cat([off[:2], off[1:]])                                   # an empty image
    _check_bwd(L, dtype, v, b, off, 64, W, hint=0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_bwd_ring_masks_256(L, dtype):
    v, b, m, off = _objs(12, 4, 3, 20, 64, M=16)
    _check_bwd(L, dtype, v, b, off, 256, 256, masks=m, hint=20)
    fm = m.float() * 0.5 + 0.25
    _check_bwd(L, dtype, v, b, off, 64, 128, masks=fm, hint=20)        # float masks: dboxes and dmasks as well


@pytest.mark.parametrize("dtype", DTYPES)
def test_bwd_ring_boxes_w192(L, dtype):
    v, b, _, off = _objs(13, 4, 3, 40, 32)
    _check_bwd(L, dtype, v, b, off, 64, 192)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("W,masks", [pytest.param(40, False, id="generic-W40-boxes"),
                                     pytest.param(40, True, id="generic-W40-masks"),
                                     pytest.param(37, False, id="generic-W37-scalar")])
def test_bwd_generic(L, dtype, W, masks):
    v, b, m, off = _objs(14, 4, 3, 20, 32, M=8)
    _check_bwd(L, dtype, v, b, off, 48, W, masks=m.float() if masks else None, hint=20)


# ------------------------------------------------------------------------------------------------------ pipeline
def test_inference_pipeline_fp16_canvas():
    from canonicalsg2im_b200.pipeline import SgToLayoutInference, HostBatch
    sizes = list(synth.CLEVR_ATTR_SIZES)
    vocab = synth.Vocab(0, num_attributes=4)
    graphs = synth.make_graphs(4, 4400, 32, 64, vocab, include_dummies=True, box_mode="clevr", mask_size=16)
    for g in graphs:
        for k, n in enumerate(sizes):
            g.objs[:-1, k] = 1 + (g.objs[:-1, k] - 1) % (n - 1)
    hb = HostBatch(graphs, seed=4, with_geometry=True, num_uniforms=sum(4 * len(g.objs) ** 2 for g in graphs))
    out = {}
    for dt in (torch.float32, torch.float16):
        inf = SgToLayoutInference(vocab, "cuda", precision="fp16", H=128, W=128, embedding_dim=32, attr_sizes=sizes,
                                  canvas_dtype=dt)
        out[dt] = inf.step(hb.to_device("cuda"))[0]
    assert_rounded(out[torch.float16], out[torch.float32], torch.float16, "inference canvas")


@pytest.mark.parametrize("use_graph", [pytest.param(False, id="eager"), pytest.param(True, id="graph")])
def test_training_step_bf16_canvas(use_graph):
    """One training step with a bf16 canvas and canvas_grad = g16 gives the gradients of the fp32 step with
    g16.float(), eagerly and under CUDA-graph replay (second step: captured and replayed)."""
    from canonicalsg2im_b200.pipeline import SgToLayoutStep, HostBatch
    vocab = synth.Vocab(0)
    hb = HostBatch(synth.make_graphs(16, 1000, 3, 30, vocab, include_dummies=True), seed=0)
    g16 = (torch.randn((16, 128, 64, 64), device="cuda", generator=torch.Generator("cuda").manual_seed(9)) * 1e-3
           ).to(torch.bfloat16)
    grads = {}
    for dt in (torch.bfloat16, torch.float32):
        step = SgToLayoutStep(vocab, "cuda", seed=0, use_graph=use_graph, canvas_dtype=dt)
        d = hb.to_device("cuda")
        G = g16 if dt == torch.bfloat16 else g16.float()
        if use_graph:
            step.step(d, G)                      # eager (fills the host-side caches)
            step.step(d, G)                      # captured, then replayed
            step.finish()
            assert step.graph_replays == 1
            ent = next(iter(step._graphs.values()))
            grads[dt] = [g.detach().clone() for g in ent["grads"]]
        else:
            step.backward(d, G)
            grads[dt] = [g.detach().clone() for g in step.named_grads().values()]
    assert len(grads[torch.bfloat16]) == len(grads[torch.float32]) > 0
    for i, (a, b) in enumerate(zip(grads[torch.bfloat16], grads[torch.float32])):
        assert torch.equal(a, b), i
    with pytest.raises(ValueError):
        step.step(hb.to_device("cuda"), g16)          # the fp32 step refuses a bf16 canvas gradient
