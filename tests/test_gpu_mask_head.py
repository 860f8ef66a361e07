"""Mask head of Sg2LayoutModel (mask_size > 0) against the reference-structured nn.Sequential (sg2im/model.py:62-75)
run in float64 on the GPU with the same state: masks, running buffers after one step, and the gradients wrt obj_vecs
and every parameter.

Tolerances (relative L2).  Masks and running buffers: 1e-5 on the fp32 engine, 1e-2 on the tensor-core engines.
Gradients go through up to 5 ReLUs per element, and a pre-activation within rounding distance of zero flips its mask
under ANY change of arithmetic (DESIGN.md section 4.1): one flipped element changes its gradient by O(1), so the error
of a gradient is about sqrt(fraction of flipped pre-activations).  With 2 200 objects at M = 16 (72 M pre-activations
per stage) PyTorch's own fp32 run of the reference module differs from float64 by ~1e-3; with bf16 by 4e-2 .. 2e-1.
So a gradient must be within max(1e-5, 3 x err(PyTorch fp32)) on the fp32 engine -- 1e-5 wherever no mask flips, as
at 1 and 7 objects -- and within max(3e-2, 2 x err(PyTorch bf16)) on the bf16 engine, the errors of PyTorch measured on
the same inputs in the same test."""
import argparse

import pytest
import torch
import torch.nn as nn

from canonicalsg2im_b200 import synth, _lib
from canonicalsg2im_b200.mask_head import build_mask_net, mask_head
from tests.util import t

pytestmark = pytest.mark.gpu

CFG2_OBJS = 2200          # a cfg2 batch: 128 graphs of 3-30 objects plus __image__
TOL_F32 = 1e-5
TOL_TC_FWD = 1e-2
TOL_TC_BWD = 3e-2


def oracle_net(dim, mask_size):
    """sg2im's _build_mask_net, written out as the reference has it."""
    layers, cur = [], 1
    while cur < mask_size:
        layers += [nn.Upsample(scale_factor=2, mode="nearest"), nn.BatchNorm2d(dim),
                   nn.Conv2d(dim, dim, kernel_size=3, padding=1), nn.ReLU()]
        cur *= 2
    layers.append(nn.Conv2d(dim, 1, kernel_size=1))
    return nn.Sequential(*layers)


def _state(dim, mask_size, seed):
    g = torch.Generator().manual_seed(seed)
    net = oracle_net(dim, mask_size)
    st = {}
    for k, v in net.state_dict().items():
        if k.endswith("num_batches_tracked"):
            st[k] = torch.tensor(3, dtype=torch.int64)
        elif k.endswith("running_var"):
            st[k] = torch.rand(v.shape, generator=g) + 0.5
        elif k.endswith("running_mean") or k.endswith("bias"):
            st[k] = (torch.rand(v.shape, generator=g) - 0.5) * 0.4
        elif v.dim() == 1:                                                      # BatchNorm weight
            st[k] = torch.rand(v.shape, generator=g) + 0.5
        else:
            fan_in = v[0].numel()
            st[k] = (torch.rand(v.shape, generator=g) * 2 - 1) * (3.0 / fan_in) ** 0.5
    return st


def rel_l2(a, b):
    a, b = a.detach().double(), b.detach().double().to(a.device)
    return ((a - b).norm() / max(b.norm().item(), 1e-6)).item()


def _run_oracle(st, dim, mask_size, x, train, dmask, dtype=torch.float64):
    """The reference module in `dtype` on the GPU (float64: the oracle; float32 with TF32 off / bfloat16: PyTorch's own
    execution at that precision, the yardstick of the gradient tolerances)."""
    net = oracle_net(dim, mask_size).to(dtype).cuda()
    net.load_state_dict({k: v.to(dtype) if v.is_floating_point() else v for k, v in st.items()})
    net.train(train)
    xo = x.detach().to(dtype).clone().requires_grad_(True)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        out = net(xo.view(x.shape[0], -1, 1, 1)).squeeze(1).sigmoid()
        (out.double() * dmask.double()).sum().backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    return out, xo.grad, net


def _run(st, dim, mask_size, x, train, dmask, precision):
    net = build_mask_net(dim, mask_size).cuda()
    net.load_state_dict({k: v.clone() for k, v in st.items()}, strict=True)
    net.train(train)
    xin = x.detach().clone().requires_grad_(True)
    out = mask_head(net, xin, precision)
    (out * dmask).sum().backward()
    return out, xin.grad, net


def _inputs(O, dim, M, seed):
    x = t(synth.det_tensor((O, dim), seed, 1.0))
    dmask = t(synth.det_tensor((O, M, M), seed + 1, 1.0))
    return x, dmask


def _grads(net, dx):
    return [("d obj_vecs", dx)] + [("d " + k, p.grad) for k, p in net.named_parameters()]


def _check(net, dx, onet, odx, ynet, ydx, floor, factor, what):
    """Gradients within max(floor, factor x PyTorch's error at the same precision); running buffers within floor."""
    bad = {}
    for (k, g), (_, og), (_, yg) in zip(_grads(net, dx), _grads(onet, odx), _grads(ynet, ydx)):
        e, tol = rel_l2(g, og), max(floor, factor * rel_l2(yg, og))
        if e > tol:
            bad[k] = (e, tol)
    for (k, b), (_, c) in zip(net.named_buffers(), onet.named_buffers()):
        e = rel_l2(b.float(), c.float()) if b.is_floating_point() else float(int(b) != int(c))
        if e > (TOL_F32 if floor == TOL_F32 else TOL_TC_FWD):
            bad[k] = e
    assert not bad, "%s: %s" % (what, bad)


@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("O", [1, 7, CFG2_OBJS])
@pytest.mark.parametrize("mask_size", [1, 2, 4, 16])
def test_fp32_engine_matches_float64(mask_size, O, train):
    dim = 128
    st = _state(dim, mask_size, 10 + mask_size)
    x, dmask = _inputs(O, dim, mask_size, 100 + O)
    out, dx, net = _run(st, dim, mask_size, x, train, dmask, "fp32")
    ref, rdx, onet = _run_oracle(st, dim, mask_size, x, train, dmask)
    _, ydx, ynet = _run_oracle(st, dim, mask_size, x, train, dmask, torch.float32)
    assert out.dtype == torch.float32 and out.shape == (O, mask_size, mask_size)
    assert rel_l2(out, ref) < TOL_F32, rel_l2(out, ref)
    _check(net, dx, onet, rdx, ynet, ydx, TOL_F32, 3.0, "fp32 mask_size=%d O=%d train=%s" % (mask_size, O, train))


@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("O", [7, CFG2_OBJS])
@pytest.mark.parametrize("mask_size", [1, 4, 16])
def test_bf16_engine(mask_size, O, train):
    dim = 128
    st = _state(dim, mask_size, 20 + mask_size)
    x, dmask = _inputs(O, dim, mask_size, 200 + O)
    out, dx, net = _run(st, dim, mask_size, x.to(torch.bfloat16), train, dmask, "bf16")
    ref, rdx, onet = _run_oracle(st, dim, mask_size, x, train, dmask)
    _, ydx, ynet = _run_oracle(st, dim, mask_size, x, train, dmask, torch.bfloat16)
    assert out.dtype == torch.float32
    assert rel_l2(out, ref) < TOL_TC_FWD, rel_l2(out, ref)
    assert dx.dtype == torch.bfloat16
    _check(net, dx, onet, rdx, ynet, ydx, TOL_TC_BWD, 2.0, "bf16 mask_size=%d O=%d train=%s" % (mask_size, O, train))


@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
def test_fp16_forward(train):
    dim, M, O = 128, 16, CFG2_OBJS
    st = _state(dim, M, 30)
    x, dmask = _inputs(O, dim, M, 300)
    net = build_mask_net(dim, M).cuda()
    net.load_state_dict(st)
    net.train(train)
    with torch.no_grad():
        out = mask_head(net, x.half(), "fp16")
    ref, _, onet = _run_oracle(st, dim, M, x, train, dmask)
    assert rel_l2(out, ref) < TOL_TC_FWD, rel_l2(out, ref)
    for (k, b), (_, c) in zip(net.named_buffers(), onet.named_buffers()):
        if b.is_floating_point():
            assert rel_l2(b, c) < TOL_TC_FWD, k
    with pytest.raises(_lib.CsgError, match="inference-only"):
        mask_head(net, x.half().requires_grad_(True), "fp16")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
def test_empty_batch(precision, train):
    dim, M = 128, 4
    st = _state(dim, M, 40)
    net = build_mask_net(dim, M).cuda()
    net.load_state_dict(st)
    net.train(train)
    onet = oracle_net(dim, M)                   # torch's BatchNorm2d on an empty batch, on the CPU
    onet.load_state_dict(st)
    onet.train(train)
    x = torch.zeros((0, dim), device="cuda", requires_grad=True)
    out = mask_head(net, x, precision)
    ref = onet(torch.zeros((0, dim, 1, 1))).squeeze(1).sigmoid()
    assert out.shape == ref.shape == (0, M, M)
    out.sum().backward()
    assert x.grad is not None and x.grad.shape == (0, dim)
    for p in net.parameters():
        assert p.grad is not None and not p.grad.any()
    for (k, b), (_, c) in zip(net.named_buffers(), onet.named_buffers()):
        assert torch.equal(b.cpu(), c), k      # num_batches_tracked += 1 in training mode, running stats kept


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_deterministic(precision):
    dim, M, O = 128, 16, CFG2_OBJS
    st = _state(dim, M, 50)
    x, dmask = _inputs(O, dim, M, 500)
    runs = []
    for _ in range(2):
        out, dx, net = _run(st, dim, M, x, True, dmask, precision)
        runs.append([out, dx] + [p.grad for p in net.parameters()] + list(net.buffers()))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def _model_opt(mask_size):
    vocab = synth.Vocab(0)
    return vocab, argparse.Namespace(
        vocab={"attributes": {"objects": {str(i): i for i in range(vocab.num_obj_classes)}},
               "pred_idx_to_name": vocab.pred_names, "pred_name_to_idx": vocab.pred_ids},
        embedding_dim=128, gconv_dim=128, gconv_hidden_dim=512, gconv_pooling="avg", gconv_num_layers=5,
        mlp_normalization="none", mask_size=mask_size, learned_init="uniform")


def _reference_state(vocab, M):
    st = {k: torch.from_numpy(v) for k, v in synth.make_state(vocab, seed=3).items()}
    for i in range(5):
        st["gconvs.%d.predicates_transitive_weights" % i] = st["trans_candidates_weights"]
    st.update({"mask_net." + k: v for k, v in _state(128, M, 60).items()})
    return st


def test_model_loads_reference_state_and_masks_reach_the_gcn():
    """Sg2LayoutModel(mask_size=16) loads a reference state strictly; masks_to_layout(vecs, boxes,
    model.masks_from_vecs(obj_vecs)) backpropagates into the GCN, as the float64 oracle chain does."""
    from canonicalsg2im_b200.model import Sg2LayoutModel
    from canonicalsg2im_b200.layout import masks_to_layout
    from oracle import graph as ograph, layout as olayout
    M = 16
    vocab, opt = _model_opt(M)
    st = _reference_state(vocab, M)
    model = Sg2LayoutModel(opt).cuda()
    model.load_state_dict(st, strict=True)
    assert set(model.state_dict()) == set(st)
    # BatchNorm with the running buffers: batch statistics over the 8 rows of one graph are ill-conditioned (the GCN's
    # output rows are ReLU outputs, a channel that is zero for all but one object has a variance near 0 and an invstd
    # near 1/sqrt(eps), which multiplies any rounding of obj_vecs by ~300) -- the training-mode head is checked against
    # the reference above, on 7 and 2 200 rows
    model.eval()
    g = synth.make_graph(777, 8, 8, vocab, include_dummies=False, mask_size=M)
    O = len(g.objs)
    objs = torch.from_numpy(g.objs).view(1, O, -1)
    trips = torch.from_numpy(g.triplets).view(1, -1, 3)
    types = torch.zeros(trips.shape[:2], dtype=torch.int64)
    obj_vecs, boxes_pred, masks_pred = model(objs.cuda(), trips.cuda(), types.cuda())
    assert masks_pred.shape == (1, O, M, M)
    flat = obj_vecs.view(O, -1)
    masks = model.masks_from_vecs(flat)
    assert rel_l2(masks, masks_pred.view(O, M, M)) < 1e-6
    vecs = t(synth.det_tensor((O, 32), 7, 1.0))
    boxes = t(g.boxes)
    canvas = masks_to_layout(vecs, boxes, masks, 32)
    canvas.pow(2).sum().backward()

    # the oracle chain on the CPU: GCN (oracle/graph.py), reference mask net, masks_to_layout -- in float64, and in
    # float32 as the yardstick of the gradient tolerance (module docstring)
    def chain(dtype):
        sd = {k: v.to(dtype).requires_grad_(True) if v.is_floating_point() else v for k, v in st.items()}
        ov, _ = ograph.sg2layout_forward(sd, objs, trips, types, vocab.padding_id)
        onet = oracle_net(128, M).to(dtype)
        onet.load_state_dict({k[len("mask_net."):]: v.detach() for k, v in sd.items() if k.startswith("mask_net.")})
        onet.eval()
        omasks = onet(ov.view(O, -1, 1, 1)).squeeze(1).sigmoid()
        ocanvas = olayout.masks_to_layout(vecs.to(dtype).cpu(), boxes.to(dtype).cpu(), omasks, 32)
        ocanvas.pow(2).sum().backward()
        return sd, omasks, ocanvas

    sd, omasks, ocanvas = chain(torch.float64)
    sd32, _, _ = chain(torch.float32)
    assert rel_l2(masks, omasks) < TOL_F32
    assert rel_l2(canvas, ocanvas) < TOL_F32
    checked = 0
    for name, p in model.named_parameters():
        if name.startswith("gconvs.") and name in sd and sd[name].grad is not None:
            assert p.grad is not None, name
            e, tol = rel_l2(p.grad, sd[name].grad), max(1e-4, 3.0 * rel_l2(sd32[name].grad, sd[name].grad))
            assert e < tol, (name, e, tol)
            checked += 1
    assert checked >= 40


def _small_batch(vocab, M):
    g = synth.make_graph(777, 8, 8, vocab, include_dummies=False, mask_size=M)
    O = len(g.objs)
    objs = torch.from_numpy(g.objs).view(1, O, -1).cuda()
    trips = torch.from_numpy(g.triplets).view(1, -1, 3).cuda()
    return O, (objs, trips, torch.zeros(trips.shape[:2], dtype=torch.int64, device="cuda"))


def test_cached_mask_weight_copies_follow_the_optimizer(monkeypatch):
    """The mask head's cached 16-bit weight copies (Sg2LayoutModel.refresh_weight_copies) give bit-identical results to
    casting per call (CSG_WCOPIES=0), and FusedAdam, which rewrites the parameters through raw pointers, leaves no stale
    copy behind: without a refresh hook the next forward sees the new weights, with one the copies are rebuilt."""
    from canonicalsg2im_b200 import mask_head as mh, graph_tc
    from canonicalsg2im_b200.model import Sg2LayoutModel
    from canonicalsg2im_b200.optim import FusedAdam
    M = 4
    vocab, opt = _model_opt(M)
    model = Sg2LayoutModel(opt, precision="bf16").cuda()
    model.load_state_dict(_reference_state(vocab, M), strict=True)
    O, args = _small_batch(vocab, M)
    dm = t(synth.det_tensor((1, O, M, M), 91, 1.0))

    def run():
        for p in model.parameters():
            p.grad = None
        obj_vecs, boxes, masks = model(*args)
        (masks * dm).sum().backward()
        return masks.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}

    def both():
        model.eval()                  # the running buffers stay put, so the two runs see the same normalisation
        monkeypatch.setenv("CSG_WCOPIES", "1")
        a = run()
        monkeypatch.setenv("CSG_WCOPIES", "0")
        b = run()
        assert torch.equal(a[0], b[0])
        for n in a[1]:
            assert torch.equal(a[1][n], b[1][n]), n
        return a

    w0 = model.mask_net[2].weight
    graph_tc.invalidate_weight_copies()
    first = both()
    model.refresh_weight_copies()
    assert mh._WCOPIES[w0.data_ptr()]["versions"] is not None
    cached = both()
    assert torch.equal(first[0], cached[0])
    fopt = FusedAdam([p for p in model.parameters() if p.grad is not None], lr=1e-2)
    fopt.step()                       # no refresh hook: the mask head's copies must be stale now
    assert mh._WCOPIES[w0.data_ptr()]["versions"] is None
    after = both()
    assert not torch.equal(after[0], cached[0])
    fopt.post_step.append(model.refresh_weight_copies)
    fopt.step()
    assert mh._WCOPIES[w0.data_ptr()]["versions"] is not None
    both()


def test_tensor_core_model_matches_fp32_model():
    """Sg2LayoutModel(mask_size=16) at precision 'bf16' (forward + backward) and 'fp16' (forward) against the same model
    at 'fp32': obj_vecs and masks_pred within the forward contract 1e-2, every gradient within 2e-1 relative L2.  The
    gradients are those of a loss on the masks, so they reach the GCN through the four mask stages and then up to five
    GCN layers: the ReLU-flip error of DESIGN.md 4.1 (1e-1 for the GCN alone) compounds over both -- measured 1.6e-1
    for the embedding tables and layer 0, <= 1.5e-1 for the mask head (section 3.2, PyTorch's own bf16 alike).  Every
    kernel is deterministic, so the measured values are those of every run.  Eval mode, for the reason given in the
    end-to-end test."""
    from canonicalsg2im_b200.model import Sg2LayoutModel
    M = 16
    vocab, opt = _model_opt(M)
    st = _reference_state(vocab, M)
    O, args = _small_batch(vocab, M)
    dm = t(synth.det_tensor((1, O, M, M), 92, 1.0))
    res = {}
    for prec in ("fp32", "bf16"):
        model = Sg2LayoutModel(opt, precision=prec).cuda()
        model.load_state_dict(st, strict=True)
        model.eval()
        model.refresh_weight_copies()
        obj_vecs, boxes, masks = model(*args)
        assert masks.dtype == torch.float32 and masks.shape == (1, O, M, M)
        ((masks * dm).sum() + boxes.float().pow(2).sum()).backward()
        res[prec] = (obj_vecs.float(), masks, {n: p.grad for n, p in model.named_parameters() if p.grad is not None})
    f32, b16 = res["fp32"], res["bf16"]
    assert rel_l2(b16[0], f32[0]) < TOL_TC_FWD, rel_l2(b16[0], f32[0])
    assert rel_l2(b16[1], f32[1]) < TOL_TC_FWD, rel_l2(b16[1], f32[1])
    assert set(b16[2]) == set(f32[2])
    bad = {}
    for n, g in f32[2].items():
        e = rel_l2(b16[2][n], g)
        if e > 2e-1:
            bad[n] = e
    assert not bad, bad
    model = Sg2LayoutModel(opt, precision="fp16").cuda()
    model.load_state_dict(st, strict=True)
    model.eval()
    with torch.no_grad():
        _, _, masks16 = model(*args)
    assert rel_l2(masks16, f32[1]) < TOL_TC_FWD, rel_l2(masks16, f32[1])
