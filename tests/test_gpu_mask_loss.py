"""The mask term of the generator loss on GT masks (csg_mask_loss, model.mask_pred_loss) and the training step that
uses it (SgToLayoutStep(mask_size=M, gt_masks=True)): the canvas is composited from the GT masks, and the mask head is
trained by weight * BCE(masks_pred, masks_gt).

Tolerances.  The kernel against torch's BCE + autograd evaluated in float64 on the same fp32 inputs: loss within 1e-5
relative, dpred within 1e-5 of its max-norm; at the saturated tails, and pushed through the mask head's sigmoid
backward, bitwise torch's fp32 CPU autograd.  The fp32 step against the float64 oracle step: loss, masks_pred and canvas
within 1e-5, every gradient within max(1e-5, 4 x the oracle's own fp32 error) in relative L2 (the law of DESIGN.md
section 3.2), BatchNorm buffers within 1e-5.  The bf16 step against the fp32 step: BF16_GRAD_TOL = 3e-1 relative L2 on
the gradients (measured up to 0.18), masks_pred within 5e-2 (measured 2.2e-2), loss within 1e-3 (measured 2.6e-4).
Zero weight, graph replay and the 16-bit canvas are checked bit for bit."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from canonicalsg2im_b200 import _lib, synth
from canonicalsg2im_b200.model import mask_pred_loss
from canonicalsg2im_b200.ops import lib, ptr, workspace, _stream
from canonicalsg2im_b200.pipeline import HostBatch, SgToLayoutStep
from tests.mask_loss_ref import mask_pred_loss as ref_mask_pred_loss
from tests.test_gpu_mask_step import _eager, _grad, _oracle_net, _state_after, rel_l2
from tests.util import rel_err

pytestmark = pytest.mark.gpu
M = 16
NO_CFG2 = 2349                     # objects of the cfg2 batch (bench.workload_graphs(128, 0))
# bf16 step against the fp32 step, relative L2 over every gradient: measured up to 0.18 on a B200 (the first stage's
# conv bias mask_net.2.bias, a sum over every pixel of every object; two batches of 32 graphs), DESIGN.md section 3.2
BF16_GRAD_TOL = 3e-1


def _loss_and_grad(pred, target, weight=1.0):
    x = pred.detach().clone().requires_grad_()
    loss = mask_pred_loss(x, target, weight)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), x.grad


# ------------------------------------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("target", ["int64", "soft"])
def test_kernel_matches_torch_float64(target):
    g = torch.Generator("cuda").manual_seed(11)
    pred = torch.sigmoid(2 * torch.randn((NO_CFG2, M, M), device="cuda", generator=g))
    if target == "int64":
        tgt = (torch.rand(pred.shape, device="cuda", generator=g) < 0.6).to(torch.int64)
    else:
        tgt = torch.rand(pred.shape, device="cuda", generator=g)
    loss, dpred = _loss_and_grad(pred, tgt, 2.5)
    x = pred.double().cpu().requires_grad_()
    ref = ref_mask_pred_loss(x, tgt.cpu(), 2.5)
    ref.backward()
    assert rel_err(loss, ref.detach()) <= 1e-5
    assert rel_err(dpred, x.grad) <= 1e-5


def _sigmoid_bwd(dy, y):
    """The mask head's backward (csg_head_bwd_ex with the sigmoid folded in) on a 1x1 head of weight 1 over a constant
    input: dh[:, k] = dy * sigmoid' = dy y (1 - y), as the head computes it for d masks_pred."""
    L, R, K = lib(), y.numel(), 2
    h, w = torch.ones((R, K), device="cuda"), torch.ones((1, K), device="cuda")
    dh, dw, db = torch.empty((R, K), device="cuda"), torch.empty((1, K), device="cuda"), torch.empty(1, device="cuda")
    ws = workspace(L.csg_head_bwd_ex_workspace(R, K, 1), "cuda")
    _lib.check(L.csg_head_bwd_ex(ptr(dy), ptr(y), ptr(h), K, 0, ptr(w), R, K, 1, ptr(dh), K, 0, 0, ptr(dw), ptr(db),
                                 ptr(ws), ws.numel(), _stream()), "csg_head_bwd_ex")
    torch.cuda.synchronize()
    return dh[:, 0]


def test_saturated_tails_equal_torch_fp32():
    tails = [0.0, 1.0, 1e-13, 1.0 - 2.0 ** -24]
    p = torch.tensor(tails * 2, dtype=torch.float32)
    t = torch.tensor([0.0] * 4 + [1.0] * 4)
    loss, dp = _loss_and_grad(p.cuda(), t.cuda())
    x = p.clone().requires_grad_()
    ref = F.binary_cross_entropy(x, t)
    ref.backward()
    dz_ref = torch.ops.aten.sigmoid_backward(x.grad, p)          # what autograd of sigmoid -> BCE computes
    assert torch.equal(dp.cpu(), x.grad)
    dz = _sigmoid_bwd(dp, p.cuda()).cpu()
    assert torch.equal(dz, dz_ref), (dz, dz_ref)
    assert (dz[p == 1.0] == 0).all() and (dz[p == 0.0] == 0).all()
    assert rel_err(loss, ref.detach()) <= 1e-6


def test_int64_target_equals_float_target_and_is_deterministic():
    g = torch.Generator("cuda").manual_seed(12)
    pred = torch.sigmoid(2 * torch.randn((NO_CFG2, M, M), device="cuda", generator=g))
    t64 = (torch.rand(pred.shape, device="cuda", generator=g) < 0.6).to(torch.int64)
    a = _loss_and_grad(pred, t64, 0.7)
    b = _loss_and_grad(pred, t64.float(), 0.7)
    c = _loss_and_grad(pred, t64.bool(), 0.7)
    d = _loss_and_grad(pred, t64, 0.7)
    for other in (b, c, d):
        assert torch.equal(a[0], other[0]) and torch.equal(a[1], other[1])


def test_empty_nan_and_shape_errors():
    loss, dpred = _loss_and_grad(torch.empty((0, M, M), device="cuda"), torch.empty((0, M, M), device="cuda"))
    assert torch.isnan(loss) and dpred.shape == (0, M, M)
    p = torch.full((3, M, M), 0.5, device="cuda")
    with pytest.raises(ValueError):
        mask_pred_loss(p, torch.zeros((3, M, M + 1), device="cuda"))
    with pytest.raises(ValueError):
        mask_pred_loss(p, torch.zeros((3 * M, M), device="cuda"))
    # padded [B, O, M, M] is the ragged batch's loss
    g = torch.Generator("cuda").manual_seed(13)
    pp = torch.rand((2, 5, M, M), device="cuda", generator=g)
    tt = (torch.rand(pp.shape, device="cuda", generator=g) < 0.5).to(torch.int64)
    a, b = _loss_and_grad(pp, tt), _loss_and_grad(pp.view(10, M, M), tt.view(10, M, M))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(10, M, M), b[1])


def test_nan_poisons_loss_and_own_element():
    p = torch.full((4, M, M), 0.25, device="cuda")
    p[1, 2, 3] = float("nan")
    loss, dpred = _loss_and_grad(p, torch.zeros_like(p))
    assert torch.isnan(loss)
    bad = torch.isnan(dpred)
    assert bad.sum() == 1 and bad[1, 2, 3]


# --------------------------------------------------------------------------------------------------------- step
def _gt_graphs(n, seed, lo, hi):
    return synth.make_graphs(n, seed, lo, hi, synth.Vocab(42), include_dummies=True, mask_size=M)


def _oracle_step_gt(vocab, graphs, uni, G, dtype, weight):
    """The reference's step in `dtype` on the CPU for a dataset with GT masks: collate, Sg2LayoutModel, mask_net on
    every row, per-image masks_to_layout of the generator embedding on the GT boxes with the GT masks, and the loss
    box term + weight * BCE(masks_pred, masks_gt)."""
    from oracle import graph as ograph, layout as olayout
    from oracle.step import CpuStep, bbox_pred_loss, collate
    st = synth.make_state(vocab, seed=0)
    tri = np.triu(st["converse_candidates_weights"])
    step = CpuStep(vocab, st, (tri + tri.T).astype(np.float64), synth.make_layout_state(vocab, 128, seed=0))
    tri_off = np.concatenate([[0], np.cumsum([len(g.triplets) for g in graphs])])
    objs, boxes, trips, types = collate(vocab, graphs, step.canonicalize(graphs, uni, tri_off))
    state = {k: v.detach().to(dtype).requires_grad_(v.requires_grad) for k, v in step.state.items()}
    net = _oracle_net(128, M).to(dtype)
    net.load_state_dict({k[len("mask_net."):]: torch.from_numpy(np.asarray(v)) for k, v in
                         synth.make_mask_state(128, M, seed=0).items()})
    net.train()
    obj_vecs, boxes_pred = ograph.sg2layout_forward(state, objs, trips, types, vocab.padding_id)
    B, O = objs.shape[0], objs.shape[1]
    masks = net(obj_vecs.reshape(B * O, -1, 1, 1)).squeeze(1).sigmoid()
    gt = torch.from_numpy(np.stack([g.masks for g in graphs])).to(dtype)          # equal sizes: no padded rows
    layout_vecs = ograph.attribute_embeddings(state, "generator.attribute_embedding.", objs)
    canvas = torch.cat([olayout.masks_to_layout(layout_vecs[b], boxes[b].to(dtype), gt[b], 64, 64) for b in range(B)], 0)
    loss = bbox_pred_loss(boxes_pred, boxes.to(dtype), objs, 10.0)[0] + ref_mask_pred_loss(masks, gt.view(B * O, M, M),
                                                                                           weight)
    torch.autograd.backward([canvas, loss], [G.cpu().to(dtype), None])
    grads = {("model." + k if not k.startswith("generator.") else "layout_embedding." + k[len("generator.attribute_embedding."):]): v.grad
             for k, v in state.items() if v.grad is not None}
    grads.update({"model.mask_net." + k: p.grad for k, p in net.named_parameters()})
    return loss.detach(), canvas.detach(), masks.detach(), grads, dict(net.named_buffers())


def test_fp32_step_matches_oracle():
    vocab = synth.Vocab(42)
    graphs = _gt_graphs(8, 700, 10, 10)
    hb = HostBatch(graphs, seed=0, with_masks=True)
    G = _grad((8, 128, 64, 64), 5)
    step = SgToLayoutStep(vocab, "cuda", precision="fp32", seed=0, mask_size=M, gt_masks=True, mask_loss_weight=1.0)
    loss, canvas, masks, grads = _eager(step, hb.to_device("cuda"), G)
    uni = synth.det_uniform(int(hb.tri_off[-1]), 13)
    o64 = _oracle_step_gt(vocab, graphs, uni, G, torch.float64, 1.0)
    o32 = _oracle_step_gt(vocab, graphs, uni, G, torch.float32, 1.0)
    assert rel_err(loss, o64[0]) <= 1e-5
    assert rel_l2(masks, o64[2]) <= 1e-5
    assert rel_l2(canvas, o64[1]) <= 1e-5
    bad = {}
    for k, g64 in o64[3].items():
        e, tol = rel_l2(grads[k], g64), max(1e-5, 4 * rel_l2(o32[3][k], g64))
        if e > tol:
            bad[k] = (e, tol)
    assert not bad, bad
    assert any(k.startswith("model.mask_net.") for k in grads)
    assert set(grads) <= set(o64[3]) | {"model.converse_candidates_weights"}
    for k, b in step.model.mask_net.named_buffers():
        ref = o64[4][k]
        if b.is_floating_point():
            assert rel_err(b, ref) <= 1e-5, k
        else:
            assert int(b) == int(ref), k


def test_zero_weight_leaves_head_without_gradient():
    vocab = synth.Vocab(42)
    hb = HostBatch(_gt_graphs(16, 760, 3, 30), seed=4, with_masks=True)
    G = _grad((16, 128, 64, 64), 10)
    gt = SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0, mask_size=M, gt_masks=True, mask_loss_weight=0.0)
    base = SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0)
    a = _eager(gt, hb.to_device("cuda"), G)
    b = _eager(base, hb.to_device("cuda"), G)
    assert not any(k.startswith("model.mask_net.") for k in a[3])
    assert all(p.grad is None for p in gt.model.mask_net.parameters())
    gcn = [k for k in b[3] if k.startswith("model.")]
    assert gcn and set(gcn) == {k for k in a[3] if k.startswith("model.")}
    for k in gcn:
        assert torch.equal(a[3][k], b[3][k]), k
    assert torch.equal(a[0], b[0])                       # the loss is the box term alone
    nbt = [int(x) for k, x in gt.model.mask_net.named_buffers() if k.endswith("num_batches_tracked")]
    assert nbt and all(n == 1 for n in nbt), "the head's forward still updates the BatchNorm buffers"


def test_bf16_step_matches_fp32_step():
    vocab = synth.Vocab(42)
    hb = HostBatch(_gt_graphs(32, 710, 3, 30), seed=1, with_masks=True)
    G = _grad((32, 128, 64, 64), 6)
    out = {}
    for prec in ("fp32", "bf16"):
        step = SgToLayoutStep(vocab, "cuda", precision=prec, seed=0, mask_size=M, gt_masks=True)
        out[prec] = _eager(step, hb.to_device("cuda"), G)
    assert set(out["bf16"][3]) == set(out["fp32"][3])
    errs = {k: rel_l2(g, out["fp32"][3][k]) for k, g in out["bf16"][3].items()}
    bad = {k: e for k, e in errs.items() if e > BF16_GRAD_TOL}
    assert not bad, sorted(errs.items(), key=lambda x: -x[1])
    assert rel_l2(out["bf16"][2], out["fp32"][2]) <= 5e-2
    assert rel_err(out["bf16"][0], out["fp32"][0]) <= 1e-3


def test_graph_replay_equals_eager_steps():
    """Four bf16 steps on two alternating batch buffers: parameters, Adam state and BatchNorm buffers equal bit for bit
    with and without CUDA-graph replay.  The graph key carries the masks buffer's address."""
    vocab = synth.Vocab(42)
    hbs = [HostBatch(_gt_graphs(12, 720 + i, 3, 20), seed=i, with_masks=True) for i in range(2)]
    G = _grad((12, 128, 64, 64), 7)
    res = []
    for use_graph in (False, True):
        step = SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0, use_graph=use_graph, mask_size=M,
                              gt_masks=True, mask_loss_weight=0.5)
        ds = [hb.to_device("cuda") for hb in hbs]
        losses = [float(step.step(ds[it & 1], G, prefetch=ds[(it + 1) & 1])[0]) for it in range(4)]
        if use_graph:
            assert step.graph_replays >= 2
            other = dict(ds[0], masks=ds[0]["masks"].clone())
            assert step._graph_key(ds[0], G, 100) != step._graph_key(other, G, 100)
        res.append((losses, _state_after(step)))
    assert res[0][0] == res[1][0]
    for a, b in zip(res[0][1], res[1][1]):
        for x, y in zip(a, b):
            if isinstance(x, tuple):
                assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])
            else:
                assert torch.equal(x, y)


@pytest.mark.parametrize("use_graph", [pytest.param(False, id="eager"), pytest.param(True, id="graph")])
def test_bf16_canvas_with_gt_masks(use_graph):
    vocab = synth.Vocab(42)
    hb = HostBatch(_gt_graphs(16, 730, 3, 30), seed=2, with_masks=True)
    g16 = _grad((16, 128, 64, 64), 8, torch.bfloat16)
    grads = {}
    for dt in (torch.bfloat16, torch.float32):
        step = SgToLayoutStep(vocab, "cuda", seed=0, use_graph=use_graph, canvas_dtype=dt, mask_size=M, gt_masks=True)
        d = hb.to_device("cuda")
        G = g16 if dt == torch.bfloat16 else g16.float()
        if use_graph:
            step.step(d, G)
            step.step(d, G)
            step.finish()
            assert step.graph_replays == 1
            grads[dt] = [g.detach().clone() for g in next(iter(step._graphs.values()))["grads"] if g is not None]
        else:
            grads[dt] = [g.detach().clone() for g in _eager(step, d, G)[3].values()]
    assert len(grads[torch.bfloat16]) == len(grads[torch.float32]) > 0
    for i, (a, b) in enumerate(zip(grads[torch.bfloat16], grads[torch.float32])):
        assert torch.equal(a, b), i


def test_missing_or_wrong_masks_raise():
    vocab = synth.Vocab(42)
    step = SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0, mask_size=M, gt_masks=True)
    G = _grad((4, 128, 64, 64), 9)
    with pytest.raises(ValueError, match="masks"):
        step.step(HostBatch(_gt_graphs(4, 770, 3, 10), seed=0).to_device("cuda"), G)
    d = HostBatch(synth.make_graphs(4, 770, 3, 10, vocab, include_dummies=True, mask_size=8), seed=0,
                  with_masks=True).to_device("cuda")
    with pytest.raises(ValueError, match="masks"):
        step.step(d, G)
