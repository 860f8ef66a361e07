"""The training step and the inference pipeline with the mask head (mask_size > 0): the canvas is composited from the
PREDICTED masks on the GT boxes (sg2im meta_models.py:48), so its gradient reaches the generator's embedding, the mask
head and the GCN.

Tolerances.  Against the float64 oracle step (oracle/step.CpuStep's pieces plus the reference-structured mask net and
per-image masks_to_layout): the loss within 1e-5 of its scale, masks_pred and canvas within 1e-5 relative L2; every
gradient within max(1e-5, 4 x the oracle's own float32 error) in relative L2, the law of DESIGN.md section 3.2 (ReLU
flips under any change of arithmetic) with the factor 4 because the last GCN layer's net2 bias, the sum of the mask
head's d obj_vecs over all objects, measured 3.1 x; BatchNorm running buffers within 1e-5.  The bf16 step against the
fp32 step: 6e-1 relative L2 (measured up to 0.55, on the GCN's parameters: the canvas gradient reaches them through
four bf16 mask stages and then up to five GCN layers, and the ReLU-flip error of both compounds, DESIGN.md 3.2), masks_pred
within 5e-2.  Graph replay, the 16-bit canvas and the bucket layout are checked bit for bit."""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from canonicalsg2im_b200 import synth
from canonicalsg2im_b200.pipeline import HostBatch, SgToLayoutInference, SgToLayoutStep
from tests.util import rel_err, t

pytestmark = pytest.mark.gpu
M = 16


def rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / max(b.norm().item(), 1e-12)).item()


def _grad(shape, seed, dtype=torch.float32):
    return (torch.randn(shape, device="cuda", generator=torch.Generator("cuda").manual_seed(seed)) * 1e-3).to(dtype)


def _eager(step, d, G):
    """One eager forward + backward of ``step`` (no optimizer step): (loss, canvas, masks_pred, named grads)."""
    res = step.canonicalize(d)
    canvas, loss = step.forward(d, res)
    torch.autograd.backward([canvas, loss], [G, None])
    torch.cuda.synchronize()
    return loss.detach(), canvas.detach(), step.last_masks, step.named_grads()


# ------------------------------------------------------------------------------------------------- oracle step
def _oracle_net(dim, mask_size):
    layers, cur = [], 1
    while cur < mask_size:
        layers += [nn.Upsample(scale_factor=2, mode="nearest"), nn.BatchNorm2d(dim),
                   nn.Conv2d(dim, dim, kernel_size=3, padding=1), nn.ReLU()]
        cur *= 2
    layers.append(nn.Conv2d(dim, 1, kernel_size=1))
    return nn.Sequential(*layers)


def _oracle_step(vocab, graphs, uni, G, dtype):
    """The reference's step in `dtype` on the CPU: collate, Sg2LayoutModel, mask_net on every row of the (unpadded)
    batch, per-image masks_to_layout of the generator embedding on the GT boxes with the predicted masks."""
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
    masks.retain_grad()
    layout_vecs = ograph.attribute_embeddings(state, "generator.attribute_embedding.", objs)
    canvas = torch.cat([olayout.masks_to_layout(layout_vecs[b], boxes[b].to(dtype), masks.view(B, O, M, M)[b], 64, 64)
                        for b in range(B)], 0)
    loss, _ = bbox_pred_loss(boxes_pred, boxes.to(dtype), objs, 10.0)
    torch.autograd.backward([canvas, loss], [G.cpu().to(dtype), None])
    grads = {("model." + k if not k.startswith("generator.") else "layout_embedding." + k[len("generator.attribute_embedding."):]): v.grad
             for k, v in state.items() if v.grad is not None}
    grads.update({"model.mask_net." + k: p.grad for k, p in net.named_parameters()})
    return loss.detach(), canvas.detach(), masks.detach(), grads, dict(net.named_buffers())


def test_fp32_step_matches_oracle():
    vocab = synth.Vocab(42)
    graphs = synth.make_graphs(8, 700, 10, 10, vocab, include_dummies=True)      # equal sizes: no padded rows
    hb = HostBatch(graphs, seed=0)
    G = _grad((8, 128, 64, 64), 5)
    step = SgToLayoutStep(vocab, "cuda", precision="fp32", seed=0, mask_size=M)
    loss, canvas, masks, grads = _eager(step, hb.to_device("cuda"), G)
    uni = synth.det_uniform(int(hb.tri_off[-1]), 13)
    o64 = _oracle_step(vocab, graphs, uni, G, torch.float64)
    o32 = _oracle_step(vocab, graphs, uni, G, torch.float32)
    assert rel_err(loss, o64[0]) <= 1e-5
    assert rel_l2(masks, o64[2]) <= 1e-5        # relative L2, as test_gpu_mask_head's masks
    assert rel_l2(canvas, o64[1]) <= 1e-5
    bad = {}
    for k, g64 in o64[3].items():
        e, tol = rel_l2(grads[k], g64), max(1e-5, 4 * rel_l2(o32[3][k], g64))
        if e > tol:
            bad[k] = (e, tol)
    assert not bad, bad
    assert set(grads) <= set(o64[3]) | {"model.converse_candidates_weights"}
    for k, b in step.model.mask_net.named_buffers():
        ref = o64[4][k]
        if b.is_floating_point():
            assert rel_err(b, ref) <= 1e-5, k
        else:
            assert int(b) == int(ref), k


def test_bf16_step_matches_fp32_step():
    vocab = synth.Vocab(42)
    hb = HostBatch(synth.make_graphs(32, 710, 3, 30, vocab, include_dummies=True), seed=1)
    G = _grad((32, 128, 64, 64), 6)
    out = {}
    for prec in ("fp32", "bf16"):
        step = SgToLayoutStep(vocab, "cuda", precision=prec, seed=0, mask_size=M)
        out[prec] = _eager(step, hb.to_device("cuda"), G)
    errs = {k: rel_l2(g, out["fp32"][3][k]) for k, g in out["bf16"][3].items()}
    bad = {k: e for k, e in errs.items() if e > 6e-1}
    assert not bad, sorted(errs.items(), key=lambda x: -x[1])
    # masks_pred: the bf16 GCN's forward error (1e-2) carried through the four stages of the head (measured 2.2e-2)
    assert rel_l2(out["bf16"][2], out["fp32"][2]) <= 5e-2


def _state_after(step):
    step.finish()
    torch.cuda.synchronize()
    params = [p.detach().clone() for p in step.opt.params]
    adam = [(step.opt.state[p]["exp_avg"].clone(), step.opt.state[p]["exp_avg_sq"].clone()) for p in step.opt.params
            if p in step.opt.state]
    bufs = [b.detach().clone() for b in step.model.mask_net.buffers()]
    return params, adam, bufs


def test_graph_replay_equals_eager_steps():
    """Four bf16 steps on two alternating batch buffers with Adam and the refresh of the 16-bit weight copies between
    them: parameters, Adam state and BatchNorm buffers equal bit for bit with and without CUDA-graph replay."""
    vocab = synth.Vocab(42)
    hbs = [HostBatch(synth.make_graphs(12, 720 + i, 3, 20, vocab, include_dummies=True), seed=i) for i in range(2)]
    G = _grad((12, 128, 64, 64), 7)
    res = []
    for use_graph in (False, True):
        step = SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0, use_graph=use_graph, mask_size=M)
        ds = [hb.to_device("cuda") for hb in hbs]
        losses = [float(step.step(ds[it & 1], G, prefetch=ds[(it + 1) & 1])[0]) for it in range(4)]
        if use_graph:
            assert step.graph_replays >= 2
        res.append((losses, _state_after(step)))
    assert res[0][0] == res[1][0]
    for a, b in zip(res[0][1], res[1][1]):
        for x, y in zip(a, b):
            if isinstance(x, tuple):
                assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])
            else:
                assert torch.equal(x, y)


@pytest.mark.parametrize("use_graph", [pytest.param(False, id="eager"), pytest.param(True, id="graph")])
def test_bf16_canvas_with_predicted_masks(use_graph):
    vocab = synth.Vocab(42)
    hb = HostBatch(synth.make_graphs(16, 730, 3, 30, vocab, include_dummies=True), seed=2)
    g16 = _grad((16, 128, 64, 64), 8, torch.bfloat16)
    grads = {}
    for dt in (torch.bfloat16, torch.float32):
        step = SgToLayoutStep(vocab, "cuda", seed=0, use_graph=use_graph, canvas_dtype=dt, mask_size=M)
        d = hb.to_device("cuda")
        G = g16 if dt == torch.bfloat16 else g16.float()
        if use_graph:
            step.step(d, G)
            step.step(d, G)
            step.finish()
            assert step.graph_replays == 1
            grads[dt] = [g.detach().clone() for g in next(iter(step._graphs.values()))["grads"]]
        else:
            grads[dt] = [g.detach().clone() for g in _eager(step, d, G)[3].values()]
    assert len(grads[torch.bfloat16]) == len(grads[torch.float32]) > 0
    for i, (a, b) in enumerate(zip(grads[torch.bfloat16], grads[torch.float32])):
        assert torch.equal(a, b), i


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_inference_with_predicted_masks(precision):
    from canonicalsg2im_b200.layout import layout_batched
    sizes = list(synth.CLEVR_ATTR_SIZES)
    vocab = synth.Vocab(0, num_attributes=4)
    graphs = synth.make_graphs(4, 4400, 32, 64, vocab, include_dummies=True, box_mode="clevr", mask_size=16)
    for g in graphs:
        for k, n in enumerate(sizes):
            g.objs[:-1, k] = 1 + (g.objs[:-1, k] - 1) % (n - 1)
    hb = HostBatch(graphs, seed=4, with_geometry=True, num_uniforms=sum(4 * len(g.objs) ** 2 for g in graphs))
    inf = SgToLayoutInference(vocab, "cuda", precision=precision, H=128, W=128, embedding_dim=32, attr_sizes=sizes,
                              mask_size=M)
    d = hb.to_device("cuda")
    d.pop("masks")
    with torch.no_grad():
        canvas, boxes_pred, _ = inf.step(d)
        res = inf.build_graph(d)
        obj_vecs, _ = inf.model.forward_ragged(d["objs"], res.triplets, res.triplet_type, res.tri_off, d["obj_off"])
        dummy = (d["objs"][:, :1] == 0)
        boxes = torch.where(dummy, torch.full_like(boxes_pred, -1.0), boxes_pred.float())
        ref = layout_batched(inf.layout_embedding(d["objs"]), boxes, d["obj_off"], 128, 128,
                             masks=inf.model.masks_from_vecs(obj_vecs), test_mode=True)
    assert torch.equal(canvas, ref)
    assert canvas.abs().sum() > 0
    nbt = [int(b) for k, b in inf.model.mask_net.named_buffers() if k.endswith("num_batches_tracked")]
    assert nbt and all(n == 0 for n in nbt), "eval mode must leave the running buffers alone"


def test_every_parameter_in_one_bucket(tmp_path):
    import torch.distributed as dist
    vocab = synth.Vocab(42)
    hb = HostBatch(synth.make_graphs(12, 740, 3, 20, vocab, include_dummies=True), seed=3)
    G = _grad((12, 128, 64, 64), 9)
    ref = _eager(SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0, mask_size=M), hb.to_device("cuda"), G)[3]
    dist.init_process_group("nccl", store=dist.FileStore(os.path.join(str(tmp_path), "store"), 1), rank=0, world_size=1)
    try:
        step = SgToLayoutStep(vocab, "cuda", precision="bf16", seed=0, mask_size=M, distributed=True)
        trainable = [p for p in step.opt.params]
        counts = {id(p): 0 for p in trainable}
        for params in step.reducer.params:
            for p in params:
                assert id(p) in counts
                counts[id(p)] += 1
        assert all(c == 1 for c in counts.values())
        assert any(p is step.model.mask_net[2].weight for p in step.reducer.params[0])
        step.backward(hb.to_device("cuda"), G)
        torch.cuda.synchronize()
        got = step.named_grads()
        assert set(got) == set(ref)
        for k in ref:
            assert torch.equal(got[k], ref[k]), k
    finally:
        dist.destroy_process_group()
