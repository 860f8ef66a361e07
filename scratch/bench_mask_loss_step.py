"""The training step on GT masks (SgToLayoutStep(mask_size=16, gt_masks=True)) on the GPU.

1. Mask loss kernel alone (csg_mask_loss, loss + dpred in one pass) at the cfg2 predicted-mask size (2 349 objects x
   16 x 16 = 601 k elements), fp32 and int64 targets: CUDA events, L2 flushed (a 256 MB write) before every timed call.
2. Whole step, bf16 GCN, CUDA-graph replay, cfg2 batch (bench.workload_graphs(128, 0), with the GT masks
   synth.make_graphs gives the same graphs at mask_size = 16): mask_size = 0, predicted masks (mask_size = 16) and GT
   masks + mask loss (mask_size = 16, gt_masks=True), alternated block by block in one run (median ms per step).

The card's name, power limit and SM clock limit are read in the same run.

Usage: python scratch/bench_mask_loss_step.py [--reps 50] [--steps 20] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from canonicalsg2im_b200 import synth, _lib  # noqa: E402
from canonicalsg2im_b200.ops import lib, ptr, workspace, _stream  # noqa: E402


def cfg2_graphs():
    import bench
    vocab, graphs = bench.workload_graphs(128, 0)
    with_masks = synth.make_graphs(128, 1000, 3, 30, vocab, include_dummies=True, mask_size=16)
    for g, h in zip(graphs, with_masks):      # the same seeded graphs, plus their GT masks
        assert np.array_equal(g.objs, h.objs) and np.array_equal(g.boxes, h.boxes)
    return vocab, with_masks


def loss_kernel(args):
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    L = lib()
    n = 2349 * 16 * 16
    g = torch.Generator("cuda").manual_seed(0)
    pred = torch.sigmoid(torch.randn(n, device="cuda", generator=g))
    t64 = (torch.rand(n, device="cuda", generator=g) < 0.6).to(torch.int64)
    targets = {"fp32 target": t64.float(), "int64 target": t64}
    loss, dpred = torch.empty(1, device="cuda"), torch.empty_like(pred)
    ws = workspace(L.csg_mask_loss_workspace(n), "cuda")

    def call(t):
        _lib.check(L.csg_mask_loss(ptr(pred), ptr(t), int(t.dtype == torch.int64), n, 1.0, ptr(loss), ptr(dpred),
                                   ptr(ws), ws.numel(), _stream()))

    res = {k: [] for k in targets}
    for t in targets.values():
        call(t); call(t)
    for _ in range(args.reps):
        for k, t in targets.items():
            flush_buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(t); e1.record()
            torch.cuda.synchronize()
            res[k].append(e0.elapsed_time(e1) * 1e3)
    out = {}
    for k, t in targets.items():
        nbytes = n * (4 + t.element_size() + 4)            # read pred and target, write dpred
        us = float(np.median(res[k]))
        out[k] = {"us": round(us, 2), "bytes": nbytes, "GB/s": round(nbytes / us / 1e3, 1)}
        print("mask loss kernel, %d elements, %-13s %s" % (n, k, out[k]))
    return out


def _step_setup(vocab, graphs, mask_size, gt_masks):
    from canonicalsg2im_b200.pipeline import HostBatch, SgToLayoutStep
    step = SgToLayoutStep(vocab, torch.device("cuda"), precision="bf16", seed=0, use_graph=True, mask_size=mask_size,
                          gt_masks=gt_masks)
    hbs = [HostBatch(graphs, seed=s, with_masks=gt_masks) for s in (0, 1)]
    ds = [hb.to_device("cuda") for hb in hbs]
    G = torch.randn((128, 128, 64, 64), device="cuda", generator=torch.Generator("cuda").manual_seed(1)) * 1e-3
    return step, ds, G


def whole_step(args):
    vocab, graphs = cfg2_graphs()
    variants = {"mask_size=0": (0, False), "predicted masks (mask_size=16)": (16, False),
                "GT masks + mask loss (mask_size=16, gt_masks)": (16, True)}
    runs = {k: _step_setup(vocab, graphs, *v) for k, v in variants.items()}
    it = {k: 0 for k in runs}

    def block(k, n):
        step, ds, G = runs[k]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            i = it[k]
            step.step(ds[i & 1], G, prefetch=ds[(i + 1) & 1])
            it[k] += 1
        step.finish()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    for k in runs:
        block(k, 6)                           # eager step, two captures, replays
    res = {k: [] for k in runs}
    for _ in range(5):
        for k in runs:
            res[k].append(block(k, args.steps))
    out = {k + " ms/step": round(float(np.median(v)), 3) for k, v in res.items()}
    out["spread"] = {k: [round(x, 3) for x in v] for k, v in res.items()}
    out["graph_replays"] = {k: runs[k][0].graph_replays for k in runs}
    print("whole step (bf16, graph replay, cfg2):", json.dumps(out, indent=1))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", torch.cuda.get_device_name(0), "|", smi)
    report = {"gpu": smi, "reps": args.reps, "l2_flush": "256 MB write before every timed kernel call"}
    report["loss_kernel"] = loss_kernel(args)
    report["step"] = whole_step(args)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_mask_loss_step.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
