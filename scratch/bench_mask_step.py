"""The training step with predicted masks on the GPU.

1. Canvas backward wrt (vecs, float masks), boxes fixed: today's pair (csg_layout_bwd_vecs ring kernel +
   csg_layout_bwd_geom, one CTA per object) against csg_layout_bwd_vecs_masks (ring kernel + band-tiled d masks), and the
   ring kernel alone, with an fp32 and a bf16 gradient, on the cfg2 predicted-mask canvas (128 x 128 x 64 x 64, M = 16,
   the cfg2 boxes) and the cfg3 shape (16 x 128 x 256 x 256, float masks).  CUDA events, L2 flushed (a 256 MB write)
   before every timed pass, variants alternated in one process.  The outputs of the two paths are compared too.
2. Whole step, bf16 GCN, CUDA-graph replay, cfg2 batch (bench.workload_graphs(128, 0)): mask_size = 0 against
   mask_size = 16, alternated block by block in one run (median ms per step).
3. --profile: a run of its own under torch.profiler (eager steps, mask_size = 16): kernel time per step grouped into
   compositor forward / backward, mask-head-only kernels and the rest (GCN and the GEMMs of the mask head).

Usage: python scratch/bench_mask_step.py [--reps 20] [--steps 20] [--profile] [--out DIR]"""
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
from canonicalsg2im_b200.layout import _linspace  # noqa: E402
from canonicalsg2im_b200.ops import lib, ptr, workspace, _stream  # noqa: E402


def c(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def cfg2_canvas():
    sys.path.insert(0, ROOT)
    import bench
    vocab, graphs = bench.workload_graphs(128, 0)
    boxes = np.concatenate([g.boxes for g in graphs]).astype(np.float32)
    off = np.concatenate([[0], np.cumsum([len(g.boxes) for g in graphs])]).astype(np.int32)
    NO = len(boxes)
    vecs = synth.det_tensor((NO, 128), 91, 1.0)
    masks = synth.det_uniform(NO * 256, 92).reshape(NO, 16, 16).astype(np.float32)
    return c(vecs), c(boxes), c(masks), c(off), 64, 64


def cfg3_canvas():
    sys.path.insert(0, ROOT)
    import bench
    vecs, boxes, masks, off = bench.cfg3_objects(16)
    return c(vecs), c(boxes), c(masks), c(off), 256, 256


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", torch.cuda.get_device_name(0), "|", smi)
    report = {"gpu": smi, "reps": args.reps, "l2_flush": "256 MB write before every timed pass"}
    if args.profile:
        report["profile"] = profile(args)
    else:
        report["canvas_bwd"] = canvas_bwd(args)
        report["step"] = whole_step(args)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        name = "bench_mask_step_profile.json" if args.profile else "bench_mask_step.json"
        with open(os.path.join(args.out, name), "w") as f:
            json.dump(report, f, indent=1)


def canvas_bwd(args):
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    L = lib()
    out = {}
    for name, mk in (("cfg2 predicted masks 128x128x64x64 M16", cfg2_canvas), ("cfg3 masks 16x128x256x256 M16", cfg3_canvas)):
        v, b, m, off, H, W = mk()
        N, NO, D, M = off.numel() - 1, v.shape[0], v.shape[1], m.shape[1]
        lx, ly = _linspace(W, "cuda"), _linspace(H, "cuda")
        g32 = torch.randn((N, D, H, W), device="cuda", generator=torch.Generator("cuda").manual_seed(0))
        grads = {"fp32": g32, "bf16": g32.to(torch.bfloat16)}
        dv, dm = torch.empty((NO, D), device="cuda"), torch.empty_like(m)
        dv2, dm2, db = torch.empty_like(dv), torch.empty_like(m), torch.empty((NO, 4), device="cuda")
        ws_v = workspace(L.csg_layout_bwd_vecs_workspace(N, NO, D, H, W), "cuda")
        ws_g = workspace(L.csg_layout_bwd_geom_workspace(NO), "cuda")
        ws_n = workspace(L.csg_layout_bwd_vecs_masks_workspace(N, NO, D, H, W, M), "cuda")
        mo = int((off[1:] - off[:-1]).max())

        def ring(g):
            a = (ptr(g), ptr(b), ptr(m), ptr(off), ptr(lx), ptr(ly), ptr(dv2), N, NO, D, H, W, M, 0, mo)
            if g.dtype == torch.float32:
                _lib.check(L.csg_layout_bwd_vecs(*a, ptr(ws_v), ws_v.numel(), _stream()))
            else:
                _lib.check(L.csg_layout_bwd_vecs_bf16(*a, 0, ptr(ws_v), ws_v.numel(), _stream()))

        def old(g):
            ring(g)
            a = (ptr(g), ptr(v), ptr(b), ptr(m), ptr(off), ptr(lx), ptr(ly), ptr(db), ptr(dm2), N, NO, D, H, W, M, 0)
            if g.dtype == torch.float32:
                _lib.check(L.csg_layout_bwd_geom(*a, ptr(ws_g), ws_g.numel(), _stream()))
            else:
                _lib.check(L.csg_layout_bwd_geom_bf16(*a, 0, ptr(ws_g), ws_g.numel(), _stream()))

        def new(g):
            a = (ptr(g), ptr(v), ptr(b), ptr(m), ptr(off), ptr(lx), ptr(ly), ptr(dv), ptr(dm), N, NO, D, H, W, M, 0, mo)
            if g.dtype == torch.float32:
                _lib.check(L.csg_layout_bwd_vecs_masks(*a, ptr(ws_n), ws_n.numel(), _stream()))
            else:
                _lib.check(L.csg_layout_bwd_vecs_masks_bf16(*a, 0, ptr(ws_n), ws_n.numel(), _stream()))

        fns = {}
        for k, g in grads.items():
            fns["ring only (d vecs) " + k] = lambda g=g: ring(g)
            fns["ring + geom " + k] = lambda g=g: old(g)
            fns["ring + band d masks " + k] = lambda g=g: new(g)
        res = {k: [] for k in fns}
        for f in fns.values():
            f(); f()
        for _ in range(args.reps):
            for k, f in fns.items():
                flush_buf.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); f(); e1.record()
                torch.cuda.synchronize()
                res[k].append(e0.elapsed_time(e1) * 1e3)
        case = {k: round(float(np.median(x)), 1) for k, x in res.items()}
        for k, g in grads.items():
            old(g); new(g)
            torch.cuda.synchronize()
            fin = torch.isfinite(dm2)
            scale = max(dm2[fin].abs().max().item(), 1e-30)
            case["check " + k] = {"dvecs_equal": bool(torch.equal(dv, dv2)),
                                  "dmasks_max_rel": (dm - dm2)[fin].abs().max().item() / scale}
        for k, x in case.items():
            print("%-40s %-28s %s" % (name, k, x))
        out[name] = case
        del fns, grads, g32
        torch.cuda.empty_cache()
    return out


def _step_setup(mask_size, use_graph=True, precision="bf16"):
    import bench
    from canonicalsg2im_b200.pipeline import HostBatch, SgToLayoutStep
    vocab, graphs = bench.workload_graphs(128, 0)
    step = SgToLayoutStep(vocab, torch.device("cuda"), precision=precision, seed=0, use_graph=use_graph,
                          mask_size=mask_size)
    hbs = [HostBatch(graphs, seed=0), HostBatch(graphs, seed=1)]
    ds = [hb.to_device("cuda") for hb in hbs]
    G = torch.randn((128, 128, 64, 64), device="cuda", generator=torch.Generator("cuda").manual_seed(1)) * 1e-3
    return step, ds, G


def whole_step(args):
    runs = {ms: _step_setup(ms) for ms in (0, 16)}
    it = {ms: 0 for ms in runs}

    def block(ms, n):
        step, ds, G = runs[ms]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            i = it[ms]
            step.step(ds[i & 1], G, prefetch=ds[(i + 1) & 1])
            it[ms] += 1
        step.finish()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    for ms in runs:
        block(ms, 6)                          # eager step, two captures, replays
    res = {ms: [] for ms in runs}
    for _ in range(5):
        for ms in runs:
            res[ms].append(block(ms, args.steps))
    out = {"mask_size=%d ms/step" % ms: round(float(np.median(v)), 3) for ms, v in res.items()}
    out["spread"] = {"mask_size=%d" % ms: [round(x, 3) for x in v] for ms, v in res.items()}
    out["graph_replays"] = {"mask_size=%d" % ms: runs[ms][0].graph_replays for ms in runs}
    print("whole step (bf16, graph replay, cfg2):", out)
    return out


def profile(args):
    from torch.profiler import ProfilerActivity, profile as tprof
    step, ds, G = _step_setup(16, use_graph=False)
    for i in range(3):
        step.step(ds[i & 1], G)
    torch.cuda.synchronize()
    n = 5
    with tprof(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            step.step(ds[i & 1], G)
        torch.cuda.synchronize()
    groups = {"compositor fwd": ("layout_fwd",),
              "compositor bwd": ("layout_bwd", "layout_tables", "dmasks", "geom"),
              "mask head (BN, patches, 1x1 head, casts)": ("mask_bn", "mask_patch", "patch_kernel", "bn_", "head_")}
    tot = {k: 0.0 for k in groups}
    tot["rest (GCN, all GEMMs incl. the mask head's, optimizer)"] = 0.0
    kernels = []
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if us <= 0:
            continue
        kernels.append((e.key, us / n))
        for k, pats in groups.items():
            if any(p in e.key for p in pats):
                tot[k] += us / n
                break
        else:
            tot["rest (GCN, all GEMMs incl. the mask head's, optimizer)"] += us / n
    kernels.sort(key=lambda x: -x[1])
    for k, v in tot.items():
        print("%-60s %9.1f us/step" % (k, v))
    for k, v in kernels[:30]:
        print("  %-90s %9.1f us/step" % (k[:90], v))
    return {"groups_us_per_step": {k: round(v, 1) for k, v in tot.items()},
            "top_kernels_us_per_step": [(k, round(v, 1)) for k, v in kernels[:40]]}


if __name__ == "__main__":
    main()
