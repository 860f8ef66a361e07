"""fp32 vs bf16 vs fp16 layout canvases on the GPU: forward and d/dvecs backward on three canvases, and the
mixed-precision user's path today (fp32 canvas + .to(bf16); bf16 gradient widened + fp32 kernel) against the direct
16-bit kernels.  CUDA events, L2 flushed (a 256 MB write) before every timed pass, variants alternated in one process.
GB/s are at the canvas element size; "copy" is the fraction of a device-to-device copy of the same bytes, timed the
same way in the same run.  Usage: python scratch/bench_layout16.py [--reps 20] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from canonicalsg2im_b200 import synth  # noqa: E402
from canonicalsg2im_b200.layout import layout_batched  # noqa: E402

DT = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def objs(seed, n_img, n_min, n_max, D, M=4, box_mode="coco"):
    vocab = synth.Vocab(0)
    vecs, boxes, masks, off = [], [], [], [0]
    for i in range(n_img):
        g = synth.make_graph(seed * 100 + i, n_min, n_max, vocab, include_dummies=False, mask_size=M, box_mode=box_mode)
        vecs.append(synth.det_tensor((len(g.boxes), D), seed * 1000 + i, 1.0))
        boxes.append(g.boxes)
        masks.append(g.masks)
        off.append(off[-1] + len(g.boxes))
    c = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return (c(np.concatenate(vecs)), c(np.concatenate(boxes)), c(np.concatenate(masks).astype(np.float32)),
            c(np.array(off, np.int32)), max(np.diff(off)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", torch.cuda.get_device_name(0), "|", smi)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fns):
        """{name: median us} for the callables in `fns`, alternated, L2 flushed before each timed pass."""
        res = {k: [] for k in fns}
        for k, f in fns.items():           # warm-up
            f(); f()
        for _ in range(args.reps):
            for k, f in fns.items():
                flush_buf.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); f(); e1.record()
                torch.cuda.synchronize()
                res[k].append(e0.elapsed_time(e1) * 1e3)
        return {k: float(np.median(v)) for k, v in res.items()}

    cases = []
    v, b, m, off, mo = objs(1, 128, 3, 31, 128)
    cases.append(("cfg2 boxes 128x128x64x64", dict(vecs=v, boxes=b, obj_offsets=off, H=64, W=64, max_objs_per_image=mo), True))
    v, b, m, off, mo = objs(2, 16, 3, 8, 128, M=16)
    cases.append(("cfg3 masks 16x128x256x256", dict(vecs=v, boxes=b, obj_offsets=off, H=256, W=256, masks=m,
                                                    max_objs_per_image=mo), True))
    v, b, m, off, mo = objs(3, 10, 32, 64, 128, M=16, box_mode="clevr")
    cases.append(("cfg4 occlusion 10x128x256x256", dict(vecs=v, boxes=b, obj_offsets=off, H=256, W=256, masks=m,
                                                        test_mode=True), False))
    report = {"gpu": smi, "reps": args.reps, "l2_flush": "256 MB write before every timed pass", "cases": {}}
    for name, kw, bwd in cases:
        N, D = kw["obj_offsets"].numel() - 1, kw["vecs"].shape[1]
        n_el = N * D * kw["H"] * kw["W"]
        src32 = torch.empty(n_el, dtype=torch.float32, device="cuda")
        dst32 = torch.empty_like(src32)
        src16, dst16 = src32.view(torch.int16)[:n_el], dst32.view(torch.int16)[:n_el]
        fns = {"copy fp32": lambda: dst32.copy_(src32), "copy 16-bit": lambda: dst16.copy_(src16)}
        for k, dt in DT.items():
            fns["fwd " + k] = (lambda dt=dt: layout_batched(out_dtype=dt, **kw))
        fns["fwd fp32 + .to(bf16)"] = lambda: layout_batched(**kw).to(torch.bfloat16)
        if bwd:
            vg = kw["vecs"].clone().requires_grad_(True)
            kb = dict(kw, vecs=vg)
            g32 = torch.randn((N, D, kw["H"], kw["W"]), device="cuda", generator=torch.Generator("cuda").manual_seed(0))
            gs = {k: g32.to(dt) for k, dt in DT.items()}
            ys = {k: layout_batched(out_dtype=dt, **kb) for k, dt in DT.items()}
            for k in DT:
                fns["bwd " + k] = (lambda k=k: torch.autograd.grad(ys[k], vg, gs[k], retain_graph=True))
            fns["bwd bf16 grad -> fp32 kernel"] = lambda: torch.autograd.grad(ys["fp32"], vg, gs["bf16"].float(),
                                                                              retain_graph=True)
        t = timed(fns)
        out = {}
        for k, us in t.items():
            es = 4 if ("fp32" in k and "->" not in k and "+" not in k) or k == "copy fp32" else 2
            gbs = n_el * es / (us * 1e-6) / 1e9
            copy = t["copy fp32" if es == 4 else "copy 16-bit"]
            out[k] = {"us": round(us, 1), "GB/s": round(gbs, 1), "of_copy": round(copy / us, 3)}
            print("%-32s %-30s %9.1f us %8.1f GB/s  %.2f of copy" % (name, k, us, gbs, copy / us))
        report["cases"][name] = out
        del src32, dst32, fns
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_layout16.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
