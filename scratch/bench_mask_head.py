"""Mask head (Sg2LayoutModel, mask_size = 16) on a cfg2-sized object set: forward and forward + backward on the fp32
parity engine and the bf16 tensor-core engine, training mode.  CUDA events, L2 flushed (a 256 MB write) before every
timed pass, engines alternated in one process.  A torch.profiler pass of its own then splits the device time into the
GEMMs (achieved TFLOP/s over the algorithmic FLOPs 2 * rows * C * 9C per convolution, x3 with backward) and the
memory-bound kernels (bytes each one must move, over its time).  Prints the GPU name and power limit first.
Usage: python scratch/bench_mask_head.py [--objs 2200] [--reps 10] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from canonicalsg2im_b200.mask_head import build_mask_net, mask_head  # noqa: E402

C, M = 128, 16
ESZ = {"fp32": 4, "bf16": 2}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    except OSError:
        q = torch.cuda.get_device_name()
    return q


def kernel_bytes(O, e, backward):
    """Bytes the memory-bound kernels must move, per kernel family (e = activation element size)."""
    b = {}
    stages = [2 ** i for i in range(4)]
    for s in stages:
        n, rows = O * s * s, O * 4 * s * s
        b["patch"] = b.get("patch", 0) + rows * 9 * C * e + n * C * e          # write A, read x
        b["bn_fwd"] = b.get("bn_fwd", 0) + n * C * e                          # read x once
        if backward:
            b["patch"] += rows * 9 * C * e + n * C * e                         # the rebuilt A
            b["bn_bwd_gather"] = b.get("bn_bwd_gather", 0) + rows * 9 * C * e + n * C * (e + 4)
            b["bn_bwd_dx"] = b.get("bn_bwd_dx", 0) + n * C * (4 + e + e)
    R = O * M * M
    b["head_fwd"] = R * C * e + R * 4
    if backward:
        b["head_bwd"] = R * C * e * 2 + R * 8
    return b


def gemm_flops(O, backward):
    f = sum(2.0 * O * 4 * s * s * C * 9 * C for s in (1, 2, 4, 8))
    return f * (3 if backward else 1)


def family(name):
    for key, fam in (("patch_kernel", "patch"), ("bn_partial", "bn_fwd"), ("bn_final", "bn_fwd"),
                     ("bn_bwd_gather", "bn_bwd_gather"), ("bn_bwd_final", "bn_bwd_gather"), ("bn_bwd_dx", "bn_bwd_dx"),
                     ("head_fwd", "head_fwd"), ("head_bwd", "head_bwd"), ("gemm", "gemm"), ("split3", "gemm_split"),
                     ("colsum", "colsum"), ("cast", "cast")):
        if key in name:
            return fam
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--objs", type=int, default=2200)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    print("GPU:", gpu_info())
    O = args.objs
    torch.manual_seed(0)
    net = build_mask_net(C, M).cuda()
    x32 = torch.randn(O, C, device="cuda")
    dmask = torch.randn(O, M, M, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    inputs = {"fp32": x32, "bf16": x32.to(torch.bfloat16)}

    def run(engine, backward):
        x = inputs[engine].detach().requires_grad_(backward)
        if backward:
            out = mask_head(net, x, engine)
            out.backward(dmask)
        else:
            with torch.no_grad():
                mask_head(net, x, engine)

    res = {"gpu": gpu_info(), "objs": O, "mask_size": M}
    times = {}
    for engine in ("fp32", "bf16"):
        for bwd in (False, True):
            run(engine, bwd)
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for engine in ("fp32", "bf16"):
            for bwd in (False, True):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(engine, bwd)
                e1.record()
                torch.cuda.synchronize()
                times.setdefault((engine, bwd), []).append(e0.elapsed_time(e1))
    for (engine, bwd), ts in times.items():
        ts = sorted(ts)
        key = "%s_%s" % (engine, "fwd_bwd" if bwd else "fwd")
        res[key + "_ms_median"] = ts[len(ts) // 2]
        res[key + "_ms_min"] = ts[0]
        res[key + "_gemm_tflops_end_to_end"] = gemm_flops(O, bwd) / (ts[len(ts) // 2] * 1e-3) / 1e12
        print("%-14s median %.3f ms  min %.3f ms" % (key, ts[len(ts) // 2], ts[0]))
    # kernel split (profiler run of its own)
    from torch.profiler import profile, ProfilerActivity
    for engine in ("fp32", "bf16"):
        for bwd in (False, True):
            reps = 3
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    run(engine, bwd)
                torch.cuda.synchronize()
            fam_t = {}
            for ev in prof.key_averages():
                t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                if t:
                    f = family(ev.key)
                    fam_t[f] = fam_t.get(f, 0.0) + t / reps      # us per pass
            key = "%s_%s" % (engine, "fwd_bwd" if bwd else "fwd")
            kb = kernel_bytes(O, ESZ[engine], bwd)
            row = {}
            for f, us in sorted(fam_t.items(), key=lambda kv: -kv[1]):
                entry = {"us": round(us, 1)}
                if f == "gemm":
                    entry["tflops"] = round(gemm_flops(O, bwd) / (us * 1e-6) / 1e12, 1)
                if f in kb:
                    entry["GB"] = round(kb[f] / 1e9, 3)
                    entry["TB_per_s"] = round(kb[f] / (us * 1e-6) / 1e12, 2)
                row[f] = entry
            res[key + "_kernels"] = row
            print(key, json.dumps(row))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_mask_head.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
