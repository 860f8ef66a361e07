#!/usr/bin/env python
"""bench.py -- scene graphs/sec of the SG -> layout training step (GCN + layout, fwd + bwd).

    python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...     # CPU restatement of the reference (oracle port)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + what the last timed step computed, as .npy

Headline workload (BASELINE.json configs[1], "cfg2"): 128 scene graphs per GPU, 3-30 objects each (+ the
__image__ dummy), VG-like vocabulary (50 predicates), WSGC canonicalization with learned converse +
transitive edges, 5-layer GraphTripleConv stack (embed 128 / hidden 512) + box_net + box loss, the generator-side
object embedding composited by boxes_to_layout into a 64x64x128 canvas on the GT boxes, backward through both, Adam.
Synthetic graphs, random-init weights, all seeded: the same arguments give the same inputs in every run.  One JSON
line on rank 0.

The same line carries `configs`: BASELINE.json's other configurations measured in the same run
(cfg1 CPU-sized step, cfg3 256x256 mask canvas, cfg4 CLEVR forward-only path, cfg5 ~1M-triple batch sharded over the
ranks = strong scaling) and the fp32 parity engine on cfg2 -- each with its own roofline fraction and CPU-port number.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (no __pycache__)

import numpy as np   # noqa: E402
import torch         # noqa: E402

from canonicalsg2im_b200 import synth   # noqa: E402

METRIC = "scene_graphs_per_sec_gcn_layout_fwd_bwd"
UNIT = "graphs/s"
WORKLOAD = ("cfg2: packed_vg-like SG->layout training step with WSGC canonicalization, batch 128/GPU, 3-30 objects, "
            "P=50, 5x GraphTripleConv(128/512) + box_net + box loss + boxes_to_layout 64x64x128 of the generator "
            "embedding, fwd+bwd+Adam")
FLOP_PER_TRIPLE_LAYER = 1572864.0       # SURVEY.md section 8(d): forward, D = 128, H = 512
FLOP_PER_OBJECT_LAYER = 655360.0
FLOP_PER_OBJECT_BOXNET = 135168.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("CSG_PRECISION", "bf16"), choices=["fp32", "bf16"],
                    help="bf16 = tcgen05 tensor-core engine (north_star: bf16 MLP, fp32 accumulate, 1e-2 rel); "
                         "fp32 = the 1e-5 parity engine")
    ap.add_argument("--batch", type=int, default=128, help="graphs per GPU")
    ap.add_argument("--cpu-sample", type=int, default=16,
                    help="graphs per step of the bounded CPU sample of the cfg2 workload (cfg1's batch size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default=os.environ.get("CSG_BENCH_CONFIGS", "all"),
                    help="extra BASELINE configs measured beside the cfg2 headline: all | none | comma list of "
                         "cfg1,cfg3,cfg4,cfg5,fp32,nccl_check")
    ap.add_argument("--cfg5-graphs", type=int, default=1100, help="graphs of the cfg5 global batch (~1M triples)")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every kernel eagerly instead of replaying the captured CUDA graph of forward + backward")
    ap.add_argument("--profile", action="store_true",
                    help="profiling run: cudaProfilerStart/Stop around the timed region (ncu --profile-from-start off), "
                         "no e2e / CPU legs / extra configs; the printed numbers are not bench values")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy: its loss, its "
                         "canonicalized triple count and every parameter after its Adam update (rank 0, ~23 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ workloads
def workload_graphs(batch, seed):
    vocab = synth.Vocab(42)
    return vocab, synth.make_graphs(batch, 1000 + seed, 3, 30, vocab, include_dummies=True)


def cfg1_graphs(batch=16):
    vocab = synth.Vocab(0)
    return vocab, synth.make_graphs(batch, 3100, 3, 8, vocab, include_dummies=True)


def cfg4_graphs(batch=10):
    CFG4_ATTR_SIZES = list(synth.CLEVR_ATTR_SIZES)
    vocab = synth.Vocab(0, num_attributes=4)
    graphs = synth.make_graphs(batch, 4400, 32, 64, vocab, include_dummies=True, box_mode="clevr", mask_size=16)
    for g in graphs:
        for k, n in enumerate(CFG4_ATTR_SIZES):
            g.objs[:-1, k] = 1 + (g.objs[:-1, k] - 1) % (n - 1)
    return vocab, graphs, CFG4_ATTR_SIZES


def cfg3_objects(batch=16):
    vocab = synth.Vocab(0)
    vecs, boxes, masks, off = [], [], [], [0]
    for i in range(batch):
        g = synth.make_graph(3300 + i, 3, 8, vocab, include_dummies=False, mask_size=16)
        n = len(g.boxes)
        vecs.append(synth.det_tensor((n, 128), 3400 + i, 1.0))
        boxes.append(g.boxes); masks.append(g.masks); off.append(off[-1] + n)
    return np.concatenate(vecs), np.concatenate(boxes), np.concatenate(masks).astype(np.float32), np.array(off, np.int32)


def main_config(args, world, n_obj, n_tri):
    prec = args.precision
    return {"workload": WORKLOAD, "graphs_per_gpu": args.batch, "objects": n_obj, "triples_after_canon": n_tri,
            "precision": prec, "parallelism": "graph-sharded dp%d" % world,
            "l2": "per-step working set (net1 activations %.0f MB + 268 MB canvas + 268 MB canvas grad) exceeds the 126 MB L2"
                  % (n_tri * (1152 + 512) * (4 if prec == "fp32" else 2) / 1e6)}


# ------------------------------------------------------------------------------------------ CPU arm
def model_conv_weights(state):
    """sg2im/model.py:8-15 on the random-init state: the symmetrised converse weights the dataset samples from."""
    tri = np.triu(state["converse_candidates_weights"])
    return (tri + tri.T).astype(np.float64)


def cpu_step_runner(vocab, graphs, threads, H=64, W=64):
    from oracle.step import CpuStep
    torch.set_num_threads(threads)
    st = synth.make_state(vocab, seed=0)
    step = CpuStep(vocab, st, model_conv_weights(st), synth.make_layout_state(vocab, 128, seed=0), H=H, W=W)
    uni = synth.det_uniform(sum(len(g.triplets) for g in graphs), 13)
    return step, uni


def time_cpu_steps(step, graphs, uni, budget_s, max_steps, warm=True):
    if warm:
        step.step(graphs, uni)
    t0 = time.perf_counter()
    n = 0
    while True:
        step.step(graphs, uni)
        n += 1
        if time.perf_counter() - t0 > budget_s or n >= max_steps:
            break
    return (time.perf_counter() - t0) / n, n


CPU_NOTE = ("per-graph CPU cost of the reference grows with the batch (rows padded to the longest graph; the backward of "
            "its per-sample slicing loop, graph.py:85-107, is O(B^2)): the full cfg2 batch of 128 costs ~290 s/step = "
            "0.44 graphs/s on 8 cores (measured once, DESIGN.md section 6), so this sample OVER-states its throughput")


def run_cpu_baseline(sample, threads, budget_s=25.0):
    vocab, graphs = workload_graphs(sample, 0)
    step, uni = cpu_step_runner(vocab, graphs, threads)
    dt, n = time_cpu_steps(step, graphs, uni, budget_s, 3, warm=False)
    return {"value": sample / dt, "unit": UNIT, "cores": threads, "cpu": cpu_model(), "kind": "port",
            "ms_per_step": 1e3 * dt,
            "sample": "%d graphs of the cfg2 workload per step, %d timed steps, oracle/step.py (torch-CPU + numpy); %s"
                      % (sample, n, CPU_NOTE)}


def canon_count_cpu(vocab, graphs, seed):
    """Canonicalized triple count of the full workload with the draws the GPU arm uses (oracle, ~1 s)."""
    from oracle import canon as ocanon
    Wc = model_conv_weights(synth.make_state(vocab, seed=0))
    tri_off = np.concatenate([[0], np.cumsum([len(g.triplets) for g in graphs])])
    uni = synth.det_uniform(int(tri_off[-1]), seed * 7919 + 13)
    total = 0
    for i, g in enumerate(graphs):
        tr, _, _, _ = ocanon.add_learnt_triplets(g.triplets, vocab.num_preds, vocab.meta_ids, Wc, True, True, uni[tri_off[i]:])
        total += len(tr)
    return total


def run_reference(args):
    """The reference's CPU implementation of the path (oracle port: the reference is Python and cannot travel to the
    box, DESIGN.md section 6) on the host cores, `config` = the GPU arm's; each step a bounded sample of it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    sample = max(1, args.cpu_sample)
    vocab, full = workload_graphs(args.batch, 0)
    n_obj = sum(len(g.objs) for g in full)
    graphs = full[:sample]
    step, uni = cpu_step_runner(vocab, graphs, threads)
    for _ in range(min(args.warmup, 1)):          # one bounded warm-up step (each CPU step costs seconds, nothing to JIT)
        step.step(graphs, uni)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step.step(graphs, uni)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": main_config(args, args.gpus, n_obj, canon_count_cpu(vocab, full, 0)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "cpu": cpu_model(), "kind": "port",
                         "sample": "%d graphs (the first %d of the %d-graph cfg2 batch) per step, oracle/step.py "
                                   "(torch-CPU + numpy), 1 warm-up step; %s" % (sample, sample, args.batch, CPU_NOTE)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU helpers
class L2Flusher:
    """Writes a 256 MB buffer (2x the 126 MB L2) between timed iterations of workloads whose inputs fit in L2."""

    def __init__(self, dev):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def __call__(self):
        self.buf.fill_(1)


def time_each(fn, steps, warmup, flush=None):
    """CUDA-event timing on the current stream.  Without `flush` (working set larger than L2) the `steps` iterations
    are timed back to back in one bracket; with it, every iteration is bracketed on its own and an (untimed) L2 flush
    runs between iterations."""
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / steps
    evs = []
    for _ in range(steps):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) * 1e-3 / steps


def layout_roofline(boxes, off, max_objs, N, D, H, W, pk, masks=None, iters=20, flush=None):
    """The layout compositor pair timed alone through the C ABI (CUDA events on the launching stream).  Algorithmic
    bytes: forward = one write of N*D*H*W*4, backward = one read of the same (SURVEY.md section 8d)."""
    from canonicalsg2im_b200 import _lib
    from canonicalsg2im_b200.layout import _linspace
    from canonicalsg2im_b200.ops import lib, ptr, workspace, _stream
    L = lib()
    dev = boxes.device
    NO = boxes.shape[0]
    M = masks.shape[1] if masks is not None else 0
    gen = torch.Generator(device=dev).manual_seed(7)
    vecs = torch.randn((NO, D), device=dev, generator=gen)
    G = torch.randn((N, D, H, W), device=dev, generator=gen)
    out = torch.empty_like(G)
    dv = torch.empty((NO, D), device=dev)
    lx, ly = _linspace(W, dev), _linspace(H, dev)
    ws = workspace(L.csg_layout_bwd_vecs_workspace(N, NO, D, H, W), dev)

    def fwd():
        _lib.check(L.csg_layout_fwd(ptr(vecs), ptr(boxes), ptr(masks), ptr(off), ptr(lx), ptr(ly), ptr(out), N, D, H, W, M,
                                    0, max_objs, _stream()), "csg_layout_fwd")

    def bwd():
        _lib.check(L.csg_layout_bwd_vecs(ptr(G), ptr(boxes), ptr(masks), ptr(off), ptr(lx), ptr(ly), ptr(dv), N, NO, D, H,
                                         W, M, 0, max_objs, ptr(ws), ws.numel(), _stream()), "csg_layout_bwd_vecs")
    res = {}
    nbytes = N * D * H * W * 4
    for name, fn in (("fwd", fwd), ("bwd", bwd)):
        sec = time_each(fn, iters, 3, flush)
        res[name] = {"us": sec * 1e6, "achieved": nbytes / sec / 1e9, "frac": nbytes / sec / 1e9 / pk["hbm"]}
    kind = "masks_to_layout" if masks is not None else "boxes_to_layout"
    bwd_kernel = "layout_bwd_ring_kernel" if masks is not None else "layout_bwd_colsum_kernel"
    return {"kernel": "layout_fwd_kernel / %s (%s %dx%dx%dx%d)" % (bwd_kernel, kind, N, D, H, W),
            "bound": "hbm", "unit": "GB/s", "peak": pk["hbm"], "peak_source": pk["src"] + " copy bandwidth",
            "bytes_per_launch": nbytes, "fwd": res["fwd"], "bwd": res["bwd"],
            "l2": "canvas of %.0f MB %s the 126 MB L2%s" % (nbytes / 1e6, "exceeds" if nbytes > 126e6 else "fits in",
                                                           "" if nbytes > 126e6 else "; L2 flushed between iterations")}


def dump_outputs(out_dir, step, loss, n_tri):
    """What the last timed step hands its caller, as <out_dir>/<name>.npy: the loss it returned, its canonicalized
    triple count and every parameter after its Adam update (float32 / float64).  The inputs are seeded, so two builds
    run with the same arguments can be compared file by file."""
    step.finish()                  # under graph replay Adam of the last step runs on the look-ahead stream
    arrays = {"loss": loss.detach().float().cpu().numpy(), "triples_after_canon": np.array(n_tri, np.float64)}
    for prefix, module in (("model.", step.model), ("layout_embedding.", step.layout_embedding)):
        for name, p in module.named_parameters():
            arrays["param." + prefix + name] = p.detach().float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def mlp_flops(n_tri, n_obj, layers=5, train=True):
    f = layers * (n_tri * FLOP_PER_TRIPLE_LAYER + n_obj * FLOP_PER_OBJECT_LAYER) + n_obj * FLOP_PER_OBJECT_BOXNET
    return f * (3.0 if train else 1.0)


def train_leg(vocab, graphs, dev, precision, steps, warmup, pk, flush=None, cpu=None, H=64, W=64, seed=0):
    """K training steps of a small config (cfg1 / fp32 engine): device-timed with resident inputs, per-step events."""
    from canonicalsg2im_b200.pipeline import SgToLayoutStep, HostBatch
    hb = HostBatch(graphs, seed=seed)
    step = SgToLayoutStep(vocab, dev, precision=precision, H=H, W=W, seed=0, use_graph=True)
    G = torch.randn((len(graphs), 128, H, W), device=dev, generator=torch.Generator(device=dev).manual_seed(99)) * 1e-3
    d = hb.to_device(dev)
    box = {}

    def one():
        box["loss"], box["n_tri"] = step.step(d, G, prefetch=d)
    sec = time_each(one, steps, warmup, flush)
    n_obj, n_tri = int(hb.obj_off[-1]), box["n_tri"]
    flops = mlp_flops(n_tri, n_obj)
    out = {"ms_per_step": 1e3 * sec, "graphs_per_s": len(graphs) / sec, "graphs": len(graphs), "objects": n_obj,
           "triples_after_canon": n_tri, "precision": precision, "steps": steps,
           "mlp_tflops_whole_step": flops / sec / 1e12, "loss": float(box["loss"].item()),
           "cuda_graph_replays": step.graph_replays}
    del step, G, d
    return out


# ------------------------------------------------------------------------------------------ extra configs
def run_cfg1(dev, pk, args, flush, with_cpu):
    """BASELINE configs[0]: batch 16, <= 8 objects, P = 8, boxes_to_layout 64x64 -- the reference's CPU-runnable case.
    The working set (33 MB canvas) fits in L2, so L2 is flushed between the timed steps."""
    vocab, graphs = cfg1_graphs()
    out = {"workload": "cfg1: packed_coco-like training step, batch 16, 3-8 objects, P=8, 5x GraphTripleConv(128/512), "
                       "boxes_to_layout 64x64x128, fwd+bwd+Adam", "l2": "working set fits in L2; flushed between steps"}
    for prec in ("bf16", "fp32"):
        out[prec] = train_leg(vocab, graphs, dev, prec, max(args.steps, 10), args.warmup, pk, flush)
    boxes = torch.from_numpy(np.concatenate([g.boxes for g in graphs])).to(dev)
    off = torch.from_numpy(np.concatenate([[0], np.cumsum([len(g.objs) for g in graphs])]).astype(np.int32)).to(dev)
    out["roofline_hbm"] = layout_roofline(boxes, off, max(len(g.objs) for g in graphs), len(graphs), 128, 64, 64, pk,
                                          flush=flush)
    if with_cpu:
        threads = os.cpu_count() or 1
        step, uni = cpu_step_runner(vocab, graphs, threads)
        dt, n = time_cpu_steps(step, graphs, uni, 10.0, 5)
        out["cpu_baseline"] = {"value": len(graphs) / dt, "unit": UNIT, "cores": threads, "kind": "port",
                               "ms_per_step": 1e3 * dt,
                               "sample": "the whole cfg1 batch (16 graphs), %d timed steps, oracle/step.py" % n}
    return out


def run_fp32(dev, pk, args):
    """cfg2 on the fp32 (1e-5 parity) engine."""
    vocab, graphs = workload_graphs(args.batch, 0)
    out = train_leg(vocab, graphs, dev, "fp32", 5, 3, pk)
    out["note"] = "cfg2 batch on the fp32 FMA parity engine (csrc/gemm_f32.cu); same step as the headline"
    # the same step with every fp32 GEMM on tcgen05 through the exact three-term bf16 split (ops.F32_ENGINE = "tc"): meets
    # the same 1e-5 golden contract as the FMA engine once the products are ordered for the truncating accumulator
    # (DESIGN.md section 9)
    from canonicalsg2im_b200 import ops
    old = ops.F32_ENGINE
    try:
        ops.set_f32_engine("tc")
        tc = train_leg(vocab, graphs, dev, "fp32", 5, 3, pk)
        out["split_bf16x3_on_tcgen05"] = {"ms_per_step": tc["ms_per_step"], "graphs_per_s": tc["graphs_per_s"], "loss": tc.get("loss"),
                                          "note": "fp32 GEMMs as K-concatenated three-term bf16 splits on tcgen05 (csg_split3_bf16), products "
                                                  "ordered smallest first, hi*hi of the weight gradients in chains of <= 64 MMAs: "
                                                  "as accurate against float64 as the FMA kernel, same 1e-5 golden contract"}
    except Exception as ex:
        out["split_bf16x3_on_tcgen05"] = {"error": repr(ex)[:200]}
    finally:
        ops.set_f32_engine(old)
    return out


def run_cfg3(dev, pk, args, with_cpu):
    """BASELINE configs[2]: masks_to_layout, batch 16, 3-8 objects, 16x16 masks, D = 128, 256x256 (512 MiB canvas)."""
    from canonicalsg2im_b200.layout import layout_batched
    vecs, boxes, masks, off = cfg3_objects()
    tb, tm, to = torch.from_numpy(boxes).to(dev), torch.from_numpy(masks).to(dev), torch.from_numpy(off).to(dev)
    N = len(off) - 1
    mo = int(np.diff(off).max())
    hbm = layout_roofline(tb, to, mo, N, 128, 256, 256, pk, masks=tm, iters=max(args.steps, 10))
    # the same through the public autograd API: fwd + bwd of masks_to_layout on the flat batch
    v = torch.from_numpy(vecs).to(dev).requires_grad_(True)
    G = torch.randn((N, 128, 256, 256), device=dev, generator=torch.Generator(device=dev).manual_seed(5))

    def both():
        v.grad = None
        layout_batched(v, tb, to, 256, 256, masks=tm, max_objs_per_image=mo).backward(G)
    sec = time_each(both, max(args.steps, 10), 3)
    out = {"workload": "cfg3: masks_to_layout fwd+bwd, batch 16, 3-8 objects, 16x16 masks, D=128, 256x256 (canvas 512 MiB)",
           "objects": int(off[-1]), "ms_fwd_bwd": 1e3 * sec, "images_per_s": N / sec,
           "hbm_fwd_bwd": {"achieved": 2 * hbm["bytes_per_launch"] / sec / 1e9, "frac": 2 * hbm["bytes_per_launch"] / sec / 1e9 / pk["hbm"],
                           "unit": "GB/s", "note": "2 x 512 MiB algorithmic / time of layout_batched(...).backward(G) "
                                                    "(includes the allocation of the canvas by torch)"},
           "roofline_hbm": hbm}
    del G
    if with_cpu:
        from oracle import layout as olayout
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        vc = torch.from_numpy(vecs).requires_grad_(True)
        t0 = time.perf_counter()
        y = olayout.batched_layout([vc[off[i]:off[i + 1]] for i in range(N)],
                                   [torch.from_numpy(boxes[off[i]:off[i + 1]]) for i in range(N)],
                                   [torch.from_numpy(masks[off[i]:off[i + 1]]) for i in range(N)], 256, 256)
        y.backward(torch.ones_like(y))
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": N / dt, "unit": "images/s", "cores": threads, "kind": "port",
                               "ms_fwd_bwd": 1e3 * dt, "sample": "the whole cfg3 batch once, oracle/layout.py fwd+bwd"}
    return out


def run_cfg4(dev, pk, args, flush, with_cpu):
    """BASELINE configs[3]: CLEVR-sized graphs (10 graphs of 32-64 objects, 4 attributes x emb 32), forward only,
    test_mode: add_location_triplets + dummies -> canonicalization -> GCN -> occlusion canvas 256x256, all on device."""
    from canonicalsg2im_b200.pipeline import SgToLayoutInference, HostBatch
    vocab, graphs, sizes = cfg4_graphs()
    nu = sum(4 * len(g.objs) ** 2 for g in graphs)
    hb = HostBatch(graphs, seed=4, with_geometry=True, num_uniforms=nu)
    inf = SgToLayoutInference(vocab, dev, precision="fp16", H=256, W=256, embedding_dim=32, attr_sizes=sizes)
    d = hb.to_device(dev)
    box = {}

    def one():
        canvas, boxes_pred, n = inf.step(d)
        box["n"], box["canvas"] = n, canvas
    sec = time_each(one, max(args.steps // 2, 5), 3, flush)
    n_obj, n_tri = int(hb.obj_off[-1]), box["n"]
    # end to end: host buffers in, canvas checksum out
    chk = torch.empty(1, dtype=torch.float32, pin_memory=True)
    for _ in range(2):                       # warm the allocator for the per-step upload buffers
        dd = hb.to_device(dev)
        canvas, _, _ = inf.step(dd)
        chk.copy_(canvas.sum().reshape(1), non_blocking=False)
    t0 = time.perf_counter()
    k = 5
    for _ in range(k):
        dd = hb.to_device(dev)
        canvas, _, _ = inf.step(dd)
        chk.copy_(canvas.sum().reshape(1), non_blocking=False)
    e2e = (time.perf_counter() - t0) / k
    canvas_bytes = box["canvas"].numel() * 4
    flops = mlp_flops(n_tri, n_obj, train=False)
    out = {"workload": "cfg4: CLEVR forward-only path (generate_clevr), 10 graphs x 32-64 objects, 4 attributes x emb 32, "
                       "location+dummy triplets -> canonicalization -> 5x GraphTripleConv + box_net -> "
                       "masks_to_layout(test_mode) 256x256x128 on the predicted boxes",
           "graphs": len(graphs), "objects": n_obj, "triples_after_canon": n_tri, "ms_per_step": 1e3 * sec,
           "graphs_per_s": len(graphs) / sec, "e2e_ms_per_step": 1e3 * e2e, "e2e_graphs_per_s": len(graphs) / e2e,
           "h2d_bytes_per_step": int(hb.nbytes), "mlp_tflops_whole_step": flops / sec / 1e12,
           "canvas_bytes": canvas_bytes, "l2": "flushed between steps", "precision": "fp16 forward tensors (inference-only)",
           "note": "latency-bound: 2 host waits (location / canonicalization sizes) and ~60 launches per step"}
    del box, d
    if with_cpu:
        out["cpu_baseline"] = cfg4_cpu(vocab, graphs, sizes, hb)
    return out


def cfg4_cpu(vocab, graphs, sizes, hb):
    """Oracle port of the same forward path on 2 of the 10 graphs (the per-graph cost does not depend on the batch:
    every stage is a per-graph Python loop except the padded GCN forward)."""
    from oracle import canon as ocanon, graph as ograph, layout as olayout
    from oracle.step import collate
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sub = graphs[:2]
    st_np = synth.make_state(vocab, embedding_dim=32, seed=0, attr_vocab_sizes=sizes)
    Wc = model_conv_weights(st_np)
    st = {k: torch.from_numpy(v) for k, v in st_np.items()}
    lst = {"generator.attribute_embedding." + k: torch.from_numpy(v)
           for k, v in synth.make_layout_state(vocab, 32, seed=0, attr_vocab_sizes=sizes).items()}
    t0 = time.perf_counter()
    with torch.no_grad():
        canon = []
        for g in sub:
            cen = np.concatenate([g.centers, np.zeros((len(g.boxes) - len(g.centers), 2), np.float32)])
            trip = list(ocanon.add_location_triplets(g.boxes, cen, g.objs[:, 0], vocab.image_obj_id, vocab.pred_ids))
            trip += list(ocanon.add_dummy_triplets(g.objs[:, 0], vocab.image_obj_id, vocab.in_image_id, True))
            trip = np.array(trip, dtype=np.int64).reshape(-1, 3)
            tr, _, ty, _ = ocanon.add_learnt_triplets(trip, vocab.num_preds, vocab.meta_ids, Wc, True, True,
                                                      synth.det_uniform(2 * len(trip) + 8, 5))
            canon.append((tr, ty))
        objs, boxes, trips, types = collate(vocab, sub, canon)
        _, boxes_pred = ograph.sg2layout_forward(st, objs, trips, types, vocab.padding_id)
        lv = ograph.attribute_embeddings(lst, "generator.attribute_embedding.", objs)
        for b, g in enumerate(sub):
            keep = (objs[b] != 0)[:, 0]
            m = torch.from_numpy(g.masks.astype(np.float32))[:int(keep.sum())]
            olayout.masks_to_layout(lv[b][keep], boxes_pred[b][keep], m, 256, 256, test_mode=True)
    dt = time.perf_counter() - t0
    return {"value": len(sub) / dt, "unit": UNIT, "cores": threads, "kind": "port", "ms_per_step": 1e3 * dt,
            "sample": "2 of the 10 cfg4 graphs once: oracle add_location_triplets + add_learnt_triplets + "
                      "sg2layout_forward + masks_to_layout(test_mode)"}


def run_cfg5(dev, pk, args, world, rank, want_check):
    """BASELINE configs[4]: one GLOBAL ragged batch of ~1M canonicalized triples, cut on graph boundaries into
    `world` contiguous shards balanced by canonicalized triple count (parallel.shard_by_cost); weight gradients are
    summed over ranks by the bucketed NCCL all-reduce.  Total work is fixed: strong scaling."""
    import torch.distributed as dist
    from canonicalsg2im_b200.pipeline import SgToLayoutStep, HostBatch
    from canonicalsg2im_b200.parallel import shard_by_cost
    vocab = synth.Vocab(42)
    graphs = synth.make_graphs(args.cfg5_graphs, 4242, 3, 30, vocab, include_dummies=True)
    NG = len(graphs)
    hb_all = HostBatch(graphs, seed=3, pin=False)
    probe = SgToLayoutStep(vocab, dev, precision=args.precision, seed=0)
    d_all = hb_all.to_device(dev)
    res = probe.canonicalize(d_all)                      # per-graph canonicalized triple counts = the shard costs
    costs = (res.tri_off[1:] - res.tri_off[:-1]).cpu().tolist()
    total_tri = int(res.triplets.shape[0])
    del res
    a, b = shard_by_cost(costs, world)[rank]
    local = graphs[a:b]
    hb = HostBatch(local, seed=3, pin=True)
    u0 = int(hb_all.tri_off[a])
    hb.t["uniforms"] = hb_all.t["uniforms"][u0:u0 + int(hb.tri_off[-1])].clone()     # the global batch's draws
    gen = torch.Generator(device=dev).manual_seed(4321)
    G_all = torch.randn((NG, 128, 64, 64), device=dev, generator=gen) * 1e-3         # identical on every rank
    G = G_all[a:b]
    step = SgToLayoutStep(vocab, dev, precision=args.precision, distributed=world > 1, seed=0, global_batch=NG)
    d = hb.to_device(dev)
    check = None
    if want_check and world > 1:
        # NCCL equivalence: the all-reduced gradients of the sharded batch vs rank 0 running the whole batch alone
        step.backward(d, G)
        mine = {k: v.clone() for k, v in step.named_grads().items()}
        step.reducer.zero()
        if rank == 0:
            solo = SgToLayoutStep(vocab, dev, precision=args.precision, distributed=False, seed=0, global_batch=NG)
            solo.backward(d_all, G_all)
            ref = solo.named_grads()
            worst, worst_name = 0.0, ""
            for k, g in ref.items():
                e = ((mine[k].double() - g.double()).norm() / g.double().norm().clamp_min(1e-30)).item()
                if e > worst:
                    worst, worst_name = e, k
            check = {"max_rel_l2_grad_error_vs_single_gpu": worst, "tensor": worst_name, "tensors": len(ref),
                     "note": "rank-0 all-reduced gradients of the %d-way sharded batch vs the same global batch run on "
                             "rank 0 alone (differences: split-K / all-reduce summation order of bf16-engine "
                             "gradients)" % world}
            del solo, ref
        del mine
        # the same sharded batch through the graph-replayed step (look-ahead streams, canvas branch, Adam beside the next
        # emit pass) and through eagerly launched single-stream steps: identical weights after 4 optimizer steps
        sums = []
        for use_graph, overlap in ((False, False), (True, True)):
            st2 = SgToLayoutStep(vocab, dev, precision=args.precision, distributed=True, seed=0, global_batch=NG,
                                 use_graph=use_graph)
            st2.overlap_canvas = overlap
            for _ in range(4):
                st2.step(d, G, prefetch=d)
            st2.finish()
            torch.cuda.synchronize()
            sums.append(torch.stack([p.detach().double().sum() for p in st2.opt.params]))
            del st2
        same = bool(torch.equal(sums[0], sums[1]))
        flag = torch.tensor([1.0 if same else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if check is not None:
            check["graph_replay_with_streams_equals_eager_single_stream"] = bool(flag.item() == 1.0)
    del probe, d_all
    if not (want_check and world > 1):
        pass
    steps5 = max(3, min(args.steps, 8))
    step.tail_events = [] if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(3):
        step.step(d, G, prefetch=d)
    if step.tail_events is not None:
        step.tail_events = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    n_tri = 0
    for _ in range(steps5):
        _, n_tri = step.step(d, G, prefetch=d)
    e1.record()
    barrier()
    sec = e0.elapsed_time(e1) * 1e-3
    tail = 0.0
    if step.tail_events:
        tail = sum(x.elapsed_time(y) for x, y in step.tail_events) / len(step.tail_events)
    stats = torch.tensor([sec, float(n_tri), float(b - a), tail], device=dev, dtype=torch.float64)
    if world > 1:
        allst = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
    else:
        allst = [stats]
    allst = torch.stack(allst).cpu().numpy()
    sec = float(allst[:, 0].max())
    tri = allst[:, 1]
    n_obj_total = int(hb_all.obj_off[-1])
    flops = mlp_flops(total_tri, n_obj_total)
    out = {"workload": "cfg5: one global ragged batch of %d graphs (3-30 objects, P=50), ~1M canonicalized triples, "
                       "cut by parallel.shard_by_cost on canonicalized triple counts; training step as cfg2; weight "
                       "gradients summed by bucketed NCCL all-reduce" % NG,
           "scaling": "strong", "n_gpus": world, "graphs_total": NG, "triples_total": total_tri, "steps": steps5,
           "ms_per_step": 1e3 * sec / steps5, "graphs_per_s": NG * steps5 / sec,
           "per_rank_triples": [int(x) for x in tri], "per_rank_graphs": [int(x) for x in allst[:, 2]],
           "imbalance_max_over_mean": float(tri.max() / tri.mean()),
           "mlp_tflops_whole_step_all_gpus": flops / (sec / steps5) / 1e12,
           "allreduce_tail_ms": float(allst[:, 3].max()),
           "allreduce_tail_note": "time from the end of this rank's backward launches to the completion of the last "
                                  "gradient bucket (reducer.finish), CUDA events, max over ranks",
           "nccl_check": check}
    del step, d, G, G_all
    return out


# ------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch.distributed as dist
    from canonicalsg2im_b200 import _lib
    from canonicalsg2im_b200.pipeline import SgToLayoutStep, HostBatch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device for --impl ours (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.load()
    pk = peaks()
    want = set() if (args.profile or args.configs == "none") else (
        {"cfg1", "cfg3", "cfg4", "cfg5", "fp32", "nccl_check"} if args.configs == "all" else set(args.configs.split(",")))

    vocab, graphs = workload_graphs(args.batch, rank)
    hb = HostBatch(graphs, seed=rank)
    step = SgToLayoutStep(vocab, dev, precision=args.precision, distributed=world > 1, seed=0,
                          use_graph=not (args.no_graph or args.profile))
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    G = torch.randn((args.batch, 128, 64, 64), device=dev, generator=gen) * 1e-3
    d = hb.to_device(dev)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled every 20 ms from the warm-up to the end of the end-to-end region (all of it
    # is the same load; the device-resident timed region alone lasts ~0.1 s)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n_tri = 0
    for _ in range(max(args.warmup, 3)):
        _, n_tri = step.step(d, G, prefetch=d)
    barrier()

    # ---- timed region 1: inputs resident in HBM
    launches0 = L.csg_launch_count() + step.graph_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.profile:
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for _ in range(args.steps):
        # every step canonicalizes its own batch; the COUNTING pass of the next step's batch is enqueued one step
        # ahead (as the reference's DataLoader workers do), so K steps contain exactly K count + K emit passes
        loss, n_tri = step.step(d, G, prefetch=d)
    e1.record()
    barrier()
    if args.profile:
        torch.cuda.cudart().cudaProfilerStop()
    launches = L.csg_launch_count() + step.graph_launches - launches0     # eager launch sites + those replayed from the graph
    sec = e0.elapsed_time(e1) * 1e-3
    if args.dump_outputs and rank == 0:      # before the passes below train the same parameters further
        dump_outputs(args.dump_outputs, step, loss, n_tri)
    # ---- instrumented pass (not the headline): the same K steps with CUDA events around every GEMM / layout /
    # pooling entry point on the launching stream (csg_prof_*), for the roofline objects
    import ctypes
    prof = (ctypes.c_double * 24)()
    L.csg_prof_enable(1)
    graphed, step.use_graph = step.use_graph, False          # the instrumented pass launches eagerly (events per entry point)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(0 if args.profile else args.steps):
        step.step(d, G, prefetch=d)
    p1.record()
    torch.cuda.synchronize()
    L.csg_prof_collect(prof)
    L.csg_prof_enable(0)
    step.use_graph = graphed
    prof_sec = p0.elapsed_time(p1) * 1e-3
    cls = 1 if args.precision == "fp32" else 0
    gemm_flops, gemm_sec, gemm_n = prof[cls * 3], prof[cls * 3 + 1], int(prof[cls * 3 + 2])
    tsec = torch.tensor([sec], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tsec, op=dist.ReduceOp.MAX)
    sec = float(tsec.item())
    value = world * args.batch * args.steps / sec

    # ---- timed region 2: end to end through the public API with HOST buffers (H2D + D2H every step)
    # the data pipeline cycles through two device batch buffers (host -> device copies land in the buffer that is not
    # being trained on, on the step's look-ahead stream, behind the last step that used that buffer and beside the step
    # in flight), so the step's CUDA graph is captured once per buffer
    d.pop("_canon_plan", None)
    bufs = [hb.to_device(dev), hb.to_device(dev)]
    dd = bufs[0]
    for i in range(0 if args.profile else 4):
        nxt = hb.to_device(dev, out=bufs[(i + 1) & 1], stream=step.side)
        l, _ = step.step(dd, G, prefetch=nxt)
        dd = nxt
        float(l.item())
    barrier()
    t0 = time.perf_counter()
    lv = float("nan")
    loss_host = torch.empty(2, dtype=torch.float32, pin_memory=True)
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    for i in range(0 if args.profile else args.steps):
        # host buffers -> device for the NEXT step and its canonicalization counting pass are enqueued while this
        # step runs (one upload + one count + one emit per step inside the timed region).  Every step's loss is copied
        # to pinned host memory; the host reads it one step later (as a logging loop would), so that the read never
        # drains the launch queue.  The last loss is read before the clock stops.
        nxt = hb.to_device(dev, out=bufs[(i + 1) & 1], stream=step.side)
        l, _ = step.step(dd, G, prefetch=nxt)
        dd = nxt
        loss_host[i & 1].copy_(l, non_blocking=True)
        loss_ev[i & 1].record()
        if i > 0:
            loss_ev[(i - 1) & 1].synchronize()
            lv = float(loss_host[(i - 1) & 1])
    if not args.profile and args.steps > 0:
        loss_ev[(args.steps - 1) & 1].synchronize()
        lv = float(loss_host[(args.steps - 1) & 1])
    torch.cuda.synchronize()
    e2e_sec = time.perf_counter() - t0
    tsec = torch.tensor([e2e_sec], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tsec, op=dist.ReduceOp.MAX)
    e2e_sec = float(tsec.item())
    clocks = sampler.stop() if rank == 0 else None
    e2e = {"value": world * args.batch * args.steps / max(e2e_sec, 1e-9), "unit": UNIT,
           "h2d_bytes_per_step": int(hb.nbytes), "d2h_bytes_per_step": 4 + 8,   # loss scalar + the two canonicalization size words
           "ms_per_step": 1e3 * e2e_sec / max(args.steps, 1)}

    hbm = None
    if rank == 0 and not args.profile:
        hbm = layout_roofline(d["boxes"].float().contiguous(), d["obj_off"], int(d["max_objs"]), args.batch, 128, 64, 64, pk)
    n_obj = int(hb.obj_off[-1])
    graph_info = (step.use_graph, step.graph_replays, len(step._graphs))
    # free the headline state before the other configs (cfg5 holds ~25 GB of activations)
    del step, G, d, dd, bufs
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, in the same run
    configs = {}
    flush = L2Flusher(dev) if want else None

    def leg(name, fn):
        try:
            configs[name] = fn()
        except Exception as ex:      # an extra config never costs the headline line
            configs[name] = {"error": repr(ex)[:300]}
        torch.cuda.empty_cache()
    with_cpu = not args.no_cpu_baseline
    if "cfg5" in want:               # every rank takes part (strong scaling over the world)
        leg("cfg5", lambda: run_cfg5(dev, pk, args, world, rank, "nccl_check" in want))
    if rank == 0 and world == 1:
        if "cfg1" in want:
            leg("cfg1", lambda: run_cfg1(dev, pk, args, flush, with_cpu))
        if "cfg3" in want:
            leg("cfg3", lambda: run_cfg3(dev, pk, args, with_cpu))
        if "cfg4" in want:
            leg("cfg4", lambda: run_cfg4(dev, pk, args, flush, with_cpu))
        if "fp32" in want:
            leg("cfg2_fp32_engine", lambda: run_fp32(dev, pk, args))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak_tf = pk["tf_sustained"]
    ach_tf = gemm_flops / gemm_sec / 1e12 if gemm_sec > 0 else 0.0
    alg_tf = (mlp_flops(n_tri, n_obj) * args.steps / gemm_sec / 1e12) if gemm_sec > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(args.precision)
        except Exception:
            traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": 1e3 * sec / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
        "config": main_config(args, world, n_obj, n_tri),      # objects / triples of rank 0's batch
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": {"kernel": "net1/net2 GEMMs (%s)" % ("gemm_f32_kernel" if args.precision == "fp32" else "gemm_tc_kernel"),
                     "bound": "tensor", "achieved": alg_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": alg_tf / peak_tf, "executed_tflops": ach_tf, "executed_frac": ach_tf / peak_tf,
                     "traffic": traffic, "peak_source": pk["src"] + " bf16 sustained",
                     "launches_timed": gemm_n, "share_of_step": gemm_sec / sec if sec > 0 else None,
                     "whole_step_tflops": mlp_flops(n_tri, n_obj) / (sec / max(args.steps, 1)) / 1e12,
                     "flops_note": "achieved = ALGORITHMIC MLP flops of the step (SURVEY 8(d): 1 572 864 FLOP per triple and layer "
                                   "+ 655 360 per object and layer forward, x3 with backward) / the summed durations of the "
                                   "step's GEMM launches.  executed_tflops = the flops those launches really execute / the "
                                   "same time: fewer since net1's first-layer backward runs on per-object sums of dhidden (the "
                                   "two T-sized GEMMs have N = Dp instead of 2 Din + Dp; the segment-sum kernel that makes "
                                   "this possible is NOT in the GEMM time: 45 us per layer, DESIGN.md section 9).  With the "
                                   "fp32 engine both counts coincide",
                     "note": "CUDA events around every GEMM entry point on the launching stream, in a separate eagerly launched "
                             "pass of the same %d steps (%.3f ms/step with the events); share_of_step = summed GEMM "
                             "time / the headline timed region" % (args.steps, 1e3 * prof_sec / max(args.steps, 1))},
        "roofline_hbm": hbm,
        "loss": lv,
        "cuda_graph": {"enabled": bool(graph_info[0]), "replays": graph_info[1], "graphs": graph_info[2],
                       "note": "forward + backward (+ gradient all-reduce) of a step replay one captured CUDA graph per "
                               "(batch buffer, triple count); canonicalization and Adam are launched eagerly around it"},
        "triples_after_canon_rank0": n_tri,
        "configs": configs,
    }
    if with_cpu and not args.profile and world == 1:
        try:
            line["cpu_baseline"] = run_cpu_baseline(args.cpu_sample, os.cpu_count() or 1)
        except Exception as ex:   # the baseline is a reported number, never a reason to lose the GPU line
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                                    "sample": "failed: %r" % (ex,)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
