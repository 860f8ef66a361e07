"""One scene-graph -> layout training step on one GPU (the unit ``bench.py`` times):

    canonicalization (base_dataset.py:89-139)  ->  Sg2LayoutModel GCN stack + box_net (model.py:90-124)
    ->  box loss (pix2pix_model.py:72-85)
    generator-side attribute embedding of the objects + GT boxes  ->  boxes_to_layout canvas
    (generator.py:16,80-96, layout.py:12-45)
    ->  backward of both  ->  [grad all-reduce]  ->  Adam

As in the reference's training graph the canvas is composited from the GENERATOR's own ``AttributeEmbeddings``
table (generator.py:16,80), not from the GCN output, so the canvas gradient reaches that table only; the GCN is
trained by the box loss.  With ``mask_size > 0`` the canvas is ``masks_to_layout`` with the mask head's PREDICTED masks
(meta_models.py:48), and its gradient reaches the head and the GCN as well; with ``gt_masks=True`` it is composited from
the batch's GT masks and the head is trained by the BCE mask term of the generator loss instead.  All stages are
csg2im kernels; torch provides memory and autograd bookkeeping.
"""
import numpy as np
import os

import torch
import torch.nn.functional as F

from . import synth
from .canonicalize import canon_count_async, canon_emit, canon_total, converse_tables
from .layout import layout_batched
from .model import AttributeEmbeddings, Sg2LayoutModel, bbox_pred_loss_ragged, get_conv_converse, mask_pred_loss
from .optim import FusedAdam
from .parallel import BucketedGradAllReduce


def build_opt(vocab: synth.Vocab, embedding_dim=128, gconv_dim=128, hidden_dim=512, num_layers=5, mask_size=0):
    import argparse
    attrs = {"a%d" % i: {str(j): j for j in range(vocab.num_obj_classes if vocab.num_attributes == 1 else 8)}
             for i in range(vocab.num_attributes)}
    return argparse.Namespace(
        vocab={"attributes": attrs, "pred_idx_to_name": vocab.pred_names, "pred_name_to_idx": vocab.pred_ids},
        embedding_dim=embedding_dim, gconv_dim=gconv_dim, gconv_hidden_dim=hidden_dim, gconv_pooling="avg",
        gconv_num_layers=num_layers, mlp_normalization="none", mask_size=mask_size, learned_init="uniform")


class HostBatch:
    """Flat host-side batch (pinned when CUDA is available): what a collate function would emit."""

    def __init__(self, graphs, seed=0, pin=True, with_geometry=False, num_uniforms=None, with_masks=None):
        """``with_geometry``: also upload ``centers`` and, when the graphs carry them, ``masks [NO, M, M]`` fp32.
        ``with_masks``: upload ``masks`` regardless of ``with_geometry`` (True) or never (False); ``None`` = as
        ``with_geometry`` says (e.g. ``with_masks=True`` alone: the GT-mask training step, which needs no centers)."""
        self.B = len(graphs)
        self.tri_off = np.concatenate([[0], np.cumsum([len(g.triplets) for g in graphs])]).astype(np.int32)
        self.obj_off = np.concatenate([[0], np.cumsum([len(g.objs) for g in graphs])]).astype(np.int32)
        self.max_objs = max(len(g.objs) for g in graphs)
        arrs = dict(
            triplets=np.concatenate([g.triplets for g in graphs]).astype(np.int64),
            tri_off=self.tri_off, obj_off=self.obj_off,
            objs=np.concatenate([g.objs for g in graphs]).astype(np.int64),
            boxes=np.concatenate([g.boxes for g in graphs]).astype(np.float32),
            uniforms=synth.det_uniform(int(num_uniforms or self.tri_off[-1]), seed * 7919 + 13),
        )
        if with_geometry:      # inputs of the on-device graph construction / mask compositor (cfg4)
            arrs["centers"] = np.concatenate([np.concatenate([g.centers, np.zeros((len(g.boxes) - len(g.centers), 2),
                                                                                  np.float32)]) for g in graphs])
        if (with_geometry if with_masks is None else with_masks) and graphs[0].masks is not None:
            arrs["masks"] = np.concatenate([g.masks for g in graphs]).astype(np.float32)
        self.t = {}
        for k, v in arrs.items():
            x = torch.from_numpy(np.ascontiguousarray(v))
            if pin and torch.cuda.is_available():
                x = x.pin_memory()
            self.t[k] = x
        self.nbytes = sum(x.numel() * x.element_size() for x in self.t.values())

    def to_device(self, device, out=None, stream=None):
        """Upload (asynchronously, from pinned memory).  ``out``: a dict returned by an earlier ``to_device`` of a batch
        with the same shapes: its tensors are overwritten in place, so the device addresses stay the same (a data
        pipeline cycling through a fixed set of batch buffers; what the CUDA-graph replay of the step keys on).
        ``stream``: a look-ahead stream (``SgToLayoutStep.side``): the copies are issued there, behind everything the
        current stream has been given so far (the previous user of ``out``), and overlap the step that is launched next;
        ``d["_ready"]`` is the event consumers on other streams wait for."""
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(stream):
                d = self.to_device(device, out=out)
                d["_ready"] = torch.cuda.Event()
                d["_ready"].record(stream)
            return d
        if out is not None:
            if any(out[k].shape != v.shape for k, v in self.t.items()):
                raise ValueError("to_device(out=...): shapes differ from the buffers' batch")
            for k, v in self.t.items():
                out[k].copy_(v, non_blocking=True)
            out.pop("_canon_plan", None)
            out.pop("_ready", None)
            d = out
        else:
            d = {k: v.to(device, non_blocking=True) for k, v in self.t.items()}
        d["max_objs"] = self.max_objs
        d["B"] = self.B
        return d


class SgToLayoutStep:
    def __init__(self, vocab, device, precision="fp32", H=64, W=64, learned_converse=True,
                 learned_transitivity=True, lr=1e-4, seed=0, distributed=False, bbox_pred_loss_weight=10.0,
                 global_batch=None, use_graph=False, canvas_dtype=torch.float32, mask_size=0, gt_masks=False,
                 mask_loss_weight=1.0):
        """``global_batch``: number of graphs of the GLOBAL batch this rank holds a shard of.  The box loss is a mean
        over images (pix2pix_model.py:85), so with shards of unequal graph counts (cost-balanced sharding) every rank
        scales its loss by B_local / B_global and the gradients are SUMMED over ranks: the result equals the
        single-GPU gradient of the concatenated batch.  ``None``: every rank has the same number of graphs and the
        gradients are averaged (the reference's DataParallel behaviour, meta_models.py:17).

        ``canvas_dtype``: element type of the canvas and of the ``canvas_grad`` that ``step`` takes (``torch.float32``,
        ``torch.bfloat16`` or ``torch.float16``), e.g. the dtype a mixed-precision generator consumes it in.

        ``mask_size``: 0 (default) composites the canvas from the GT boxes alone (boxes_to_layout).  A power of two
        builds the model with its mask head (model.py:62-75) and composites masks_to_layout on the GT boxes with the
        PREDICTED masks, as the reference trains on datasets without GT masks (meta_models.py:48, VG): the canvas
        gradient then reaches the generator's embedding, the mask head and, through it, the GCN.  The head's BatchNorm
        normalises over the rows of the ragged batch (every object of the batch, ``__image__`` dummies included) and
        updates its running buffers on the device inside the step, so a CUDA-graph replay updates them as an eager
        step does.  With ``distributed``, the statistics and running buffers are per rank (DataParallel's per-replica
        behaviour), so ``global_batch`` sharding no longer reproduces the single-GPU gradient of the whole batch.

        ``gt_masks=True`` (needs ``mask_size > 0``): the reference's path for datasets WITH GT masks (COCO).  Every batch
        carries ``masks [NO, M, M]`` (``HostBatch(..., with_masks=True)``; fp32 or int64); the canvas is masks_to_layout
        on the GT boxes with those masks (its gradient reaches the generator's embedding only), and the step's loss is
        the box term plus ``mask_loss_weight * BCE(masks_pred, masks)`` (``model.mask_pred_loss``), which trains the head
        and, through it, the GCN.  ``mask_loss_weight = 0`` still runs the head's forward (BatchNorm buffers update as in
        the reference's forward) but adds no term: the head's parameters get no gradient.  With ``global_batch`` the mask
        term is scaled by B_local / B_global as the box term (not exact: the element count differs per rank)."""
        if gt_masks and int(mask_size) <= 0:
            raise ValueError("gt_masks=True needs a mask head (mask_size > 0)")
        if canvas_dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise ValueError("canvas_dtype must be torch.float32, torch.bfloat16 or torch.float16")
        self.canvas_dtype = canvas_dtype
        self.vocab, self.device, self.H, self.W = vocab, device, H, W
        self.flags = (learned_converse, learned_transitivity)
        self.mask_size = int(mask_size)
        self.gt_masks, self.mask_loss_weight = bool(gt_masks), float(mask_loss_weight)
        self.model = Sg2LayoutModel(build_opt(vocab, mask_size=self.mask_size), precision=precision).to(device)
        st = {k: torch.from_numpy(v) for k, v in synth.make_state(vocab, seed=seed).items()}
        for i in range(len(self.model.gconvs)):
            st["gconvs.%d.predicates_transitive_weights" % i] = st["trans_candidates_weights"]
        if self.mask_size > 0:
            st.update({k: torch.from_numpy(np.asarray(v)) for k, v in
                       synth.make_mask_state(self.model.args["gconv_dim"], self.mask_size, seed=seed).items()})
        self.model.load_state_dict(st, strict=True)
        # the generator's own object embedding (generator.py:16), the source of the canvas vectors (generator.py:80)
        opt = build_opt(vocab)
        self.layout_embedding = AttributeEmbeddings(opt.vocab["attributes"], opt.embedding_dim).to(device)
        self.layout_embedding.load_state_dict(
            {k: torch.from_numpy(v) for k, v in synth.make_layout_state(vocab, opt.embedding_dim, seed=seed).items()},
            strict=True)
        self.bbox_pred_loss_weight = bbox_pred_loss_weight
        self.last_masks = None         # masks_pred of the last eager forward (mask_size > 0)
        self.last_mask_loss = None     # mask term of the last eager forward (gt_masks, mask_loss_weight != 0)
        self.refresh_tables()
        # gradient buckets in the order they complete: box_net, gconvs 4..0, then embeddings + shared weights
        layers = list(self.model.gconvs)
        buckets = [list(self.model.box_net.parameters())]
        if self.model.mask_net is not None:      # the head's gradients are final together with box_net's
            buckets[0] += list(self.model.mask_net.parameters())
        for layer in reversed(layers):
            buckets.append([p for n, p in layer.named_parameters() if "predicates_transitive_weights" not in n])
        buckets.append(list(self.model.attribute_embedding.parameters()) + list(self.model.pred_embeddings.parameters())
                       + [self.model.trans_candidates_weights] + list(self.layout_embedding.parameters()))
        self.global_batch = global_batch
        self.reducer = (BucketedGradAllReduce(buckets, average=global_batch is None,
                                              launch_groups=self._launch_groups(len(buckets)))
                        if distributed else None)
        self.tail_events = None      # set to [] to time the part of the all-reduce that trails the backward pass
        # CUDA-graph replay of forward + backward (see _step_graphed): one captured graph per (batch buffers, sizes)
        self.use_graph = use_graph
        self.side = torch.cuda.Stream(device=device)     # look-ahead stream: uploads and counting passes of the next batch
        self._opt_done = None          # event of an optimizer step that was issued on the look-ahead stream
        self.branch = torch.cuda.Stream(device=device)   # the canvas branch of forward / backward (see forward())
        # (the bucketed gradient all-reduce copes with gradients that become final on the branch stream: reducer.home)
        self.overlap_canvas = os.environ.get("CSG_OVERLAP_CANVAS", "1") != "0"
        self._graphs = {}
        self.graph_replays = 0
        self.graph_launches = 0
        self._eager_steps = 0
        params = [p for p in self.model.parameters() if p is not self.model.converse_candidates_weights]
        params += list(self.layout_embedding.parameters())
        self.opt = FusedAdam(params, lr=lr)                      # torch.optim.Adam arithmetic, one multi-tensor launch
        # 16-bit copies of all layers' weights: one cast launch behind every optimizer step instead of one per layer and forward
        self.opt.post_step.append(self.model.refresh_weight_copies)
        self.model.refresh_weight_copies()

    @staticmethod
    def _launch_groups(nb):
        """Which gradient buckets are all-reduced by one coalesced NCCL launch (``BucketedGradAllReduce.launch_groups``).
        ``CSG_GRAD_GROUPS``: ``layers`` (default) = one launch per bucket, ``two`` = [box_net, gconv 4..1] as soon as
        layer 1's gradients are final + [gconv 0, embeddings, shared weights] at the end, ``end`` = one launch behind
        the backward pass.  Measured on one 8-GPU box (cfg2, weak scaling, ms per step): N = 2: 4.59 / 4.52 / 4.51,
        N = 8: 4.60 / 4.62 / 4.59 for layers / two / end against 4.40 at N = 1 -- the grouping is worth < 2 % at N = 2 and
        nothing at N = 8, i.e. the N = 1 -> N = 8 gap is not the number of collective launches (DESIGN.md section 5)."""
        mode = os.environ.get("CSG_GRAD_GROUPS", "layers")
        if mode == "layers" or nb < 3:
            return None
        if mode == "end":
            return [list(range(nb))]
        return [list(range(nb - 2)), [nb - 2, nb - 1]]

    def refresh_tables(self):
        """The reference pushes the symmetrised converse weights into the dataset every step
        (train.py:311-313); the CDF table is rebuilt from them here."""
        W = get_conv_converse(self.model).detach().double().cpu().numpy()
        cdf, vals = converse_tables(W, self.vocab.num_preds, self.vocab.meta_ids)
        self.tables = (torch.from_numpy(cdf).to(self.device), torch.from_numpy(vals).to(self.device))

    def prefetch(self, d):
        """Launch the counting pass of the canonicalization of batch ``d`` now (no host wait); ``step(d, ...)``
        later finds the output sizes on the host.  The reference canonicalizes in DataLoader workers ahead of the
        training step (base_dataset.py:89-139 inside ``__getitem__``); this is the same look-ahead on the device, on
        its own stream (``self.side``): the pass (one CTA per graph, ~40 us) then runs beside the kernels of the step in
        flight instead of in front of them."""
        side = self.side
        ready = d.get("_ready")
        if ready is not None:
            side.wait_event(ready)                 # upload of `d` (HostBatch.to_device(stream=...))
        else:
            side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            d["_canon_plan"] = canon_count_async(d["triplets"], d["tri_off"], d["obj_off"], self.vocab.num_preds,
                                                 self.vocab.meta_ids, None, self.flags[0], self.flags[1], d["uniforms"],
                                                 max_objs_per_graph=d["max_objs"], tables=self.tables)

    def canonicalize(self, d):
        if d.get("_canon_plan") is None:
            self.prefetch(d)
        return canon_emit(d.pop("_canon_plan"))

    def _gt_masks(self, d):
        masks = d.get("masks")
        if masks is None:
            raise ValueError("gt_masks=True needs the batch's GT masks d['masks'] [NO, M, M] (HostBatch(with_masks=True))")
        want = (int(d["objs"].shape[0]), self.mask_size, self.mask_size)
        if tuple(masks.shape) != want:
            raise ValueError("d['masks'] is %s, expected %s" % (tuple(masks.shape), want))
        return masks

    def forward(self, d, res):
        # canvas: the generator's own embedding of the objects on the GT boxes (train.py:358, generator.py:80-96).
        # remove_dummy_objects (utils.py:56-63) needs no filtering pass: the __image__ dummy has box -1 and
        # contributes exact zeros to the canvas and receives an exactly zero gradient.
        # The canvas branch shares nothing with the GCN but the batch, so it is issued on its own stream: autograd runs
        # a node's backward on the stream of its forward, so both the compositor (bandwidth-bound, every SM) and its
        # backward run beside the GCN's latency-bound first / last kernels (triple index + CSR build, box head) -- as a
        # parallel branch of the captured graph under CUDA-graph replay.
        # With GT masks (gt_masks) the canvas does not depend on the head: it is issued up front as well, and the head
        # runs on the main stream for the mask loss only.
        gt = self._gt_masks(d) if self.gt_masks else None
        main = torch.cuda.current_stream()
        branch = self.branch if self.overlap_canvas else main
        if branch is not main:
            branch.wait_stream(main)
        with torch.cuda.stream(branch):
            layout_vecs = self.layout_embedding(d["objs"])
            if self.mask_size == 0 or gt is not None:
                canvas = layout_batched(layout_vecs, d["boxes"], d["obj_off"], self.H, self.W, masks=gt,
                                        max_objs_per_image=d["max_objs"], out_dtype=self.canvas_dtype)
        obj_vecs, boxes_pred = self.model.forward_ragged(d["objs"], res.triplets, res.triplet_type, res.tri_off,
                                                         d["obj_off"])
        mask_loss = None
        if gt is not None:
            if self.mask_loss_weight == 0:
                with torch.no_grad():          # BatchNorm buffers still update; nothing to differentiate
                    masks_pred = self.model.masks_from_vecs(obj_vecs)
            else:
                masks_pred = self.model.masks_from_vecs(obj_vecs)
                mw = self.mask_loss_weight
                if self.global_batch is not None:
                    mw = mw * d["B"] / float(self.global_batch)
                mask_loss = mask_pred_loss(masks_pred, gt, mw)
            self.last_masks = masks_pred.detach()
        elif self.mask_size > 0:
            # predicted masks (meta_models.py:48): the compositor waits for the head; the embedding lookup above stayed
            # on the branch stream
            masks_pred = self.model.masks_from_vecs(obj_vecs)
            if branch is not main:
                branch.wait_stream(main)
            with torch.cuda.stream(branch):
                canvas = layout_batched(layout_vecs, d["boxes"], d["obj_off"], self.H, self.W, masks=masks_pred,
                                        max_objs_per_image=d["max_objs"], out_dtype=self.canvas_dtype)
            self.last_masks = masks_pred.detach()
        if branch is not main:
            main.wait_stream(branch)
        weight = self.bbox_pred_loss_weight
        if self.global_batch is not None:
            weight = weight * d["B"] / float(self.global_batch)
        loss, _ = bbox_pred_loss_ragged(boxes_pred, d["boxes"], d["objs"], d["obj_off"], weight)   # pix2pix_model.py:72-85
        if mask_loss is not None:
            self.last_mask_loss = mask_loss.detach()
            loss = loss + mask_loss
        return canvas, loss

    def backward(self, d, canvas_grad, prefetch=None):
        """Canonicalization + forward + backward (+ the gradient all-reduce): leaves the final gradients in ``.grad``."""
        res = self.canonicalize(d)
        if prefetch is not None:
            self.prefetch(prefetch)
        if self.reducer is not None:
            self.reducer.home = torch.cuda.current_stream()
        canvas, loss = self.forward(d, res)
        torch.autograd.backward([canvas, loss], [canvas_grad, None])
        if self.reducer is not None:
            if self.tail_events is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                self.reducer.finish()
                e1.record()
                self.tail_events.append((e0, e1))
            else:
                self.reducer.finish()
        return loss, int(res.triplets.shape[0])

    # ------------------------------------------------------------------------------------------ CUDA-graph replay
    # Everything after the canonicalization emit pass has static shapes once the canonicalized triple count is known
    # (the one host read of a step).  The ~150 launches of forward + backward then cost more HOST time (Python, ctypes,
    # cudaLaunchKernelEx: ~5 us each) than the device needs to run them, so the device idles ~10 % of a step.  A step
    # whose (input buffers, object / triple counts) were seen before replays a captured graph instead: one
    # cudaGraphLaunch for the whole forward + backward (+ gradient all-reduce).  The graph reads the batch from the
    # buffers it was captured on (a data pipeline cycles through a fixed set of device batch buffers, two in bench.py's
    # end-to-end leg) and the canonicalized triples from buffers owned by the cache entry, which the eager emit pass
    # fills right before the replay.  A step with a new key is captured (and replayed once); a triple count never seen
    # on these buffers simply captures another graph, up to `max_graphs`, then falls back to eager launches.
    max_graphs = 8

    def _graph_key(self, d, G, total):
        # with GT masks the captured graph reads them from the batch's masks buffer too
        masks = d.get("masks") if self.gt_masks else None
        return (int(total), int(d["objs"].shape[0]), int(d["B"]), int(d["max_objs"]), d["objs"].data_ptr(),
                d["boxes"].data_ptr(), d["obj_off"].data_ptr(), G.data_ptr(), tuple(G.shape),
                None if masks is None else (masks.data_ptr(), masks.dtype))

    def _capture(self, key, d, G, plan, total):
        dev = self.device
        ent = {"triplets": torch.empty((max(total, 1), 3), dtype=torch.int64, device=dev),
               "types": torch.empty(max(total, 1), dtype=torch.int64, device=dev),
               "tri_off": torch.empty(d["B"] + 1, dtype=torch.int32, device=dev),
               "keep": (d["objs"], d["boxes"], d["obj_off"], G, d.get("masks") if self.gt_masks else None)}
        res = canon_emit(plan, out=(ent["triplets"], ent["types"]))
        ent["tri_off"].copy_(res.tri_off)
        from .canonicalize import CanonResult
        static = CanonResult(ent["triplets"][:total], ent["types"][:total], ent["tri_off"], res.conv_counts)
        params = list(self.opt.params)
        for p in params:
            p.grad = None
        torch.cuda.synchronize()
        from .ops import lib
        launches0 = lib().csg_launch_count()
        graph = torch.cuda.CUDAGraph()
        try:      # the parameters' AccumulateGrad nodes predate the capture stream: expected here, not a bug to warn about
            torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
        except AttributeError:
            pass
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            if self.reducer is not None:
                self.reducer.home = torch.cuda.current_stream()       # the capture stream
            canvas, loss = self.forward(d, static)
            torch.autograd.backward([canvas, loss], [G, None])
            if self.reducer is not None:
                self.reducer.finish()
        ent.update(graph=graph, canvas=canvas, loss=loss.detach(), grads=[p.grad for p in params], total=total,
                   launches=int(lib().csg_launch_count() - launches0))
        return ent

    def _step_graphed(self, d, canvas_grad, prefetch):
        if self._eager_steps == 0:         # the first step runs eagerly: it fills the host-side caches (linspace tables,
            return None                    # scratch buffers, function attributes) that must not be created under capture
        if d.get("_canon_plan") is None:
            self.prefetch(d)
        plan = d.pop("_canon_plan")
        total = canon_total(plan)
        key = self._graph_key(d, canvas_grad, total)
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= self.max_graphs:
                d["_canon_plan"] = plan
                return None
            ent = self._graphs[key] = self._capture(key, d, canvas_grad, plan, total)
        else:
            res = canon_emit(plan, out=(ent["triplets"], ent["types"]))
            ent["tri_off"].copy_(res.tri_off)
        if prefetch is not None:
            self.prefetch(prefetch)
        main = torch.cuda.current_stream()
        if self._opt_done is not None:     # the optimizer step of the previous iteration (look-ahead stream, below)
            main.wait_event(self._opt_done)
            self._opt_done = None
        ent["graph"].replay()
        self.graph_replays += 1
        self.graph_launches += ent["launches"]      # kernel-launch sites executed by the replay (counted at capture)
        for p, g in zip(self.opt.params, ent["grads"]):
            p.grad = g
        # Adam and the refresh of the 16-bit weight copies go to the look-ahead stream: the next step's emit pass (main
        # stream, ~50 us, independent of the weights) then runs beside them instead of behind them
        self.side.wait_stream(main)
        with torch.cuda.stream(self.side):
            self.opt.step()
            self._opt_done = torch.cuda.Event()
            self._opt_done.record(self.side)
        for p in self.opt.params:          # the entry keeps its gradient buffers; an eager step must not accumulate into them
            p.grad = None
        return ent["loss"], total

    def step(self, d, canvas_grad, prefetch=None):
        """One training step on batch ``d``.  ``prefetch``: the batch of the NEXT step (may be ``d`` itself); its
        canonicalization counting pass is enqueued right behind this step's emit pass."""
        if canvas_grad.dtype != self.canvas_dtype:
            raise ValueError("canvas_grad is %s, the canvas is %s" % (canvas_grad.dtype, self.canvas_dtype))
        if self.gt_masks:
            self._gt_masks(d)                      # before any work (and outside a graph capture)
        if d.get("_ready") is not None:            # `d` was uploaded on the look-ahead stream
            torch.cuda.current_stream().wait_event(d["_ready"])
        if self.use_graph:
            out = self._step_graphed(d, canvas_grad, prefetch)
            if out is not None:
                return out
        if self._opt_done is not None:
            torch.cuda.current_stream().wait_event(self._opt_done)
            self._opt_done = None
        loss, n_tri = self.backward(d, canvas_grad, prefetch)
        self._eager_steps += 1
        self.opt.step()
        if self.reducer is not None:
            self.reducer.zero()
        else:
            self.opt.zero_grad(set_to_none=True)
        return loss.detach(), n_tri

    def finish(self):
        """Make the current stream wait for the optimizer step of the last ``step()`` call.  With CUDA-graph replay Adam
        and the refresh of the 16-bit weight copies are issued on the look-ahead stream (so that the next step's emit
        pass overlaps them); the next ``step()`` waits for them by itself, anything ELSE that reads the parameters
        (evaluation, checkpoints, tests) calls this first."""
        if self._opt_done is not None:
            torch.cuda.current_stream().wait_event(self._opt_done)

    def named_grads(self):
        out = {"model." + n: p.grad for n, p in self.model.named_parameters() if p.grad is not None}
        out.update({"layout_embedding." + n: p.grad for n, p in self.layout_embedding.named_parameters() if p.grad is not None})
        return out


class SgToLayoutInference:
    """Forward-only scene graph -> layout canvas, the call path of ``scripts/generate_clevr.py:249-301``
    (``model(objs, triplets, triplet_type, test_mode=True)``) with graph construction on the device:

        add_location_triplets + add_dummy_triplets (base_dataset.py:35-87,141-150)  ->  add_learnt_triplets (:89-139)
        ->  Sg2LayoutModel (model.py:90-124; 4 attributes -> attribute_fc_gen)  ->  generator-side embedding
        (generator.py:16,80)  ->  masks_to_layout(test_mode=True) occlusion compositor on the PREDICTED boxes
        (layout.py:48-77,135-147), dummy objects removed (utils.py:56-63)

    ``step(d)`` expects the device tensors of :class:`HostBatch` plus ``centers [NO, 2]`` and ``masks [NO, M, M]``;
    the canvas it returns has dtype ``canvas_dtype`` (fp32, or the fp32 canvas rounded once to bf16 / fp16).

    ``mask_size > 0`` builds the model with its mask head, in eval mode (BatchNorm on its running buffers): a batch
    without ``masks`` is then composited from the PREDICTED masks (``model.masks_from_vecs(obj_vecs)``, model.py:121-123),
    a batch with GT masks as before."""

    def __init__(self, vocab, device, precision="fp16", H=256, W=256, embedding_dim=32, attr_sizes=None,
                 learned_converse=True, learned_transitivity=True, seed=0, canvas_dtype=torch.float32, mask_size=0):
        import argparse
        if canvas_dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise ValueError("canvas_dtype must be torch.float32, torch.bfloat16 or torch.float16")
        self.canvas_dtype = canvas_dtype
        self.vocab, self.device, self.H, self.W = vocab, device, H, W
        self.flags = (learned_converse, learned_transitivity)
        A = vocab.num_attributes
        sizes = attr_sizes or [vocab.num_obj_classes if A == 1 else 8] * A
        attrs = {"a%d" % i: {str(j): j for j in range(sizes[i])} for i in range(A)}
        opt = argparse.Namespace(
            vocab={"attributes": attrs, "pred_idx_to_name": vocab.pred_names, "pred_name_to_idx": vocab.pred_ids},
            embedding_dim=embedding_dim, gconv_dim=128, gconv_hidden_dim=512, gconv_pooling="avg", gconv_num_layers=5,
            mlp_normalization="none", mask_size=int(mask_size), learned_init="uniform")
        self.mask_size = int(mask_size)
        self.model = Sg2LayoutModel(opt, precision=precision).to(device)
        st = {k: torch.from_numpy(v) for k, v in
              synth.make_state(vocab, embedding_dim=embedding_dim, seed=seed, attr_vocab_sizes=sizes).items()}
        for i in range(len(self.model.gconvs)):
            st["gconvs.%d.predicates_transitive_weights" % i] = st["trans_candidates_weights"]
        if self.mask_size > 0:
            st.update({k: torch.from_numpy(np.asarray(v)) for k, v in
                       synth.make_mask_state(opt.gconv_dim, self.mask_size, seed=seed).items()})
        self.model.load_state_dict(st, strict=True)
        if self.mask_size > 0:
            self.model.eval()
        self.layout_embedding = AttributeEmbeddings(attrs, embedding_dim).to(device)
        self.layout_embedding.load_state_dict(
            {k: torch.from_numpy(v) for k, v in
             synth.make_layout_state(vocab, embedding_dim, seed=seed, attr_vocab_sizes=sizes).items()}, strict=True)
        Wc = get_conv_converse(self.model).detach().double().cpu().numpy()
        cdf, vals = converse_tables(Wc, vocab.num_preds, vocab.meta_ids)
        self.tables = (torch.from_numpy(cdf).to(device), torch.from_numpy(vals).to(device))

    @torch.no_grad()
    def build_graph(self, d):
        """Location + dummy triplets on the device, then the WSGC completion."""
        from .canonicalize import add_location_triplets_batched, add_learnt_triplets_batched
        v = self.vocab
        trip, tri_off = add_location_triplets_batched(d["boxes"], d["centers"], d["objs"], d["obj_off"], v.image_obj_id,
                                                      v.pred_ids, max_objs_per_graph=d["max_objs"],
                                                      in_image_pred=v.in_image_id)
        if d["uniforms"].numel() < trip.shape[0]:
            raise ValueError("need one converse draw per input triple (%d > %d)" % (trip.shape[0], d["uniforms"].numel()))
        return add_learnt_triplets_batched(trip, tri_off, d["obj_off"], v.num_preds, v.meta_ids, None, self.flags[0],
                                           self.flags[1], d["uniforms"], max_objs_per_graph=d["max_objs"],
                                           tables=self.tables)

    @torch.no_grad()
    def step(self, d):
        res = self.build_graph(d)
        obj_vecs, boxes_pred = self.model.forward_ragged(d["objs"], res.triplets, res.triplet_type, res.tri_off,
                                                         d["obj_off"])
        # the __image__ dummy is removed from the canvas (utils.py:56-63): a box of -1 samples nothing
        dummy = (d["objs"][:, :1] == 0)
        boxes = torch.where(dummy, torch.full_like(boxes_pred, -1.0), boxes_pred.float())
        masks = d.get("masks")
        if masks is None:
            if self.mask_size == 0:
                raise ValueError("a batch without masks needs a model with a mask head (mask_size > 0)")
            masks = self.model.masks_from_vecs(obj_vecs)
        canvas = layout_batched(self.layout_embedding(d["objs"]), boxes, d["obj_off"], self.H, self.W, masks=masks,
                                test_mode=True, out_dtype=self.canvas_dtype)
        return canvas, boxes_pred, int(res.triplets.shape[0])
