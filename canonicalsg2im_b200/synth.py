"""Seeded synthetic scene graphs and weights (SURVEY.md §8(d)).

Everything here is host-side input generation for tests and ``bench.py``: it
is reproducible from integers alone (splitmix64 hashing, no dependence on a
torch/numpy RNG stream), so the GPU box regenerates exactly the tensors the
golden fixtures were made with.  Shapes and vocabularies follow the
reference's packed datasets:

* relation ids: dataset predicates first, then ``__padding__``,
  ``__in_image__`` and the six spatial relations
  (``sg2im/data/base_dataset.py:14-15,152-161``);
* boxes are ``[x0, y0, w, h]`` in [0, 1] (``sg2im/layout.py:95-96``), the
  ``__image__`` dummy object has class 0 and box ``-1``
  (``sg2im/data/packed_coco.py:325-329``);
* base triples are the minimal per-relation spatial triples of
  ``add_location_triplets`` (``base_dataset.py:35-87``) plus the
  ``__in_image__`` dummies (``:141-150``).
"""
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

META_RELATIONS = ("__padding__", "__in_image__")
AUGMENTED_RELATIONS = ("__below__", "__above__", "__left of__", "__right of__",
                       "__inside__", "__surrounding__")

CLEVR_ATTR_SIZES = (4, 9, 3, 3)     # vocabulary sizes of CLEVR's shape / color / material / size (+ 0 = none)

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _splitmix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
    z = x
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
    return z ^ (z >> np.uint64(31))


def det_uniform(n, seed):
    """n float64 values in [0, 1), a pure function of (seed, index)."""
    with np.errstate(over="ignore"):
        idx = np.arange(n, dtype=np.uint64)
        base = _splitmix64(np.full(1, seed, dtype=np.uint64) * np.uint64(0x2545F4914F6CDD1D))[0]
        h = _splitmix64(idx ^ base)
    return (h >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def det_tensor(shape, seed, scale=1.0):
    """float32 tensor with entries uniform in [-scale, scale)."""
    n = int(np.prod(shape)) if len(shape) else 1
    u = det_uniform(n, seed)
    return ((u * 2.0 - 1.0) * scale).astype(np.float32).reshape(shape)


def det_int(n, seed, lo, hi):
    """n int64 values uniform in [lo, hi]."""
    return (lo + np.floor(det_uniform(n, seed) * (hi - lo + 1))).astype(np.int64)


# ----------------------------------------------------------------------------
# vocabularies
# ----------------------------------------------------------------------------
@dataclass
class Vocab:
    num_base_preds: int = 0                 # 0: COCO/CLEVR packed (P=8); 42: VG-like (P=50)
    num_obj_classes: int = 184              # class 0 == __image__ / padding
    num_attributes: int = 1                 # 1: COCO/VG 'objects'; 4: CLEVR shape/color/material/size

    @property
    def pred_names(self):
        return ["pred_%d" % i for i in range(self.num_base_preds)] + \
            list(META_RELATIONS) + list(AUGMENTED_RELATIONS)

    @property
    def num_preds(self):
        return self.num_base_preds + 8

    @property
    def pred_ids(self):
        return {n: i for i, n in enumerate(self.pred_names)}

    @property
    def padding_id(self):
        return self.num_base_preds

    @property
    def in_image_id(self):
        return self.num_base_preds + 1

    @property
    def meta_ids(self):
        return (self.padding_id, self.in_image_id)

    @property
    def image_obj_id(self):
        return 0


# ----------------------------------------------------------------------------
# spatial triples (fast host version of add_location_triplets, for generation)
# ----------------------------------------------------------------------------
def _closure(adj):
    p = adj.copy()
    for i in range(p.shape[0]):
        absorb = p[:, i].copy()
        absorb[i] = False
        p[absorb] |= p[i]
    return p


def location_triplets(boxes, centers, real, vocab: Vocab):
    """Minimal per-relation spatial triples in the reference's emission order
    (``base_dataset.py:35-87``).  ``real`` lists the indices of real objects.
    Spatial relations built from strict comparisons are acyclic, for which
    the reference's sequential reduction equals ``C & ~(C @ C)``; relations
    with fewer than three raw triples are passed through unreduced."""
    boxes = np.asarray(boxes, dtype=np.float32)
    cen = np.asarray(centers, dtype=np.float32)
    real = np.asarray(real, dtype=np.int64)
    n = len(boxes)
    ids = vocab.pred_ids
    out = []
    if len(real) < 2:
        return np.zeros((0, 3), dtype=np.int64)
    x0, y0 = boxes[:, 0], boxes[:, 1]
    xc = x0 + boxes[:, 2] / np.float32(2)
    yc = y0 + boxes[:, 3] / np.float32(2)
    isreal = np.zeros(n, dtype=bool)
    isreal[real] = True
    pair = isreal[:, None] & isreal[None, :] & ~np.eye(n, dtype=bool)
    S, O = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    sur = (x0[S] < x0[O]) & (xc[S] > xc[O]) & (y0[S] < y0[O]) & (yc[S] > yc[O]) & pair
    ins = (x0[S] > x0[O]) & (xc[S] < xc[O]) & (y0[S] > y0[O]) & (yc[S] < yc[O]) & pair & ~sur
    rest = pair & ~sur & ~ins
    dx = cen[S, 0] - cen[O, 0]
    dy = cen[S, 1] - cen[O, 1]
    rel = {
        "__surrounding__": sur, "__inside__": ins,
        "__right of__": rest & (dx > 0), "__left of__": rest & (dx < 0),
        "__below__": rest & (dy > 0), "__above__": rest & (dy < 0),
    }
    for name in AUGMENTED_RELATIONS:
        a = rel[name]
        cnt = int(a.sum())
        if cnt == 0:
            continue
        if cnt >= 3:
            # adjacency is sized max index + 1 in the reference; cells outside are empty anyway
            c = _closure(a)
            a = c & ~((c.astype(np.int32) @ c.astype(np.int32)) > 0)
        r, cix = np.nonzero(a)
        t = np.stack([r, np.full_like(r, ids[name]), cix], axis=1)
        out.append(t)
    return np.concatenate(out, axis=0).astype(np.int64) if out else np.zeros((0, 3), dtype=np.int64)


# ----------------------------------------------------------------------------
# graphs
# ----------------------------------------------------------------------------
@dataclass
class Graph:
    objs: np.ndarray            # [O, A] int64 (last row = __image__ dummy when include_dummies)
    boxes: np.ndarray           # [O, 4] float32 xywh (dummy = -1)
    centers: np.ndarray         # [O_real, 2] float32
    triplets: np.ndarray        # [T, 3] int64 base triples (before add_learnt_triplets)
    masks: Optional[np.ndarray] = None   # [O, M, M] int64


def make_graph(seed, n_min, n_max, vocab: Vocab, include_dummies=True, box_mode="coco",
               mask_size=0, extra_pred_triples=True) -> Graph:
    n = int(det_int(1, seed * 7 + 1, n_min, n_max)[0])
    A = vocab.num_attributes
    if A == 1:
        objs = det_int(n, seed * 7 + 2, 1, vocab.num_obj_classes - 1).reshape(n, 1)
    else:
        objs = det_int(n * A, seed * 7 + 2, 1, 7).reshape(n, A)
    u = det_uniform(4 * n, seed * 7 + 3).reshape(n, 4)
    if box_mode == "clevr":      # packed_clevr_dialog.py:487-498: sizes in {0.1, 0.2}
        s = np.where(u[:, 2] < 0.5, 0.1, 0.2)
        w, h = s, s
    else:
        w = 0.15 + 0.45 * u[:, 2]
        h = 0.15 + 0.45 * u[:, 3]
    x0 = u[:, 0] * (1.0 - w)
    y0 = u[:, 1] * (1.0 - h)
    boxes = np.stack([x0, y0, w, h], axis=1).astype(np.float32)
    centers = np.stack([boxes[:, 0] + np.float32(0.5) * boxes[:, 2],
                        boxes[:, 1] + np.float32(0.5) * boxes[:, 3]], axis=1).astype(np.float32)
    masks = None
    if mask_size:
        masks = (det_uniform(n * mask_size * mask_size, seed * 7 + 4) < 0.6).astype(np.int64)
        masks = masks.reshape(n, mask_size, mask_size)
    real = np.arange(n)
    if include_dummies:
        objs = np.concatenate([objs, np.zeros((1, A), dtype=np.int64)], axis=0)
        boxes = np.concatenate([boxes, -np.ones((1, 4), dtype=np.float32)], axis=0)
        if masks is not None:
            masks = np.concatenate([masks, np.ones((1, mask_size, mask_size), dtype=np.int64)], axis=0)
    trip = [location_triplets(boxes, np.concatenate([centers, np.zeros((len(boxes) - n, 2), np.float32)]),
                              real, vocab)]
    if vocab.num_base_preds and extra_pred_triples and n >= 2:
        k = n
        s = det_int(k, seed * 7 + 5, 0, n - 1)
        o = (s + det_int(k, seed * 7 + 6, 1, n - 1)) % n
        p = det_int(k, seed * 7 + 8, 0, vocab.num_base_preds - 1)
        trip.append(np.stack([s, p, o], axis=1))
    if include_dummies:
        trip.append(np.stack([real, np.full(n, vocab.in_image_id), np.full(n, n)], axis=1))
    return Graph(objs=objs, boxes=boxes, centers=centers,
                 triplets=np.concatenate(trip, axis=0).astype(np.int64), masks=masks)


def make_graphs(num, seed, n_min, n_max, vocab, **kw) -> List[Graph]:
    return [make_graph(seed * 100003 + i, n_min, n_max, vocab, **kw) for i in range(num)]


def make_conv_weights(vocab: Vocab, seed=0):
    """Symmetrised converse weights (``sg2im/model.py:13-14``) from U(-1, 1)
    (``sg2im/graph.py:116-118``), float64 as the dataset sees them."""
    P = vocab.num_preds
    w = det_tensor((P, P), seed * 31 + 5, 1.0).astype(np.float64)
    tri = np.triu(w)
    return tri + tri.T


# ----------------------------------------------------------------------------
# weights with the reference's state-dict keys
# ----------------------------------------------------------------------------
def make_state(vocab: Vocab, embedding_dim=128, gconv_dim=128, hidden_dim=512, num_layers=5,
               seed=0, attr_vocab_sizes=None):
    """Random-init weights of ``Sg2LayoutModel`` (``sg2im/model.py:18-60``) keyed like its
    state dict.  Linear weights are uniform with Kaiming-normal variance
    (2 / fan_in, ``sg2im/graph.py:11-14``), biases U(-1/sqrt(fan_in), ..)."""
    st = {}
    k = [seed * 1009 + 11]

    def nxt():
        k[0] += 1
        return k[0]

    def lin(name, out_f, in_f):
        st[name + ".weight"] = det_tensor((out_f, in_f), nxt(), float(np.sqrt(6.0 / in_f)))
        st[name + ".bias"] = det_tensor((out_f,), nxt(), float(1.0 / np.sqrt(in_f)))

    A = vocab.num_attributes
    sizes = attr_vocab_sizes or [vocab.num_obj_classes if A == 1 else 8] * A
    for a in range(A):
        st["attribute_embedding.att_emb_%d.weight" % a] = det_tensor((sizes[a], embedding_dim), nxt(), 1.0)
    if A > 1:
        lin("attribute_embedding.attribute_fc_gen", A * embedding_dim, A * embedding_dim)
    P = vocab.num_preds
    st["pred_embeddings.weight"] = det_tensor((P, embedding_dim), nxt(), 1.0)
    st["trans_candidates_weights"] = det_tensor((P,), nxt(), 1.0)
    st["converse_candidates_weights"] = det_tensor((P, P), nxt(), 1.0)
    d_obj, d_pred = A * embedding_dim, embedding_dim
    for i in range(num_layers):
        pre = "gconvs.%d." % i
        lin(pre + "net1.0", hidden_dim, 2 * d_obj + d_pred)
        lin(pre + "net1.2", 2 * hidden_dim + gconv_dim, hidden_dim)
        lin(pre + "net2.0", hidden_dim, hidden_dim)
        lin(pre + "net2.2", gconv_dim, hidden_dim)
        d_obj, d_pred = gconv_dim, gconv_dim
    lin("box_net.0", hidden_dim, gconv_dim)
    lin("box_net.2", 4, hidden_dim)
    return st


def make_layout_state(vocab: Vocab, embedding_dim=128, seed=0, attr_vocab_sizes=None):
    """Random-init weights of the generator-side ``AttributeEmbeddings`` (``spade/models/networks/generator.py:16``),
    the table the training canvas is composited from (``generator.py:80``), keyed like that module's state dict."""
    st = {}
    A = vocab.num_attributes
    sizes = attr_vocab_sizes or [vocab.num_obj_classes if A == 1 else 8] * A
    k = seed * 2003 + 501
    for a in range(A):
        k += 1
        st["att_emb_%d.weight" % a] = det_tensor((sizes[a], embedding_dim), k, 1.0)
    if A > 1:
        n = A * embedding_dim
        st["attribute_fc_gen.weight"] = det_tensor((n, n), k + 1, float(np.sqrt(6.0 / n)))
        st["attribute_fc_gen.bias"] = det_tensor((n,), k + 2, float(1.0 / np.sqrt(n)))
    return st


def make_mask_state(gconv_dim=128, mask_size=16, seed=0):
    """Random-init weights and running buffers of the mask head (``sg2im/model.py:62-75``, ``mask_size > 0``) keyed like
    ``Sg2LayoutModel``'s state dict (``mask_net.*``).  BatchNorm weights and running variances are uniform in
    [0.5, 1.5), running means and all biases in [-0.2, 0.2), convolution weights in +-sqrt(3 / fan_in);
    ``num_batches_tracked`` starts at 0."""
    from .mask_head import build_mask_net
    st = {}
    k = seed * 3001 + 907
    for name, v in build_mask_net(gconv_dim, mask_size).state_dict().items():
        k += 1
        shape = tuple(v.shape)
        if name.endswith("num_batches_tracked"):
            st["mask_net." + name] = np.zeros((), np.int64)
        elif name.endswith("running_var") or (v.dim() == 1 and name.endswith("weight")):
            st["mask_net." + name] = det_tensor(shape, k, 0.5) + np.float32(1.0)
        elif name.endswith("running_mean") or name.endswith("bias"):
            st["mask_net." + name] = det_tensor(shape, k, 0.2)
        else:
            fan_in = int(np.prod(shape[1:]))
            st["mask_net." + name] = det_tensor(shape, k, float(np.sqrt(3.0 / fan_in)))
    return st
