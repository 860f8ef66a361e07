"""CPU side of the predicted-mask pipelines: the seeded mask-head state loads into Sg2LayoutModel(mask_size > 0) with
strict=True under the reference's keys, follows the documented init law, and mask_size = 0 builds today's model."""
import numpy as np
import torch

from canonicalsg2im_b200 import synth
from canonicalsg2im_b200.model import Sg2LayoutModel
from canonicalsg2im_b200.pipeline import build_opt


def _full_state(vocab, mask_size):
    st = {k: torch.from_numpy(v) for k, v in synth.make_state(vocab, seed=0).items()}
    for i in range(5):
        st["gconvs.%d.predicates_transitive_weights" % i] = st["trans_candidates_weights"]
    if mask_size:
        st.update({k: torch.from_numpy(np.asarray(v)) for k, v in synth.make_mask_state(128, mask_size, seed=0).items()})
    return st


def test_mask_state_loads_strict():
    vocab = synth.Vocab(42)
    for M in (2, 16):
        model = Sg2LayoutModel(build_opt(vocab, mask_size=M))
        model.load_state_dict(_full_state(vocab, M), strict=True)
        assert model.mask_net is not None
    model = Sg2LayoutModel(build_opt(vocab))
    assert model.mask_net is None
    model.load_state_dict(_full_state(vocab, 0), strict=True)


def test_mask_state_law_and_seed():
    st = synth.make_mask_state(128, 16, seed=0)
    assert set(st) == {"mask_net." + k for k in Sg2LayoutModel(build_opt(synth.Vocab(42), mask_size=16)).mask_net
                       .state_dict()}
    for k, v in st.items():
        if k.endswith("num_batches_tracked"):
            assert int(v) == 0
        elif k.endswith("running_var") or (k.endswith("weight") and v.ndim == 1):
            assert v.min() >= 0.5 and v.max() < 1.5, k
        elif k.endswith("running_mean") or k.endswith("bias"):
            assert np.abs(v).max() <= 0.2, k
        else:
            assert np.abs(v).max() <= np.sqrt(3.0 / np.prod(v.shape[1:])), k
    other = synth.make_mask_state(128, 16, seed=1)
    assert not np.array_equal(st["mask_net.2.weight"], other["mask_net.2.weight"])
    again = synth.make_mask_state(128, 16, seed=0)
    assert all(np.array_equal(np.asarray(st[k]), np.asarray(again[k])) for k in st)
