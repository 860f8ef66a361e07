"""CPU side of the GT-mask training path: the restated mask loss (tests/mask_loss_ref.py) follows the formula the CUDA
kernel implements, saturated tails included; the step rejects gt_masks=True without a mask head before any CUDA work;
HostBatch's with_masks switch."""
import numpy as np
import pytest
import torch

from canonicalsg2im_b200 import synth
from canonicalsg2im_b200.pipeline import HostBatch, SgToLayoutStep
from tests.mask_loss_ref import mask_pred_loss


def _formula(p, t, w):
    p, t = np.asarray(p, np.float64), np.asarray(t, np.float64)
    with np.errstate(divide="ignore"):
        el = -(t * np.maximum(np.log(p), -100) + (1 - t) * np.maximum(np.log1p(-p), -100))
    eps = float(np.float32(1e-12))          # torch's clamp is the float constant 1e-12f, in float64 too
    return w * el.mean(), w * (p - t) / np.maximum((1 - p) * p, eps) / p.size


@pytest.mark.parametrize("soft", [False, True])
def test_reference_matches_formula(soft):
    g = torch.Generator().manual_seed(0)
    p = torch.rand((7, 16, 16), generator=g, dtype=torch.float64)
    t = torch.rand(p.shape, generator=g, dtype=torch.float64)
    if not soft:
        t = (t < 0.6).to(torch.int64)
    p[0, 0, :4] = torch.tensor([0.0, 1.0, 1e-13, 1 - 2.0 ** -24], dtype=torch.float64)      # clamped tails
    x = p.clone().requires_grad_()
    loss = mask_pred_loss(x, t, 2.5)
    loss.backward()
    ref_loss, ref_grad = _formula(p.numpy(), t.numpy(), 2.5)
    assert abs(loss.item() - ref_loss) <= 1e-12 * abs(ref_loss)
    np.testing.assert_allclose(x.grad.numpy(), ref_grad, rtol=1e-12, atol=0)


def test_saturated_tails_through_sigmoid():
    """sigmoid(z) then BCE against t = 0 in float32 (torch 2.11): p rounds to exactly 1 at z = 17, 20, 40, the loss
    saturates at the -100 clamp and d/dz is exactly 0; at z = -30 d/dz is p (1 - p) / max((1 - p) p, 1e-12) p = 8.76e-15,
    not the logit-form p = 9.36e-14."""
    z = torch.tensor([17.0, 20.0, 40.0, -30.0], requires_grad=True)
    p = z.sigmoid()
    el = torch.stack([mask_pred_loss(p[i:i + 1], torch.zeros(1)) for i in range(4)])
    el.sum().backward()
    assert p[:3].tolist() == [1.0, 1.0, 1.0]
    assert el[:3].tolist() == [100.0, 100.0, 100.0]
    assert z.grad[:3].tolist() == [0.0, 0.0, 0.0]
    assert abs(z.grad[3].item() - 8.7565e-15) <= 1e-18
    assert abs(z.grad[3].item() - p[3].item()) > 5e-14


def test_empty_input_is_nan():
    x = torch.empty((0, 16, 16), requires_grad=True)
    loss = mask_pred_loss(x, torch.empty((0, 16, 16)))
    loss.backward()
    assert torch.isnan(loss) and x.grad.shape == (0, 16, 16)


def test_gt_masks_needs_mask_head():
    with pytest.raises(ValueError, match="mask_size"):
        SgToLayoutStep(synth.Vocab(42), "cpu", gt_masks=True, mask_size=0)


def test_host_batch_with_masks_switch():
    vocab = synth.Vocab(42)
    graphs = synth.make_graphs(3, 750, 3, 6, vocab, include_dummies=True, mask_size=4)
    keys = lambda **kw: set(HostBatch(graphs, pin=False, **kw).t)          # noqa: E731
    base = {"triplets", "tri_off", "obj_off", "objs", "boxes", "uniforms"}
    assert keys() == base
    assert keys(with_geometry=True) == base | {"centers", "masks"}
    assert keys(with_masks=True) == base | {"masks"}
    assert keys(with_geometry=True, with_masks=False) == base | {"centers"}
    hb = HostBatch(graphs, pin=False, with_masks=True)
    m = hb.t["masks"]
    assert m.dtype == torch.float32 and m.shape == (int(hb.obj_off[-1]), 4, 4)
    assert torch.equal(m[-1], torch.ones(4, 4))                          # the __image__ dummy's all-ones mask
