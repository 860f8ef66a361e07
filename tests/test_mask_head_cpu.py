"""The identities the mask head's kernels rest on (csrc/mask_head.cu), checked in numpy against torch's own modules in
float64 on the CPU: BatchNorm at low resolution equals BatchNorm after nearest upsampling (forward, backward, running
variance), and the patch-matrix / gather index maps equal F.unfold / F.fold.  Plus the module layout of the head."""
import argparse

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from canonicalsg2im_b200 import synth


def _bn_low(x, gamma, beta, eps=1e-5):
    """x [O, s, s, C] (NHWC): BatchNorm with batch statistics over (O, s, s), as csg_mask_bn_fwd computes them."""
    mean = x.mean(axis=(0, 1, 2))
    var = ((x - mean) ** 2).mean(axis=(0, 1, 2))
    inv = 1.0 / np.sqrt(var + eps)
    return (x - mean) * inv * gamma + beta, mean, var, inv


def _patch(u, O, S, C):
    """A[(o*S + Y)*S + X, c*9 + ky*3 + kx] = u[o, Y+ky-1, X+kx-1, c] inside the image, else 0 (u: upsampled NHWC)."""
    A = np.zeros((O * S * S, 9 * C))
    for o in range(O):
        for Y in range(S):
            for X in range(S):
                for ky in range(3):
                    for kx in range(3):
                        yy, xx = Y + ky - 1, X + kx - 1
                        if 0 <= yy < S and 0 <= xx < S:
                            A[(o * S + Y) * S + X, np.arange(C) * 9 + ky * 3 + kx] = u[o, yy, xx]
    return A


def _gather(dA, O, s, C):
    """G[o, y, x, c]: the adjoint of _patch on the nearest-upsampled, low-resolution input (csg_mask_bn_bwd's gather)."""
    S = 2 * s
    G = np.zeros((O, s, s, C))
    for o in range(O):
        for y in range(s):
            for x in range(s):
                for dy in range(2):
                    for dx in range(2):
                        P, Q = 2 * y + dy, 2 * x + dx
                        for ky in range(3):
                            for kx in range(3):
                                Y, X = P - ky + 1, Q - kx + 1
                                if 0 <= Y < S and 0 <= X < S:
                                    G[o, y, x] += dA[(o * S + Y) * S + X, np.arange(C) * 9 + ky * 3 + kx]
    return G


def test_batchnorm_commutes_with_nearest_upsampling():
    rng = np.random.default_rng(0)
    O, C, s = 5, 6, 3
    x = rng.standard_normal((O, C, s, s))
    gamma, beta = rng.uniform(0.5, 1.5, C), rng.uniform(-1, 1, C)
    rm0, rv0 = rng.standard_normal(C), rng.uniform(0.5, 2, C)
    bn = nn.BatchNorm2d(C).double()
    with torch.no_grad():
        bn.weight.copy_(torch.from_numpy(gamma)); bn.bias.copy_(torch.from_numpy(beta))
        bn.running_mean.copy_(torch.from_numpy(rm0)); bn.running_var.copy_(torch.from_numpy(rv0))
    xt = torch.from_numpy(x).requires_grad_(True)
    y = bn(F.interpolate(xt, scale_factor=2, mode="nearest"))
    g = torch.from_numpy(rng.standard_normal(y.shape))
    y.backward(g)

    xl = x.transpose(0, 2, 3, 1)
    yl, mean, var, inv = _bn_low(xl, gamma, beta)
    # forward: the upsampled low-resolution result
    up = yl.repeat(2, axis=1).repeat(2, axis=2)
    assert np.abs(up - y.detach().numpy().transpose(0, 2, 3, 1)).max() < 1e-12
    # running buffers: momentum 0.1, unbiased variance over the 4n upsampled elements
    n_up = O * (2 * s) ** 2
    assert np.abs(0.9 * rm0 + 0.1 * mean - bn.running_mean.numpy()).max() < 1e-12
    assert np.abs(0.9 * rv0 + 0.1 * var * n_up / (n_up - 1) - bn.running_var.numpy()).max() < 1e-12
    assert int(bn.num_batches_tracked) == 1
    # backward at low resolution from the 2x2 block sums G of the upsampled gradient
    gn = g.numpy().transpose(0, 2, 3, 1)
    G = gn.reshape(O, s, 2, s, 2, C).sum(axis=(2, 4))
    n = O * s * s
    xh = (xl - mean) * inv
    dbeta, dgamma = G.sum(axis=(0, 1, 2)), (G * xh).sum(axis=(0, 1, 2))
    dx = gamma * inv * (G - (dbeta + xh * dgamma) / n)
    assert np.abs(dx - xt.grad.numpy().transpose(0, 2, 3, 1)).max() < 1e-12
    assert np.abs(dgamma - bn.weight.grad.numpy()).max() < 1e-12
    assert np.abs(dbeta - bn.bias.grad.numpy()).max() < 1e-12


def test_patch_and_gather_maps_match_unfold_and_fold():
    rng = np.random.default_rng(1)
    O, C, s = 3, 4, 2
    S = 2 * s
    x = rng.standard_normal((O, s, s, C))
    u = x.repeat(2, axis=1).repeat(2, axis=2)                                      # nearest upsampling, NHWC
    A = _patch(u, O, S, C)
    # F.unfold: [O, C*9, S*S] with the channel-major (c, ky, kx) order of conv.weight.view(C_out, 9 C)
    ut = torch.from_numpy(u.transpose(0, 3, 1, 2))
    cols = F.unfold(ut, kernel_size=3, padding=1).numpy()
    assert np.array_equal(A, cols.transpose(0, 2, 1).reshape(O * S * S, 9 * C))
    # a convolution is then one GEMM with the weight as it is stored
    w = rng.standard_normal((C, C, 3, 3))
    ref = F.conv2d(ut, torch.from_numpy(w), padding=1).numpy().transpose(0, 2, 3, 1).reshape(-1, C)
    assert np.abs(A @ w.reshape(C, 9 * C).T - ref).max() < 1e-12
    # adjoint: F.fold scatters dA back onto the upsampled image, the 2x2 block sums give the low-resolution gradient
    dA = rng.standard_normal(A.shape)
    folded = F.fold(torch.from_numpy(dA.reshape(O, S * S, 9 * C).transpose(0, 2, 1)), (S, S), kernel_size=3,
                    padding=1).numpy().transpose(0, 2, 3, 1)
    G_ref = folded.reshape(O, s, 2, s, 2, C).sum(axis=(2, 4))
    assert np.abs(_gather(dA, O, s, C) - G_ref).max() < 1e-12


def _opt(mask_size):
    vocab = synth.Vocab(0)
    return argparse.Namespace(
        vocab={"attributes": {"objects": {str(i): i for i in range(vocab.num_obj_classes)}},
               "pred_idx_to_name": vocab.pred_names, "pred_name_to_idx": vocab.pred_ids},
        embedding_dim=128, gconv_dim=128, gconv_hidden_dim=512, gconv_pooling="avg", gconv_num_layers=5,
        mlp_normalization="none", mask_size=mask_size, learned_init="uniform")


def test_mask_net_state_dict_keys():
    from canonicalsg2im_b200.model import Sg2LayoutModel
    m = Sg2LayoutModel(_opt(16))
    keys = {k for k in m.state_dict() if k.startswith("mask_net.")}
    want = {"mask_net.%d.%s" % (i, p) for i in (1, 5, 9, 13)
            for p in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")}
    want |= {"mask_net.%d.%s" % (i, p) for i in (2, 6, 10, 14, 16) for p in ("weight", "bias")}
    assert keys == want
    assert m.mask_net[2].weight.shape == (128, 128, 3, 3) and m.mask_net[16].weight.shape == (1, 128, 1, 1)
    assert Sg2LayoutModel(_opt(0)).mask_net is None


def test_mask_size_not_power_of_two():
    from canonicalsg2im_b200.model import Sg2LayoutModel
    with pytest.raises(ValueError, match="Mask size must be a power of 2"):
        Sg2LayoutModel(_opt(12))
