"""TEST INFRASTRUCTURE — the torch restatement of local normalised cross-correlation (csrc/lncc.cu), not product code.

VoxelMorph's NCC with the sign turned so the loss is >= 0, written with torch convolutions so that it runs in fp64 and
fp32 on any device.  tests/test_lncc.py pins it to a brute-force loop and to autograd and compares the kernels with it;
tools/bench_lncc.py times its fp32 form.  The warp, the global terms and the smoothness penalty come from
oracle/torch_port.py.
"""
from __future__ import annotations

import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle.torch_port import flow_warp, smoothness_l2, weighted_loss     # noqa: E402


def lncc_box(x, win):
    """Zero-padded box sum over an odd window win^nd of x [N,1,...]: conv with a ones kernel, padding win//2.  TF32 is
    off so that the fp32 restatement is fp32 on any device."""
    nd = x.dim() - 2
    k = torch.ones((1, 1) + (win,) * nd, dtype=x.dtype, device=x.device)
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        return (F.conv3d if nd == 3 else F.conv2d)(x, k, padding=win // 2)


def lncc_terms(t, w, win):
    """-> (S_I, S_J, A, B, C, n) of the LNCC definition (csrc/lncc.cu), target t and warped w [N,1,...]."""
    n = win ** (t.dim() - 2)
    SI, SJ, SII, SJJ, SIJ = (lncc_box(v, win) for v in (t, w, t * t, w * w, t * w))
    return SI, SJ, SIJ - SI * SJ / n, SII - SI * SI / n, SJJ - SJ * SJ / n, n


def lncc_loss(t, w, win=9, eps=1e-5):
    """1 - mean over every voxel (of every pair) of cc = A^2 / (B C + eps), algebraically VoxelMorph's
    cross^2 / (I_var J_var + eps).  Differentiable (autograd)."""
    _, _, A, B, C, _ = lncc_terms(t, w, win)
    return 1 - torch.mean(A * A / (B * C + eps))


def lncc_grad(t, w, win=9, eps=1e-5):
    """d lncc_loss / d w in closed form: the box filter of the three per-voxel coefficients of cc."""
    SI, SJ, A, B, C, n = lncc_terms(t, w, win)
    den = B * C + eps
    gam = 2 * A / den
    bet = -A * A * B / den ** 2
    alp = -gam * SI / n - 2 * bet * SJ / n
    return -(lncc_box(alp, win) + 2 * w * lncc_box(bet, win) + t * lncc_box(gam, win)) / t.numel()


def direct_flow_lncc_loop(moving, target, lr, epochs, w_lncc=1.0, win=9, lncc_eps=1e-5, weights=(0.0, 0.0), smooth=0.0,
                          optimiser="sgd", betas=(0.9, 0.999), eps=1e-8, flow0=None):
    """torch_port.direct_flow_loop with the local NCC term added: loss = w_lncc * lncc_loss(target, warped) + w_mse * MSE +
    w_ncc * NCC + smooth * smoothness_l2(flow), optimised with torch SGD / Adam on the flow, on the inputs' device."""
    nd = moving.dim() - 2
    flow = (torch.zeros(1, nd, *moving.shape[2:], dtype=moving.dtype, device=moving.device) if flow0 is None
            else flow0.clone().detach().to(moving.device, moving.dtype)).requires_grad_(True)
    opt = (torch.optim.SGD([flow], lr) if optimiser == "sgd"
           else torch.optim.Adam([flow], lr, betas=betas, eps=eps))
    losses = []
    for _ in range(epochs):
        opt.zero_grad()
        warped = flow_warp(moving, flow)
        err = w_lncc * lncc_loss(target, warped, win, lncc_eps) + weighted_loss(target, warped, (weights[0], weights[1], 0.0))
        if smooth:
            err = err + smooth * smoothness_l2(flow)
        err.backward()
        opt.step()
        losses.append(err.item())
    return {"losses": losses, "flow": flow.detach().clone()}
