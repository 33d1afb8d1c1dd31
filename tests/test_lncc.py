"""Local normalised cross-correlation (csrc/lncc.cu, utils.LNCCLoss, the LNCC direct-flow epoch).

Every GPU result is compared with the fp64 torch restatement of the definition (tests/lncc_reference.py: lncc_loss,
lncc_grad, direct_flow_lncc_loop).  Tolerances follow DESIGN.md §2: the error against fp64 may be max(floor, 2 x the fp32
restatement's own error against fp64), the fp32 restatement running with TF32 off.  Floors: loss 1e-5 relative; gradient
1e-4 L2-relative and 1e-3 of max|g| per element.
CPU: the restatement against a brute-force loop, the closed-form gradient against autograd, and the host / ABI refusals."""
import itertools

import numpy as np
import pytest
import torch
import torch.nn as nn

import lncc_reference as lref
from oracle import torch_port as tp

DEV = "cuda:0"
gpu = pytest.mark.gpu


def _pair(shape, n=1, seed=0, dtype=torch.float64):
    """n (target, warped) pairs [n,1,*shape]: a smooth blob image and a perturbed, partly correlated copy."""
    from torchregister_b200.synth import make_pair
    ms, ts = [], []
    for i in range(n):
        mov, tgt = make_pair(tuple(shape), "flow", seed=1234 + i)
        g = torch.Generator().manual_seed(seed + i)
        ms.append(0.8 * mov.double() + 0.2 * torch.rand(mov.shape, generator=g, dtype=torch.float64))
        ts.append(tgt.double())
    return torch.cat(ts).to(dtype), torch.cat(ms).to(dtype)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the restatement itself
# ---------------------------------------------------------------------------------------------------------------------
def _brute_lncc(t, w, win, eps):
    """numpy loop over every voxel and every window offset; out-of-volume positions are zeros, n = win^nd fixed."""
    t, w = t[0, 0], w[0, 0]
    nd, r, n = t.ndim, win // 2, win ** t.ndim
    tot = 0.0
    for p in itertools.product(*[range(s) for s in t.shape]):
        s = np.zeros(5)
        for off in itertools.product(range(-r, r + 1), repeat=nd):
            q = tuple(a + b for a, b in zip(p, off))
            if all(0 <= q[k] < t.shape[k] for k in range(nd)):
                i, j = t[q], w[q]
                s += (i, j, i * i, j * j, i * j)
        A = s[4] - s[0] * s[1] / n
        B = s[2] - s[0] ** 2 / n
        C = s[3] - s[1] ** 2 / n
        tot += A * A / (B * C + eps)
    return 1.0 - tot / t.size


@pytest.mark.parametrize("shape,win", [((5, 6), 3), ((4, 7), 9), ((3, 4, 5), 3), ((2, 3, 4), 5), ((3, 2, 4), 7)])
def test_restatement_matches_brute_force(shape, win):
    """Zero padding and the fixed n, including windows wider than every axis."""
    t, w = _pair(shape)
    got = lref.lncc_loss(t, w, win, 1e-5).item()
    ref = _brute_lncc(t.numpy(), w.numpy(), win, 1e-5)
    assert abs(got - ref) <= 1e-12 * max(1.0, abs(ref)), (got, ref)


@pytest.mark.parametrize("shape,win", [((12, 13), 9), ((12, 13), 3), ((5, 6, 7), 3), ((4, 9, 11), 5), ((3, 8, 10), 9),
                                       ((2, 5, 4), 15)])
def test_closed_form_gradient_matches_autograd(shape, win):
    t, w = _pair(shape, n=2)
    w = w.clone().requires_grad_(True)
    lref.lncc_loss(t, w, win).backward()
    g = lref.lncc_grad(t, w.detach(), win)
    assert ((g - w.grad).abs().max() / w.grad.abs().max()).item() < 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# CPU: refusals
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("win", [2, 4, 1, 17, 0, -3, 9.5, True])
def test_lnccloss_refuses_bad_windows(win):
    import torchregister_b200 as tr
    with pytest.raises(ValueError):
        tr.LNCCLoss(win=win)


def test_lnccloss_refuses_bad_inputs():
    import torchregister_b200 as tr
    crit = tr.LNCCLoss()
    y = torch.rand(1, 1, 6, 7)
    with pytest.raises(RuntimeError, match="CUDA"):
        crit(y, y.clone().requires_grad_(True))                      # CPU tensors: no fallback
    with pytest.raises(TypeError, match="float32"):
        crit(y.double(), y.double())                                 # fp64
    with pytest.raises(TypeError, match="float32"):
        crit(y.half(), y.half())
    with pytest.raises(ValueError, match="target"):
        crit(y.clone().requires_grad_(True), y)                      # gradient to the target is not offered
    with pytest.raises(ValueError):
        tr.LNCCLoss(eps=0.0)


def test_direct_flow_register_accepts_lncc_and_refuses_other_criteria():
    import torchregister_b200 as tr
    r = tr.direct_flow_register((8, 9, 10), criterions=[tr.LNCCLoss(win=5)], weights=[1.0])
    assert (r.w_mse, r.w_ncc, r.w_lncc, r.lncc_win) == (0.0, 0.0, 1.0, 5)
    r = tr.direct_flow_register((8, 9, 10), criterions=[nn.MSELoss(), tr.NCCLoss(), tr.LNCCLoss()], weights=[0.5, 0.3, 2.0])
    assert (r.w_mse, r.w_lncc, r.lncc_win) == (0.5, 2.0, 9) and abs(r.w_ncc - 0.3) < 1e-12
    with pytest.raises(NotImplementedError):
        tr.direct_flow_register((8, 9, 10), criterions=[tr.LNCCLoss(), nn.L1Loss()], weights=[1.0, 1.0])
    with pytest.raises(NotImplementedError):
        tr.direct_flow_register((8, 9, 10), criterions=[tr.LNCCLoss(win=5), tr.LNCCLoss(win=7)], weights=[1.0, 1.0])
    r = tr.direct_flow_register((8, 9, 10), criterions=[nn.MSELoss(), tr.NCCLoss()], weights=[0.5, 0.5])
    assert r.w_lncc == 0.0


def test_abi_refusals():
    """Window, shape and overlap rules of the C ABI (fake device addresses: every case is refused before a launch)."""
    from torchregister_b200 import _lib
    lib = _lib.load()
    ws = lib.trb_lncc_workspace_bytes()
    assert ws >= 8 * 2048
    P, Q = 1 << 40, 1 << 41                  # never dereferenced
    nb = 4 * 8 * 8 * 8

    def fwd(win=9, D=8, coef=Q, eps=1e-5, w=P + nb, stats=Q + 3 * nb + 64):
        return lib.trb_lncc_forward(3, P, w, 1, D, 8, 8, win, eps, coef, stats, Q + (1 << 30), ws, None)

    for win in (2, 4, 1, 17, 0):
        assert fwd(win=win) == -3 and "window" in lib.trb_last_error().decode()
        assert lib.trb_lncc_backward(3, P, P + nb, Q, 1, 8, 8, 8, win, 1.0, None, 0.0, 0.0, Q + 3 * nb, None) == -3
    assert fwd(D=(1 << 22) + 8) == -3                      # an axis beyond 2^22
    assert fwd(D=0) == -1
    assert fwd(coef=P + nb // 2) == -1 and "overlaps" in lib.trb_last_error().decode()
    assert fwd(coef=P - 2 * nb) == -1                      # the gamma plane runs into the target
    assert fwd(eps=0.0) == -1
    assert lib.trb_lncc_forward(3, P, P + nb, 1, 8, 8, 8, 9, 1e-5, Q, Q + 3 * nb, None, 0, None) == -2
    assert lib.trb_lncc_backward(3, P, P + nb, Q, 1, 8, 8, 8, 9, 1.0, None, 0.0, 0.0, Q + nb, None) == -1   # grad in coef
    assert lib.trb_lncc_backward(3, P, P + nb, Q, 2, 8, 8, 8, 9, 1.0, Q + 9 * nb, 1.0, 0.0, Q + 6 * nb, None) == -1  # moments, N > 1
    assert lib.trb_flow_direct_update_lncc(3, P, Q, Q + nb, P + nb, 8, 8, 8, Q, Q, 0.0, 0.0, 1.0, 0.0, 1.0, 0, 0.9, 0.999,
                                           1e-8, 1, None, None, None, 0, None) == -1            # flow_out overlaps flow_in


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernels against fp64
# ---------------------------------------------------------------------------------------------------------------------
def _check_against_fp64(t64, w64, win, eps=1e-5):
    import torchregister_b200.functional as TF
    t32, w32 = t64.float(), w64.float()
    loss, grad = TF.lncc_loss_grad(w32.to(DEV), t32.to(DEV), win, eps)
    loss, grad = loss.item(), grad.cpu().double()
    L64, g64 = lref.lncc_loss(t64, w64, win, eps).item(), lref.lncc_grad(t64, w64, win, eps)
    L32, g32 = lref.lncc_loss(t32, w32, win, eps).item(), lref.lncc_grad(t32, w32, win, eps).double()
    # loss: floor 1e-5 relative, or twice the fp32 restatement's own gap
    assert abs(loss - L64) <= max(1e-5 * abs(L64), 2 * abs(L32 - L64)), (loss, L64, L32)
    # gradient: floor 1e-4 L2-relative and 1e-3 of max|g| per element, or twice the restatement's own errors
    l2 = ((grad - g64).norm() / g64.norm()).item()
    l2_32 = ((g32 - g64).norm() / g64.norm()).item()
    assert l2 <= max(1e-4, 2 * l2_32), (l2, l2_32)
    mx = (grad - g64).abs().max().item()
    mx32 = (g32 - g64).abs().max().item()
    assert mx <= max(1e-3 * g64.abs().max().item(), 2 * mx32), (mx, mx32, g64.abs().max().item())
    return loss, grad


KERNEL_CASES = [
    ((37, 45), 9),              # 2-D
    ((64, 33), 3),              # 2-D, W one past a tile
    ((5, 40), 15),              # 2-D, H shorter than the window
    ((13, 19, 37), 5),          # ragged: W not a multiple of 4 or 32
    ((18, 20, 24), 9),
    ((21, 17, 34), 3),
    ((4, 20, 30), 9),           # D shorter than the window
    ((3, 5, 7), 15),            # every axis shorter than the window
    ((9, 12, 70), 15),          # several x tiles, a wide halo
    ((320, 12, 20), 5),         # tall: many z chunks, no drift along z
]


@gpu
@pytest.mark.parametrize("shape,win", KERNEL_CASES, ids=lambda v: str(v))
def test_kernels_match_fp64(shape, win):
    t, w = _pair(shape)
    _check_against_fp64(t, w, win)


@gpu
@pytest.mark.parametrize("shape,win", [((11, 14, 35), 5), ((30, 41), 9)])
def test_pairs_are_never_mixed(shape, win):
    """N = 3 pairs in one call: each pair's alpha/beta/gamma equal its own single call bit for bit; the loss is the mean
    of the three and the gradient a third of each single one (1/N_vox)."""
    import torchregister_b200.functional as TF
    t, w = (v.float().to(DEV) for v in _pair(shape, n=3))
    stats, coef = TF.lncc_forward(t, w, win)
    grad = TF.lncc_backward(t, w, coef, win)
    vol = t[0].numel()
    singles = []
    for i in range(3):
        s1, c1 = TF.lncc_forward(t[i:i + 1], w[i:i + 1], win)
        assert torch.equal(coef.view(3, 3, vol)[:, i], c1), i
        g1 = TF.lncc_backward(t[i:i + 1], w[i:i + 1], c1, win)
        assert torch.allclose(grad[i:i + 1] * 3, g1, rtol=1e-6, atol=1e-6 * g1.abs().max().item())
        singles.append(s1[1].item())
    assert abs(stats[1].item() - sum(singles) / 3) <= 1e-12
    _check_against_fp64(*(v.double().cpu() for v in (t, w)), win)


@gpu
def test_two_calls_give_identical_bits():
    import torchregister_b200.functional as TF
    t, w = (v.float().to(DEV) for v in _pair((40, 33, 70)))
    a = TF.lncc_loss_grad(w, t, 9)
    b = TF.lncc_loss_grad(w, t, 9)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@gpu
def test_lnccloss_in_an_autograd_graph():
    import torchregister_b200 as tr
    t64, w64 = _pair((12, 21, 30))
    t, w = t64.float().to(DEV), w64.float().to(DEV)
    leaf = w.clone().requires_grad_(True)
    crit = tr.LNCCLoss(win=7)
    out = 3.0 * crit(t, 2.0 * leaf) + (leaf ** 2).sum()
    out.backward()
    # d/dleaf = 3 * 2 * g(2w) + 2 w, g the loss gradient at 2w
    g64 = lref.lncc_grad(t64, 2 * w64, 7)
    expect = 6.0 * g64 + 2 * w64
    got = leaf.grad.cpu().double()
    g32 = 6.0 * lref.lncc_grad(t64.float(), 2 * w64.float(), 7).double() + 2 * w64.float().double()
    err, err32 = (got - expect).norm() / expect.norm(), (g32 - expect).norm() / expect.norm()
    assert err <= max(1e-5, 2 * err32), (err, err32)
    assert abs(crit(t, w).item() - lref.lncc_loss(t64, w64, 7).item()) <= 1e-5


@gpu
def test_unet_flow_mode_with_lncc():
    """The U-Net flow mode takes LNCCLoss among its other criteria through SpatialTransformer's VJP: two epochs, finite
    losses, the second not above the first, and the first equal to the restatement at the U-Net's initial flow."""
    import torchregister_b200 as tr
    from torchregister_b200.synth import make_pair
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(0)
    mov, tgt = (v.to(DEV) for v in make_pair((160, 168), "flow"))
    fr = tr.flow_register((160, 168), mode="bilinear", n=32, lr=1e-3, max_epochs=2, criterions=[tr.LNCCLoss()], weights=[1.0],
                          stop_crit=-1.0).to(DEV)
    fr.train()
    with torch.no_grad():
        flow0 = fr.model.flow_field(mov, DEV).double()
    fr.optimize(mov, tgt, DEV, debug=False)
    assert len(fr.losses) == 2 and all(np.isfinite(fr.losses))
    assert fr.losses[1] <= fr.losses[0] + 1e-6, (fr.losses, fr.losses[1] - fr.losses[0])   # + fp32 rounding of a loss near 1
    ref = lref.lncc_loss(tgt.double(), tp.flow_warp(mov.double(), flow0), 9).item()
    assert abs(fr.losses[0] - ref) <= 1e-4 * abs(ref), (fr.losses[0], ref)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the LNCC direct-flow epoch against torch SGD / Adam on the restatement
# ---------------------------------------------------------------------------------------------------------------------
DIRECT_CASES = [
    # shape, optimiser, lr, smooth, (w_mse, w_ncc), win
    # (SGD: dL/dflow scales with 1/N_vox, so lr 500 moves these volumes by about half a voxel in 5 epochs; the NCC
    # weight is kept small because its term carries a factor 100)
    ((18, 20, 24), "sgd", 500.0, 0.0, (0.0, 0.0), 9),
    ((13, 19, 37), "sgd", 500.0, 4.0, (0.5, 0.01), 5),
    ((18, 20, 24), "adam", 0.05, 4.0, (0.0, 0.0), 9),
    ((40, 52), "sgd", 500.0, 0.0, (0.0, 0.0), 9),
    ((40, 52), "adam", 0.05, 4.0, (0.5, 0.01), 7),
]


@gpu
@pytest.mark.parametrize("shape,opt,lr,smooth,weights,win", DIRECT_CASES, ids=lambda v: str(v))
def test_lncc_direct_flow_vs_torch_restatement(shape, opt, lr, smooth, weights, win):
    import torchregister_b200.functional as TF
    from test_oracle_golden import _loss_ok
    from torchregister_b200.synth import make_pair, smooth_flow
    mov, tgt = (v.to(DEV) for v in make_pair(shape, "flow"))
    flow0 = (0.3 * smooth_flow(shape, 1.0)).to(DEV)
    epochs = 5
    kw = dict(w_lncc=1.0, win=win, weights=weights, smooth=smooth, optimiser=opt)
    ref = lref.direct_flow_lncc_loop(mov.double(), tgt.double(), lr, epochs, flow0=flow0.double(), **kw)
    ref32 = lref.direct_flow_lncc_loop(mov, tgt, lr, epochs, flow0=flow0, **kw)
    prob = TF.DirectFlowProblem(mov, tgt, epochs, flow0=flow0, optimiser=opt)
    prob.run(epochs, lr, weights[0], weights[1], smooth, w_lncc=1.0, lncc_win=win)
    ok, worst = _loss_ok(prob.losses.cpu().numpy(), ref32["losses"], ref["losses"])
    assert ok, (worst, prob.losses.cpu().numpy(), ref["losses"])
    d = (prob.flow.double() - ref["flow"]).abs().max().item()
    step = (ref["flow"] - flow0.double()).abs().max().item()
    gap32 = (ref32["flow"].double() - ref["flow"]).abs().max().item()
    assert step > 1e-3, step                              # the flow moves
    assert d <= max(1e-4 * step, 2 * gap32), (d, step, gap32)


@gpu
def test_register_direct_flow_with_lncc_end_to_end():
    import torchregister_b200 as tr
    from torchregister_b200.synth import make_pair
    mov, tgt = make_pair((24, 28, 32), "flow")
    reg = tr.Register(mode="flow", device=DEV, criterion=[tr.LNCCLoss()], weight=[1.0], flow_param="direct")
    reg.optim(mov, tgt, lr=500.0, max_epochs=40)
    assert len(reg.losses) == 40 and all(np.isfinite(reg.losses))
    assert reg.losses[-1] < reg.losses[0] - 1e-3, (reg.losses[0], reg.losses[-1])
    assert tuple(reg.theta.shape) == (1, 3, 24, 28, 32)
