"""fp64 references for the kernels that differentiate a warp, on every kernel path they run: the affine warp and its
vector-Jacobian product (d/dtheta), the flow warp and its VJP, the fused flow node (warp + similarity + d/dflow) and the
fused U-Net head (padNd + 1x1 conv + node).  Plus the refusal of spatial axes longer than 2^22, which the kernels' fast
floor (csrc/common.cuh: floor_frac, round_idx) cannot index.

CPU: the flow reference against torch's grid_sample, and the C ABI's refusals (NULL pointers only).  GPU: every kernel
against the references, with the kernel that ran asserted.  Values are in [0, 1] (synth pairs) unless stated."""
import functools
import itertools
import math
import operator

import numpy as np
import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
MAX_AXIS = 1 << 22          # longest axis the 1.5*2^23 floor / rint indexes exactly (kMaxFastFloorAxis)
U = 2.0 ** -24              # fp32 unit roundoff
# a zero-padded bilinear / trilinear blend of values in [0, 1] is 3 (2-D) or 7 (3-D) fp32 fmaf / subtractions whose results
# stay within [-1, 1]: each rounds by at most U, and the fractions (<= 1) do not amplify them.  16 U covers either chain
WARP_ATOL = 16 * U
# per-voxel gradients (d value / d position times an fp32 factor) are differences of the same corners blended by the same
# fractions: their rounding is a few U relative to the gradient itself, far below 1e-5 of the largest one
GRAD_RTOL = 1e-5
# a loss is formed from fp32 warped values (WARP_ATOL each) and fp32 per-thread partial moments (the kernel's own claim:
# < 4e-6 relative): 1e-5 relative.  The NCC term 100 w_ncc (1 - NCC) also carries NCC's own error, which is absolute (NCC
# lies in [-1, 1]) and no larger than the samples' WARP_ATOL: 1e-6, i.e. 1e-4 w_ncc on the loss — when the pair is nearly
# aligned, 1 - NCC is ~1e-4 and relative 1e-5 of the loss would ask NCC for 1e-11
LOSS_RTOL = 1e-5
NCC_ATOL = 1e-6


def loss_tol(loss, w_ncc):
    return LOSS_RTOL * abs(loss) + 100 * w_ncc * NCC_ATOL


def _tf():
    import torchregister_b200.functional as TF
    return TF


def _prod(xs):
    return functools.reduce(operator.mul, xs, 1.0)


# ------------------------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------------------------
def flow_positions(flow):
    """flow [nd, *shape] fp32 (voxel units, channel a displaces axis a) -> sample positions [nd, *shape] fp32, formed op for
    op as the reference's normalise / grid_sample(align_corners=True) round trip does on the CPU, and as the bilinear flow
    kernels' flow_pos reproduces it: loc = i + u, q = loc / (S - 1) (IEEE), nrm = 2 (q - 0.5), p = ((nrm + 1) 0.5)(S - 1)."""
    flow = np.asarray(flow, np.float32)
    shape = flow.shape[1:]
    pos = []
    for a, S in enumerate(shape):
        i = np.arange(S, dtype=np.float32).reshape([-1 if b == a else 1 for b in range(len(shape))])
        d = np.float32(S - 1)
        q = (i + flow[a]) / d
        nrm = np.float32(2) * (q - np.float32(0.5))
        pos.append(((nrm + np.float32(1)) * np.float32(0.5)) * d)
    return np.stack(pos)


def sample_ref(img, pos):
    """Zero-padded bi/trilinear sample of img ([*shape]) at voxel positions pos ([nd, *out], axis order of img) and its
    gradient d value / d position ([nd, *out]), in fp64 on grid_sample's cell: the one whose origin is floor(p)."""
    img = np.asarray(img, np.float64)
    nd = img.ndim
    p = np.asarray(pos, np.float64)
    fl = np.floor(p)
    t = p - fl
    i0 = fl.astype(np.int64)
    val = np.zeros(p.shape[1:])
    grad = np.zeros(p.shape)
    for corner in itertools.product((0, 1), repeat=nd):
        idx = [i0[a] + corner[a] for a in range(nd)]
        inside = _prod([(idx[a] >= 0) & (idx[a] < img.shape[a]) for a in range(nd)]).astype(bool)
        c = np.where(inside, img[tuple(np.clip(idx[a], 0, img.shape[a] - 1) for a in range(nd))], 0.0)
        w = [t[a] if corner[a] else 1.0 - t[a] for a in range(nd)]
        val += c * _prod(w)
        for a in range(nd):
            grad[a] += (c if corner[a] else -c) * _prod([w[b] for b in range(nd) if b != a])
    return val, grad


def loss_and_dwarped(target, warped, w_mse, w_ncc):
    """w_mse MSE + w_ncc 100 (1 - NCC) of (target, warped) (oracle.torch_port, EPS_NCC inside the root) and its gradient
    with respect to warped, fp64 autograd."""
    from oracle import torch_port as tp
    w = torch.as_tensor(np.asarray(warped, np.float64)).requires_grad_(True)
    t = torch.as_tensor(np.asarray(target, np.float64))
    loss = tp.weighted_loss(t[None, None], w[None, None], (w_mse, w_ncc, 0.0))
    loss.backward()
    return loss.item(), w.grad.numpy()


def affine_ref(theta, moving):
    """get_affine_warp in fp64: affine_grid + grid_sample (align_corners=False, zeros), theta [N, nd, nd+1]."""
    grid = F.affine_grid(theta.double(), list(moving.shape), align_corners=False)
    return F.grid_sample(moving.double(), grid, mode="bilinear", padding_mode="zeros", align_corners=False)


def affine_atol(theta, moving):
    """Bound on |kernel - affine_ref| per pair [N]: the kernels form source coordinate r as
    (sum_c theta_rc b_c + theta_r,nd + 1) S_r / 2 - 1/2 in fp32 from fp32 base coordinates |b_c| < 1 — fewer than 16
    roundings of at most (sum_c |theta_rc| + 1) S_r / 2 each, counting the base tables' own — and the sample moves by at
    most the largest step of the zero-padded volume along r per voxel of that error.  Plus the blend's WARP_ATOL."""
    m = moving.double().numpy()
    nd = m.ndim - 2
    sizes = m.shape[2:][::-1]                                      # (W, H[, D]) <-> theta rows (x, y[, z])
    out = []
    for n in range(m.shape[0]):
        v = np.pad(m[n], [(0, 0)] + [(1, 1)] * nd)
        tol = WARP_ATOL * max(np.abs(m[n]).max(), 1e-30)
        for r in range(nd):
            step = np.abs(np.diff(v, axis=1 + nd - 1 - r)).max()
            tol += 16 * U * (np.abs(theta[n, r].double().numpy()).sum() + 1) * sizes[r] / 2 * step
        out.append(tol)
    return np.array(out)


def vjp_flip_bound(theta, img):
    """The value of a bilinear sample is continuous, its gradient is not: it jumps to the neighbouring cell's across a
    lattice line.  The kernels place a sample within affine_atol's position error of where fp64 puts it, so wherever that
    error straddles a lattice line (every voxel of an axis the transform maps onto the lattice, e.g. an identity row) the
    kernel's d warped / d theta may be the other cell's.  -> f(gout): per theta entry, the sum over those voxels of
    |gout| |g(other cell) - g| S_r / 2 |B_c| (B = the base coordinates and 1), a bound on what the choice of cell changes."""
    img = np.asarray(img, np.float64)
    nd, shape = img.ndim, img.shape
    th = np.asarray(theta, np.float64)
    sizes = shape[::-1]                                               # (W, H[, D]) <-> theta rows (x, y[, z])
    base = [(2 * np.arange(S) + 1) / S - 1 for S in sizes]            # affine_grid's, align_corners=False
    grids = np.meshgrid(*base[::-1], indexing="ij")                   # img axis order
    B = [grids[nd - 1 - c] for c in range(nd)] + [np.ones(shape)]
    pos = np.stack([((sum(th[r, c] * B[c] for c in range(nd)) + th[r, nd] + 1) * sizes[r] - 1) / 2
                    for r in range(nd)][::-1])                        # img axis order
    _, g = sample_ref(img, pos)
    terms = []
    for r_ax in range(nd):
        a = nd - 1 - r_ax
        err = 16 * U * (np.abs(th[r_ax]).sum() + 1) * sizes[r_ax] / 2
        n = np.round(pos[a])
        near = np.abs(pos[a] - n) <= err
        q = pos[:, near]
        q[a] = np.where(q[a] >= n[near], n[near] - 1e-9, n[near] + 1e-9)
        dg = np.abs(sample_ref(img, q)[1] - g[:, near])
        terms.append((near, np.stack([np.stack([dg[nd - 1 - r] * sizes[r] / 2 * np.abs(B[c][near]) for c in range(nd + 1)])
                                      for r in range(nd)])))
    return lambda gout: sum((np.abs(np.asarray(gout)[near]) * t).sum(-1) for near, t in terms)


def _flow_case(shape, kind, seed=0):
    """[nd, *shape] fp32: 'smooth' up to 6 voxels; 'integer' the same rounded (samples on the lattice); 'edge' every sample
    exactly at -1, 0, S-1, S-1+0.5, 0.5 or outside the volume, per axis."""
    from torchregister_b200.synth import smooth_flow
    if kind == "smooth":
        return smooth_flow(shape, 6.0)[0].numpy()
    if kind == "integer":
        return np.round(smooth_flow(shape, 6.0)[0].numpy())
    g = np.random.default_rng(seed)
    out = []
    for a, S in enumerate(shape):
        i = np.arange(S, dtype=np.float32).reshape([-1 if b == a else 1 for b in range(len(shape))])
        dest = np.array([-1, 0, S - 1, S - 0.5, 0.5, -3.25, S + 2.5], np.float32)
        out.append(dest[g.integers(0, len(dest), shape)] - i)      # i + u == dest exactly in fp32
    return np.stack(out).astype(np.float32)


def _close(got, ref, tol, what):
    err = np.abs(np.asarray(got, np.float64) - ref).max()
    assert err <= tol, "%s: max |kernel - fp64| = %.3e > %.3e" % (what, err, tol)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the flow reference itself
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(9, 11), (5, 7, 6)], ids=str)
def test_flow_reference_matches_grid_sample(shape):
    """sample_ref on flow_positions against torch's fp64 grid_sample autograd (oracle.torch_port.flow_warp,
    align_corners=True) at positions at least 1e-3 from the lattice (the gradient is continuous there), zero padding
    included.  The fp32 positions differ from torch's fp64 ones by p_err; the sample moves by at most 2 nd p_err (values
    in [0, 1]) and the gradient, linear in the other coordinates within a cell, by as much again."""
    from oracle import torch_port as tp
    g = np.random.default_rng(7)
    nd = len(shape)
    img = g.random(shape)
    dest = g.integers(-2, max(shape) + 1, (nd,) + shape) + 2e-3 + 0.996 * g.random((nd,) + shape)
    ident = np.stack(np.meshgrid(*[np.arange(s) for s in shape], indexing="ij"))
    flow = (dest - ident).astype(np.float32)
    pos = flow_positions(flow)
    p64 = ident + flow.astype(np.float64)
    assert np.abs(pos - np.round(pos)).min() > 5e-4
    p_err = np.abs(pos - p64).max()
    val, grad = sample_ref(img, pos)
    gout = g.uniform(-1, 1, shape)
    fl = torch.from_numpy(flow.astype(np.float64))[None].requires_grad_(True)
    out = tp.flow_warp(torch.from_numpy(img)[None, None], fl)
    (out * torch.from_numpy(gout)).sum().backward()
    tol = 2 * nd * p_err + 1e-12
    _close(val, out.detach()[0, 0].numpy(), tol, "value")
    _close(gout * grad, fl.grad[0].numpy(), 2 * tol, "d/dflow")


# ------------------------------------------------------------------------------------------------------------------
# CPU: axes the fast floor cannot index are refused at the C ABI (NULL pointers only: a shape that slipped through
# fails on the pointer check, never in a kernel)
# ------------------------------------------------------------------------------------------------------------------
def _flow_entry_points(lib, nd, D, H, W):
    """Every flow-side entry point that samples a volume, called with NULL pointers: {name: return code}."""
    ws = lib.trb_flow_workspace_bytes()
    calls = {
        "warp_flow": lambda: lib.trb_warp_flow_ex(nd, None, None, None, 1, D, H, W, 0, None),
        "warp_flow nearest": lambda: lib.trb_warp_flow_ex(nd, None, None, None, 1, D, H, W, 8, None),
        "warp_flow_vjp": lambda: lib.trb_warp_flow_vjp(nd, None, None, None, None, D, H, W, None),
        "flow_loss_grad": lambda: lib.trb_flow_loss_grad(nd, None, None, None, D, H, W, 1.0, 0.0, None, None, None, None, ws,
                                                         None),
        "flow_head_forward": lambda: lib.trb_flow_head_forward(nd, None, None, None, 1, 1, 1, 1, None, None, D, H, W, 1.0, 0.0,
                                                               None, None, None, ws, None),
        "flow_head_backward": lambda: lib.trb_flow_head_backward(nd, None, None, None, None, 1, 1, 1, 1, None, D, H, W, None,
                                                                 None, None, ws, None),
        "flow_direct_stats": lambda: lib.trb_flow_direct_stats(nd, None, None, None, None, None, D, H, W, 0, D, 0.0, None,
                                                               None, 0, None),
        "flow_direct_update": lambda: lib.trb_flow_direct_update(nd, None, None, None, None, None, None, D, H, W, 0, D, None,
                                                                 1.0, 0.0, 0.0, 1e-3, 0, 0.9, 0.999, 1e-8, 1, None, None,
                                                                 None, 0, None),
    }
    if nd == 3:
        calls["flow_direct_step"] = lambda: lib.trb_flow_direct_step(None, None, None, None, None, None, D, H, W, 0, D, None,
                                                                     1.0, 0.0, 0.0, 1e-3, 0, 0.9, 0.999, 1e-8, 1, None, None,
                                                                     None, 0, 0, None, 0, None)
    return {name: (fn(), lib.trb_last_error().decode()) for name, fn in calls.items()}


def _affine_nearest(lib, nd, D, H, W, flags):
    rc = lib.trb_warp_affine_batch(nd, None, None, 1, 1, D, H, W, None, None, None, None, flags, None)
    return rc, lib.trb_last_error().decode()


AXIS_SHAPES = [(2, 1, 2, "W"), (2, 1, "H", 2), (3, "D", 2, 2), (3, 2, "H", 2), (3, 2, 2, "W")]


@pytest.mark.parametrize("nd,D,H,W", AXIS_SHAPES, ids=lambda v: str(v))
def test_abi_refuses_axes_beyond_the_fast_floor(nd, D, H, W):
    """One axis of 2^22 + 8 voxels: every flow entry point that samples (warps, VJP, node, head, direct flow) and the
    nearest affine warp return TRB_ERR_UNSUPPORTED naming the limit.  At 2^22 exactly they accept the shape and stop at
    the NULL pointers (TRB_ERR_ARG); the bilinear affine warp, which floors with floorf, accepts either."""
    from torchregister_b200 import _lib
    lib = _lib.load()
    for n, expect in ((MAX_AXIS + 8, -3), (MAX_AXIS, -1)):
        d, h, w = (n if v in ("D", "H", "W") else v for v in (D, H, W))
        got = _flow_entry_points(lib, nd, d, h, w)
        for flags in (8, 0):                    # TRB_FLAG_NEAREST, bilinear
            ah = 1 if nd == 2 and H != "H" else h   # the affine warps allow H = 1 in 2-D
            got["warp_affine" + (" nearest" if flags else "")] = _affine_nearest(lib, nd, d, ah, w, flags)
        for name, (rc, msg) in got.items():
            want = -1 if name == "warp_affine" else expect
            assert rc == want, "%s at %dx%dx%d: rc %d (%s)" % (name, d, h, w, rc, msg)
            assert ("4194304" in msg) == (want == -3), (name, msg)


# ------------------------------------------------------------------------------------------------------------------
# GPU: affine warp and its VJP
# ------------------------------------------------------------------------------------------------------------------
def _thetas(nd):
    """theta near identity, a 45 degree rotation (x, y), and scale 1.3 with a translation that puts half the samples
    outside the volume."""
    c = s = math.sqrt(0.5)
    if nd == 3:
        return {"near_identity": [[1.01, -0.015, 0.01, 0.02], [0.012, 0.99, -0.008, -0.01], [-0.01, 0.011, 1.005, 0.015]],
                "rot45": [[c, -s, 0, 0], [s, c, 0, 0], [0, 0, 1, 0]],
                "scale_out": [[1.3, 0, 0, 1.0], [0, 1.3, 0, 0], [0, 0, 1.3, 0]]}
    return {"near_identity": [[1.01, -0.015, 0.02], [0.012, 0.99, -0.01]],
            "rot45": [[c, -s, 0], [s, c, 0]],
            "scale_out": [[1.3, 0, 1.0], [0, 1.3, 0]]}


@pytest.fixture
def kernel_path():
    TF = _tf()
    yield TF.set_kernel_path
    TF.set_kernel_path("auto")


# (3-D, W % 4 == 0, W >= 32, H >= 16 take the TMA-tile kernels; 32x16x16 output tiles)
VJP_PATHS = {
    "direct3d": ((37, 50, 68), "direct", False),
    "tma3d": ((37, 50, 68), "auto", False),              # 36 tiles: the per-epoch TMA kernel
    "persist_tma3d": ((641, 289, 36), "auto", False),    # 2 x 19 x 41 = 1558 tiles, >= 10 per SM: the persistent kernel
    "persist_gather3d": ((37, 50, 68), "auto", True),    # large_rotation: the persistent kernel's gather variant
    "direct2d": ((300, 181), "auto", False),             # 2-D has the direct-gather kernel only
}


def _tiles(shape):
    D, H, W = shape
    return -(-W // 32) * -(-H // 16) * -(-D // 16)


@pytest.mark.gpu
@pytest.mark.parametrize("theta_name", ["near_identity", "rot45", "scale_out"])
@pytest.mark.parametrize("path", list(VJP_PATHS))
def test_warp_affine_vjp_matches_fp64_autograd(path, theta_name, kernel_path):
    """d/dtheta of the affine warp against fp64 autograd of affine_grid + grid_sample, for a signed random grad_out and for
    the MSE one, 2 (w - t) / n.  It is a sum over every voxel of fp32 terms that carry their coordinates' rounding and are
    accumulated in fp32 per thread: 1e-5 of the largest entry (expected error ~1e-6, the fp64 stages above the thread
    level add nothing), plus vjp_flip_bound for the voxels whose cell fp32 and fp64 coordinates may choose apart.  A signed
    random grad_out cancels most of the sum, so those few voxels would otherwise dominate the comparison."""
    from torchregister_b200.synth import make_pair
    TF = _tf()
    shape, kp, large = VJP_PATHS[path]
    nd = len(shape)
    theta = torch.tensor(_thetas(nd)[theta_name], dtype=torch.float32)
    mov, tgt = make_pair(shape, "rigid")
    th = theta.double()[None].requires_grad_(True)
    w = F.grid_sample(mov.double(), F.affine_grid(th, list(mov.shape), align_corners=False), mode="bilinear",
                      padding_mode="zeros", align_corners=False)
    g = np.random.default_rng(3)
    gouts = {"signed": torch.from_numpy(g.uniform(-1, 1, mov.shape).astype(np.float32)),
             "mse": (2 * (w.detach() - tgt.double()) / mov.numel()).float()}
    flips = vjp_flip_bound(theta, mov[0, 0].numpy())
    sms = TF._lib.load().trb_sm_count()
    kernel_path(kp)
    mdev = mov.to(DEV)
    for name, gout in gouts.items():
        ref = torch.autograd.grad((w * gout.double()).sum(), th, retain_graph=True)[0][0].numpy()
        tol = GRAD_RTOL * np.abs(ref).max() + flips(gout[0, 0].numpy())
        got = TF.warp_affine_vjp(theta, mdev, gout.to(DEV), large_rotation=large).cpu().numpy()
        status = TF._lib.load().trb_affine_kernel_status().decode()
        if path.startswith("persist"):
            assert status.startswith("launched") and (", tma variant" if path == "persist_tma3d" else ", gather variant") in status, status
            if not large:
                assert _tiles(shape) >= 10 * sms
        err = np.abs(got - ref)
        assert (err <= tol).all(), "%s %s d/dtheta: |kernel - fp64| %s > %s" % (path, name, err, tol)
        if path == "tma3d":
            # the TMA and direct kernels form coordinates with different fp32 chains: equal bits would mean one kernel ran
            assert _tiles(shape) < 10 * sms
            kernel_path("direct")
            direct = TF.warp_affine_vjp(theta, mdev, gout.to(DEV)).cpu().numpy()
            kernel_path(kp)
            assert not np.array_equal(got, direct)


AFFINE_SHAPES = [(5, 17, 68), (1, 20, 68), (6, 9, 1), (7, 18, 31), (6, 17, 33),     # 3-D
                 (1, 1), (1, 31), (1, 33), (1, 68), (19, 68), (23, 31)]              # 2-D


@pytest.mark.gpu
@pytest.mark.parametrize("shape", AFFINE_SHAPES, ids=str)
def test_warp_affine_matches_fp64_on_every_path(shape, kernel_path):
    """Forward bilinear affine warp, 3 pairs x 2 channels, each pair its own theta (near identity, 45 degrees, half
    outside), against fp64 affine_grid + grid_sample, within affine_atol.  3-D: the TMA-tile kernel (W % 4 == 0, W >= 32,
    H >= 16, D = 1 included), the gather kernel (large_rotation) and the direct path (the same gather kernel)."""
    from torchregister_b200.synth import make_pair
    TF = _tf()
    nd = len(shape)
    theta = torch.tensor(list(_thetas(nd).values()), dtype=torch.float32)
    mov = torch.cat([torch.cat(make_pair(shape, "rigid", seed=5 + i), 1) for i in range(3)])      # [3, 2, ...]
    ref = affine_ref(theta, mov).numpy()
    atol = affine_atol(theta, mov)
    mdev = mov.to(DEV)
    outs = {"gather": TF.warp_affine(theta, mdev, large_rotation=True).cpu().numpy()}
    kernel_path("direct")
    outs["direct"] = TF.warp_affine(theta, mdev).cpu().numpy()
    kernel_path("auto")
    outs["auto"] = TF.warp_affine(theta, mdev).cpu().numpy()
    for name, out in outs.items():
        for n in range(3):
            _close(out[n], ref[n], atol[n], "%s pair %d" % (name, n))
    assert np.array_equal(outs["gather"], outs["direct"])
    tma = nd == 3 and shape[2] % 4 == 0 and shape[2] >= 32 and shape[1] >= 16
    # the TMA kernel forms coordinates with another fp32 chain than the gather kernel: its bits differ
    assert np.array_equal(outs["auto"], outs["gather"]) != tma


# ------------------------------------------------------------------------------------------------------------------
# GPU: flow warp, VJP and the fused node
# ------------------------------------------------------------------------------------------------------------------
# (96, 100, 130): more row pairs than 2 x the grid's CTAs (the grid-stride loop) and W > 128 (a thread walks a row twice)
FLOW_SHAPES = [(2, 2), (37, 41), (1000, 1300), (2, 2, 2), (19, 26, 35), (96, 100, 130)]
FLOW_KINDS = ["smooth", "integer", "edge"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", FLOW_KINDS)
@pytest.mark.parametrize("shape", FLOW_SHAPES, ids=str)
def test_warp_flow_and_vjp_match_fp64(shape, kind):
    """warp_flow of 3 channels, and warp_flow_vjp, against sample_ref at the kernels' own fp32 positions: the same cell at
    every lattice and boundary position, so values are held to the blend's rounding and d/dflow per voxel to GRAD_RTOL."""
    from torchregister_b200.synth import make_pair
    TF = _tf()
    mov, tgt = make_pair(shape, "flow")
    src = torch.cat([mov, tgt, 1 - mov], 1)
    flow = _flow_case(shape, kind)
    pos = flow_positions(flow)
    s64 = src[0].double().numpy()
    refs = [sample_ref(s64[c], pos) for c in range(3)]
    fdev = torch.from_numpy(flow)[None].to(DEV)
    out = TF.warp_flow(src.to(DEV), fdev)[0].cpu().numpy()
    _close(out, np.stack([r[0] for r in refs]), WARP_ATOL, "warped")
    gout = np.random.default_rng(1).uniform(-1, 1, shape).astype(np.float32)
    dflow = TF.warp_flow_vjp(src[:, :1].to(DEV), fdev, torch.from_numpy(gout)[None, None].to(DEV))[0].cpu().numpy()
    ref = gout * refs[0][1]
    _close(dflow, ref, GRAD_RTOL * np.abs(ref).max(), "d/dflow")


@pytest.mark.gpu
@pytest.mark.parametrize("weights", [(1.0, 0.0), (0.0, 1.0), (0.5, 0.5)], ids=["mse_fused", "ncc", "mse_ncc"])
@pytest.mark.parametrize("kind", FLOW_KINDS)
@pytest.mark.parametrize("shape", FLOW_SHAPES, ids=str)
def test_flow_loss_grad_matches_fp64(shape, kind, weights):
    """The fused node: w_ncc == 0 runs flow_mse_fused_kernel, otherwise flow_stats_kernel + flow_grad_kernel.  Loss,
    warped volume and d loss / d flow against fp64 (loss and d loss / d warped by autograd of oracle.torch_port)."""
    from torchregister_b200.synth import make_pair
    TF = _tf()
    mov, tgt = make_pair(shape, "flow")
    flow = _flow_case(shape, kind)
    val, grad = sample_ref(mov[0, 0].double().numpy(), flow_positions(flow))
    loss, dw = loss_and_dwarped(tgt[0, 0].double().numpy(), val, *weights)
    ref = dw * grad
    got_loss, dflow, warped = TF.flow_loss_grad(mov.to(DEV), tgt.to(DEV), torch.from_numpy(flow)[None].to(DEV), *weights,
                                                want_warped=True)
    assert abs(got_loss.item() - loss) <= loss_tol(loss, weights[1]), (got_loss.item(), loss)
    _close(warped[0, 0].cpu().numpy(), val, WARP_ATOL, "warped")
    _close(dflow[0].cpu().numpy(), ref, GRAD_RTOL * np.abs(ref).max(), "d loss/d flow")


# ------------------------------------------------------------------------------------------------------------------
# GPU: the fused U-Net head
# ------------------------------------------------------------------------------------------------------------------
HEAD_CASES = [  # volume, feature channels, volume minus feature size per axis (odd: padNd puts the larger half after)
    ((37, 41), 1, (0, 3)), ((37, 41), 3, (1, 2)), ((37, 41), 8, (3, 1)),
    ((19, 26, 35), 1, (2, 3, 0)), ((19, 26, 35), 3, (3, 0, 1)), ((19, 26, 35), 8, (1, 2, 3)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("weights", [(1.0, 0.0), (0.5, 0.5)], ids=["mse", "mse_ncc"])
@pytest.mark.parametrize("shape,C,delta", HEAD_CASES, ids=lambda v: str(v))
def test_flow_head_matches_fp64(shape, C, delta, weights):
    """flow_head_forward / _backward against padNd + 1x1 conv in fp64 autograd, chained to the node's d loss / d flow in
    fp64 at the kernel's own flow (its fp32 sum of C products, checked first).  d feat per voxel to GRAD_RTOL; d W and d b
    are sums over the volume of fp32 terms accumulated in fp32 per thread: GRAD_RTOL of their largest entry."""
    from torchregister_b200.synth import make_pair
    TF = _tf()
    nd = len(shape)
    fshape = tuple(s - d for s, d in zip(shape, delta))
    g = torch.Generator().manual_seed(11 + C)
    feat = torch.rand((1, C) + fshape, generator=g) - 0.5
    weight = torch.randn(nd, C, generator=g) * (3.0 / math.sqrt(C))
    bias = torch.randn(nd, generator=g)
    mov, tgt = make_pair(shape, "flow")
    loss, flow = TF.flow_head_forward(mov.to(DEV), tgt.to(DEV), feat.to(DEV), weight.to(DEV), bias.to(DEV), *weights)
    dfeat, dW, db = TF.flow_head_backward(mov.to(DEV), tgt.to(DEV), flow, feat.to(DEV), weight.to(DEV))
    f64, W64, b64 = (x.double().requires_grad_(True) for x in (feat, weight, bias))
    pad = []
    for d in reversed(delta):                       # padNd: delta // 2 zeros in front, the rest after
        pad += [d // 2, d - d // 2]
    flow64 = torch.einsum("kc,bc...->bk...", W64, F.pad(f64, pad)) + b64.view((1, nd) + (1,) * nd)
    flow_k = flow[0].cpu().numpy()
    bound = (C + 1) * U * (bias.abs().max() + (weight.abs().sum(1).max() * 0.5)).item()
    _close(flow_k, flow64.detach()[0].numpy(), bound, "flow")
    val, grad = sample_ref(mov[0, 0].double().numpy(), flow_positions(flow_k))
    lref, dw = loss_and_dwarped(tgt[0, 0].double().numpy(), val, *weights)
    flow64.backward(torch.from_numpy(dw * grad)[None])
    assert abs(loss.item() - lref) <= loss_tol(lref, weights[1]), (loss.item(), lref)
    ref_feat = f64.grad.numpy()
    _close(dfeat.cpu().numpy(), ref_feat, GRAD_RTOL * np.abs(ref_feat).max(), "d feat")
    ref_wb = np.concatenate([W64.grad.numpy().ravel(), b64.grad.numpy()])
    got_wb = np.concatenate([dW.cpu().numpy().ravel(), db.cpu().numpy()])
    _close(got_wb, ref_wb, GRAD_RTOL * np.abs(ref_wb).max(), "d W, d b")


@pytest.mark.gpu
def test_flow_head_refuses_what_it_cannot_fuse():
    """More than 8 feature channels (TRB_ERR_UNSUPPORTED), and a feature map larger than the volume on some axis, in the
    forward and the backward call."""
    from torchregister_b200.synth import make_pair
    TF = _tf()
    mov, tgt = (x.to(DEV) for x in make_pair((20, 24), "flow"))
    flow = torch.zeros(1, 2, 20, 24, device=DEV)
    feat9, w9 = torch.rand(1, 9, 20, 24, device=DEV), torch.rand(2, 9, device=DEV)
    with pytest.raises(RuntimeError, match="1..8"):
        TF.flow_head_forward(mov, tgt, feat9, w9, torch.zeros(2, device=DEV), 1.0, 0.0)
    with pytest.raises(RuntimeError, match="1..8"):
        TF.flow_head_backward(mov, tgt, flow, feat9, w9)
    for fshape in ((21, 24), (20, 25)):
        feat, w = torch.rand((1, 2) + fshape, device=DEV), torch.rand(2, 2, device=DEV)
        with pytest.raises(ValueError, match="larger than the volume"):
            TF.flow_head_forward(mov, tgt, feat, w, torch.zeros(2, device=DEV), 1.0, 0.0)
        with pytest.raises(ValueError, match="larger than the volume"):
            TF.flow_head_backward(mov, tgt, flow, feat, w)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the longest axes
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flow_calls_refuse_an_axis_beyond_the_fast_floor():
    """(2, 2^22 + 8) with u = +1000.25: samples of columns 2^22 - 995 .. 2^22 - 993 fall at x in (2^22, W - 1), where the
    1.5*2^23 floor is off by hundreds of voxels and still inside the volume.  Every flow call refuses the shape."""
    TF = _tf()
    W = MAX_AXIS + 8
    src = torch.rand(1, 1, 2, W, device=DEV)
    flow = torch.zeros(1, 2, 2, W, device=DEV)
    flow[:, 1] = 1000.25
    for name, fn in (("warp_flow", lambda: TF.warp_flow(src, flow)),
                     ("warp_flow nearest", lambda: TF.warp_flow(src, flow, mode="nearest")),
                     ("warp_flow_vjp", lambda: TF.warp_flow_vjp(src, flow, src)),
                     ("flow_loss_grad", lambda: TF.flow_loss_grad(src, src, flow, 0.5, 0.5))):
        with pytest.raises(RuntimeError, match="4194304"):
            fn()


@pytest.mark.gpu
def test_flow_warp_at_the_longest_allowed_axis_matches_fp64():
    """(2, 2^22): samples a fraction of a voxel right of every column up to x = 2^22 - 1 + 0.375, where fp32 positions
    are coarsest, and (last 64 columns) 1000.25 voxels right, outside the volume."""
    TF = _tf()
    W = MAX_AXIS
    src = np.random.default_rng(2).random((2, W)).astype(np.float32)
    flow = np.zeros((2, 2, W), np.float32)
    flow[0, 0], flow[0, 1] = 0.5, -0.25
    flow[1] = 0.375
    flow[1, :, -64:] = 1000.25
    val, _ = sample_ref(src, flow_positions(flow))
    out = TF.warp_flow(torch.from_numpy(src)[None, None].to(DEV), torch.from_numpy(flow)[None].to(DEV))
    _close(out[0, 0].cpu().numpy(), val, WARP_ATOL, "warped")


@pytest.mark.gpu
def test_affine_warps_on_an_axis_beyond_the_fast_floor():
    """H = 1, W = 2^22 + 8: the nearest affine warp (round_idx) refuses it; the bilinear one (floorf) matches fp64.  A
    sine that vanishes at both ends keeps every per-voxel step tiny, so affine_atol stays far below the error of a sample
    hundreds of voxels off."""
    TF = _tf()
    W = MAX_AXIS + 8
    x = torch.arange(W, dtype=torch.float64)
    img = (0.5 * torch.sin(math.pi * x / (W - 1))).float().view(1, 1, 1, W)
    theta = torch.tensor([[1.0, 0.0, 0.2], [0.0, 1.0, 0.0]])
    with pytest.raises(RuntimeError, match="4194304"):
        TF.warp_affine(theta, img.to(DEV), mode="nearest")
    out = TF.warp_affine(theta, img.to(DEV)).cpu().numpy()
    _close(out[0], affine_ref(theta[None], img).numpy()[0], affine_atol(theta[None], img)[0], "warped")
