"""Transform algebra (csrc/transform.cu, torchregister_b200.transforms): an affine result as a flow, "first, then second"
composition with a flow second, and the inverse of a flow.

Every GPU result is compared with an fp64 restatement of its own definition (never with warping twice: that differs from
the composed field by an interpolation with no tight bound), with the tolerance derived from the fp32 arithmetic of the
kernel and the reason written beside it.  CPU tests check the host surface, the C ABI's refusals and the fp64 references
against torch's affine_grid and grid_sample."""
import inspect
import itertools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
U = 2.0 ** -24              # fp32 unit roundoff
U64 = 2.0 ** -53            # fp64 unit roundoff
SHAPES = [(37, 50, 61), (97, 130)]        # non-cubic, W not a multiple of 4
BIG = (40, 120, 130)                      # 624000 voxels: 2438 work items of 256 voxels, more than the 2048-block cap


# ------------------------------------------------------------------------------------------------------------------
# fp64 references
# ------------------------------------------------------------------------------------------------------------------
def voxel_grid(shape):
    """[nd, *shape] fp64 voxel positions p in flow channel order ((z, y, x) or (y, x))."""
    return np.stack(np.meshgrid(*[np.arange(s, dtype=np.float64) for s in shape], indexing="ij"))


def affine_map(theta, shape):
    """theta ([nd, nd+1], row r sampling coordinate r, 0 = x) -> (A, c, M) in flow channel order, fp64: T(q) = M q + c,
    A = M - I.  M_rc = theta_rc S_r / S_c, c_r = S_r/2 (theta_r,nd + 1 - sum_c theta_rc (1 - 1/S_c)) - 1/2."""
    nd = len(shape)
    th = np.asarray(theta, np.float64).reshape(nd, nd + 1)
    S = shape[::-1]                                          # by sampling coordinate: (W, H[, D])
    M, c = np.empty((nd, nd)), np.empty(nd)
    for i in range(nd):
        r = nd - 1 - i
        c[i] = S[r] / 2 * (th[r, nd] + 1 - sum(th[r, k] * (1 - 1 / S[k]) for k in range(nd))) - 0.5
        for j in range(nd):
            M[i, j] = th[r, nd - 1 - j] * S[r] / S[nd - 1 - j]
    return M - np.eye(nd), c, M


def compose_affine_ref(theta, u, shape):
    """w = T(p + u) - p = u + A (p + u) + c, fp64; u [nd, *shape] (zeros: the affine's own flow)."""
    A, c, _ = affine_map(theta, shape)
    u = np.asarray(u, np.float64)
    q = voxel_grid(shape) + u
    return u + np.einsum("ij,j...->i...", A, q) + c.reshape((-1,) + (1,) * len(shape))


def sample_border(img, pos):
    """fp64 bi/trilinear sample of img [*shape] at voxel positions pos [nd, *out] (img axis order), border padding: every
    coordinate clamped to [0, S-1] before the floor, the corner past S-1 weighted 0 and read as 0.  NaN where a position
    is non-finite; a NaN corner that is read gives NaN (its weight may be 0: 0 * NaN is NaN, as in the kernel's blend)."""
    img = np.asarray(img, np.float64)
    nd = img.ndim
    pos = np.asarray(pos, np.float64)
    fin = np.isfinite(pos).all(0)
    p = np.stack([np.clip(np.where(fin, pos[a], 0.0), 0, img.shape[a] - 1) for a in range(nd)])
    fl = np.floor(p)
    t = p - fl
    i0 = fl.astype(np.int64)
    val = np.zeros(p.shape[1:])
    for corner in itertools.product((0, 1), repeat=nd):
        idx = [i0[a] + corner[a] for a in range(nd)]
        inside = np.logical_and.reduce([idx[a] < img.shape[a] for a in range(nd)])
        cval = np.where(inside, img[tuple(np.minimum(idx[a], img.shape[a] - 1) for a in range(nd))], 0.0)
        w = np.prod([t[a] if corner[a] else 1.0 - t[a] for a in range(nd)], axis=0)
        val = val + cval * w
    return np.where(fin, val, np.nan)


def compose_flows_ref(f, u):
    """w = u + f~(p + u), fp64; f, u [nd, *shape]."""
    u = np.asarray(u, np.float64)
    q = voxel_grid(u.shape[1:]) + u
    return u + np.stack([sample_border(f[i], q) for i in range(u.shape[0])])


def residual_ref(u, v):
    """|v + u~(p + v)|_inf per voxel, fp64."""
    s = compose_flows_ref(u, v) - np.asarray(v, np.float64)            # u~(p + v)
    d = np.asarray(v, np.float64) + s
    return np.where(np.isfinite(d).all(0), np.abs(d).max(0), np.nan)


def invert_ref(u, max_iter, tol, band=0.0):
    """The kernel's iteration restated in fp64: v_0 = -u(p); iteration k evaluates r_k = |v_k + u~(p + v_k)|_inf, stops
    when r_k <= tol or k = max_iter - 1 (or a non-finite position / residual: NaN), else v_{k+1} = -u~(p + v_k).
    -> (v, r, evaluations, non-finite mask, ambiguous mask: some evaluated |r_k - tol| <= band)."""
    u = np.asarray(u, np.float64)
    nd, shape = u.shape[0], u.shape[1:]
    p = voxel_grid(shape)
    v = -u.copy()
    active = np.ones(shape, bool)
    bad, amb = np.zeros(shape, bool), np.zeros(shape, bool)
    r, k = np.zeros(shape), np.zeros(shape, np.int64)
    for it in range(max_iter):
        q = p + v
        s = np.stack([sample_border(u[i], q) for i in range(nd)])
        d = v + s
        rr = np.where(np.isfinite(d).all(0), np.abs(np.where(np.isfinite(d), d, 0)).max(0), np.nan)
        k[active] += 1
        fin = np.isfinite(rr)
        bad |= active & ~fin
        r = np.where(active, rr, r)
        amb |= active & fin & (np.abs(rr - tol) <= band)
        stop = active & (~fin | (rr <= tol) | (it == max_iter - 1))
        active &= ~stop
        v = np.where(active, -s, v)
        if not active.any():
            break
    v[:, bad] = np.nan
    return v, r, k, bad, amb


def fixed_point_ref(u, eps=1e-12, max_iter=2000):
    """The fp64 fixed point of v = -u~(p + v), iterated until the residual is <= eps everywhere."""
    u = np.asarray(u, np.float64)
    p = voxel_grid(u.shape[1:])
    v = -u.copy()
    for _ in range(max_iter):
        s = np.stack([sample_border(u[i], p + v) for i in range(u.shape[0])])
        if np.abs(v + s).max() <= eps:
            return v
        v = -s
    raise AssertionError("fp64 fixed point did not converge")


def lipschitz(u):
    """Bound on the inf-norm Lipschitz constant of u~: max over channels i of sum over axes j of max |forward difference
    of u_i along j| (within a cell the interpolant's slope along j is a blend of those differences; the border clamp is
    1-Lipschitz per coordinate)."""
    u = np.asarray(u, np.float64)
    return max(sum(np.abs(np.diff(u[i], axis=j)).max() for j in range(u.ndim - 1)) for i in range(u.shape[0]))


def steps(f):
    """[channel][axis] max |forward difference| of f: how far f~ moves per voxel of position along that axis."""
    f = np.asarray(f, np.float64)
    return np.array([[np.abs(np.diff(f[i], axis=j)).max() for j in range(f.ndim - 1)] for i in range(f.shape[0])])


def sample_bound(f, qmax):
    """Bound on |fp32 f~(q) - fp64 f~(q)| per channel, q = p + u formed in fp32: the position of axis j rounds by at most
    U |q_j| <= U qmax_j (clamp and floor_frac are exact), which moves f~ by steps[i][j] per voxel; the blend is 3 (2-D) or
    7 (3-D) fp32 fmaf / subtractions of values and differences no larger than 2 max|f_i|, each rounding by U of that: 32 U
    max|f_i| covers either."""
    st = steps(f)
    fmax = np.abs(np.asarray(f, np.float64)).reshape(f.shape[0], -1).max(1)
    return (st * U * np.asarray(qmax)).sum(1) + 32 * U * fmax


def _thetas(nd):
    from torchregister_b200.synth import affine_theta_star
    eye = np.eye(nd, nd + 1)
    trans = eye.copy()
    trans[:, nd] = [0.1, -0.05, 0.2][:nd]
    a = np.deg2rad(10.0)
    rot = eye.copy()
    rot[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    return {"identity": eye, "translation": trans, "rotation": rot, "affine_star": affine_theta_star(nd).numpy()}


def affine_bound(theta, u, shape):
    """Bound on |kernel - compose_affine_ref| per element.  The kernel forms A and c in fp64 (each term of size <= S_r/2
    (sum|theta_r| + 1) or |M_ij| q_j, a few U64 of it), rounds them to fp32 (U each), forms q = p + u (U |q|) and
    evaluates t = c + sum_j A_ij q_j with nd fmaf (each rounding by U of |c| + sum |A_ij| |q_j|), then u + t (U |w|).
    Twice the sum of those terms."""
    nd = len(shape)
    A, c, M = affine_map(theta, shape)
    th = np.abs(np.asarray(theta, np.float64)).reshape(nd, nd + 1)
    u = np.asarray(u, np.float64)
    q = np.abs(voxel_grid(shape) + u)
    w = compose_affine_ref(theta, u, shape)
    ex = (nd,) + (1,) * nd
    mag = np.abs(c).reshape(ex) + np.einsum("ij,j...->i...", np.abs(A), q)
    f64 = 8 * U64 * (np.einsum("ij,j...->i...", np.abs(M), q)
                     + (np.array(shape, np.float64) * (th.sum(1)[::-1] + 2)).reshape(ex))   # S_r, r = nd-1-i
    return 2 * ((nd + 2) * U * mag + U * np.abs(u) + U * np.abs(w) + f64)


def _outward(shape, seed=0):
    """A smooth flow plus a linear expansion that sends p + u past every face of the volume by up to ~6 voxels."""
    from torchregister_b200.synth import smooth_flow
    u = smooth_flow(shape, 2.0)[0].numpy().astype(np.float64)
    p = voxel_grid(shape)
    for j, S in enumerate(shape):
        u[j] += 6.0 * (2 * p[j] / (S - 1) - 1) + 0.37 * (seed + 1) / (j + 1)
    q = p + u
    for j, S in enumerate(shape):
        assert q[j].min() < -1 and q[j].max() > S, "the flow must reach past both faces of axis %d" % j
    return u.astype(np.float32)


def _close(got, ref, bound, what):
    got = np.asarray(got, np.float64)
    err = np.abs(got - ref)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), "%s: NaN masks differ" % what
    ok = np.isnan(ref) | (err <= bound)
    assert ok.all(), "%s: %d elements beyond the bound, worst excess %.3e" % (
        what, (~ok).sum(), np.nanmax(np.where(ok, 0, err - bound)))


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32))[None].to(DEV)


# ------------------------------------------------------------------------------------------------------------------
# CPU: host surface, C ABI refusals, the references themselves
# ------------------------------------------------------------------------------------------------------------------
def test_signatures_and_exports():
    import torchregister_b200 as tr
    from torchregister_b200 import transforms
    for name in ("affine_to_flow", "compose_flow", "invert_flow"):
        assert getattr(tr, name) is getattr(transforms, name)
    params = inspect.signature(tr.invert_flow).parameters
    for name, default in (("max_iter", 50), ("tol", 1e-3)):
        assert params[name].kind is inspect.Parameter.KEYWORD_ONLY and params[name].default == default
    assert list(inspect.signature(tr.compose_flow).parameters) == ["first", "second"]
    assert list(inspect.signature(tr.affine_to_flow).parameters) == ["theta", "shape"]


def test_no_cpu_fallback():
    import torchregister_b200 as tr
    flow = torch.zeros(1, 3, 4, 5, 6)
    for call in (lambda: tr.affine_to_flow(torch.eye(3, 4), (4, 5, 6)),
                 lambda: tr.compose_flow(torch.eye(3, 4), flow),
                 lambda: tr.compose_flow(flow, flow),
                 lambda: tr.invert_flow(flow)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()
    with pytest.raises(ValueError):
        tr.affine_to_flow(torch.eye(3, 4), (4, 5, 6, 7))


def test_abi_refusals_launch_nothing():
    """Each refusal returns before any CUDA call: without a device a call that got past its checks would return a CUDA
    error (positive) instead.  Fake device addresses are never dereferenced."""
    from torchregister_b200 import _lib
    lib = _lib.load()
    a, b, c = 1 << 40, 2 << 40, 3 << 40
    D, H, W = 4, 5, 6
    nbytes = 3 * D * H * W * 4
    ws = lib.trb_flow_workspace_bytes()
    calls = {
        "affine: NULL theta": (lib.trb_compose_affine_flow(3, None, None, D, H, W, c, None), -1),
        "affine: NULL out": (lib.trb_compose_affine_flow(3, a, b, D, H, W, None, None), -1),
        "affine: out is the flow": (lib.trb_compose_affine_flow(3, a, b, D, H, W, b, None), -1),
        "affine: out overlaps the flow": (lib.trb_compose_affine_flow(3, a, b, D, H, W, b + nbytes - 4, None), -1),
        "affine: out holds theta": (lib.trb_compose_affine_flow(3, c + 16, b, D, H, W, c, None), -1),
        "affine: 2-D, out holds theta": (lib.trb_compose_affine_flow(2, c + 8, None, 1, H, W, c, None), -1),
        "flows: NULL first": (lib.trb_compose_flows(3, None, b, D, H, W, c, None), -1),
        "flows: NULL second": (lib.trb_compose_flows(3, a, None, D, H, W, c, None), -1),
        "flows: NULL out": (lib.trb_compose_flows(3, a, b, D, H, W, None, None), -1),
        "flows: out is first": (lib.trb_compose_flows(3, a, b, D, H, W, a, None), -1),
        "flows: out is second": (lib.trb_compose_flows(2, a, b, 1, H, W, b, None), -1),
        "flows: axis of 1": (lib.trb_compose_flows(3, a, b, 1, H, W, c, None), -1),
        "invert: NULL flow": (lib.trb_invert_flow(3, None, D, H, W, 50, 1e-3, b, c, None, 0, None), -1),
        "invert: NULL out": (lib.trb_invert_flow(3, a, D, H, W, 50, 1e-3, None, c, None, 0, None), -1),
        "invert: NULL stats": (lib.trb_invert_flow(3, a, D, H, W, 50, 1e-3, b, None, None, 0, None), -1),
        "invert: out is the flow": (lib.trb_invert_flow(3, a, D, H, W, 50, 1e-3, a, c, None, 0, None), -1),
        "invert: stats in the flow": (lib.trb_invert_flow(3, a, D, H, W, 50, 1e-3, b, a + 8, None, 0, None), -1),
        # the workspace is missing too: a max_iter / tol check that let the call through would return -2, not launch
        "invert: max_iter 0": (lib.trb_invert_flow(3, a, D, H, W, 0, 1e-3, b, c, None, 0, None), -1),
        "invert: max_iter 1001": (lib.trb_invert_flow(3, a, D, H, W, 1001, 1e-3, b, c, None, 0, None), -1),
        "invert: tol 0": (lib.trb_invert_flow(3, a, D, H, W, 50, 0.0, b, c, None, 0, None), -1),
        "invert: tol < 0": (lib.trb_invert_flow(2, a, 1, H, W, 50, -1.0, b, c, None, 0, None), -1),
        "invert: tol inf": (lib.trb_invert_flow(3, a, D, H, W, 50, float("inf"), b, c, None, 0, None), -1),
        "invert: tol nan": (lib.trb_invert_flow(3, a, D, H, W, 50, float("nan"), b, c, None, 0, None), -1),
        "invert: no workspace": (lib.trb_invert_flow(3, a, D, H, W, 50, 1e-3, b, c, None, ws, None), -2),
        "invert: small workspace": (lib.trb_invert_flow(3, a, D, H, W, 50, 1e-3, b, c, 4 << 40, ws - 8, None), -2),
        "invert: axis beyond 2^22": (lib.trb_invert_flow(2, a, 1, 2, (1 << 22) + 8, 50, 1e-3, b, c, None, 0, None), -3),
    }
    for name, (rc, want) in calls.items():
        assert rc == want, "%s: rc %d, expected %d (%s)" % (name, rc, want, lib.trb_last_error().decode())


@pytest.mark.parametrize("shape", [(9, 11), (5, 7, 6)], ids=str)
def test_references_match_torch(shape):
    """sample_border against torch's fp64 grid_sample(padding_mode='border', align_corners=True) at positions inside and
    outside the volume (lattice points and the far faces included), and compose_affine_ref's T(p) against affine_grid
    (align_corners=False) un-normalised as grid_sample does.  Both are fp64 restatements: 1e-12."""
    from torchregister_b200.synth import affine_theta_star
    nd = len(shape)
    g = np.random.default_rng(5)
    img = g.random((nd,) + shape)
    pos = g.uniform(-3, max(shape) + 3, (nd,) + shape)
    pos[:, 0] = np.array(shape, np.float64).reshape((nd,) + (1,) * (nd - 1)) - 1      # exactly on the far faces
    pos[:, 1] = np.round(pos[:, 1])                                                     # lattice points
    sizes = np.array(shape, np.float64).reshape((nd,) + (1,) * nd)
    grid = torch.from_numpy(np.moveaxis((2 * pos / (sizes - 1) - 1)[::-1], 0, -1).copy())[None]
    ref = F.grid_sample(torch.from_numpy(img)[None], grid, mode="bilinear", padding_mode="border",
                        align_corners=True)[0].numpy()
    got = np.stack([sample_border(img[i], pos) for i in range(nd)])
    assert np.abs(got - ref).max() <= 1e-12
    for theta in (affine_theta_star(nd).numpy(), _thetas(nd)["rotation"]):
        ag = F.affine_grid(torch.from_numpy(theta)[None], [1, 1] + list(shape), align_corners=False)[0].numpy()
        T = np.stack([((ag[..., k] + 1) * shape[nd - 1 - k] - 1) / 2 for k in range(nd)][::-1])
        mine = voxel_grid(shape) + compose_affine_ref(theta, np.zeros((nd,) + shape), shape)
        assert np.abs(mine - T).max() <= 1e-12


# ------------------------------------------------------------------------------------------------------------------
# GPU: affine -> flow
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_affine_to_flow_matches_fp64(shape):
    import torchregister_b200 as tr
    nd = len(shape)
    zero = np.zeros((nd,) + shape)
    for name, theta in _thetas(nd).items():
        th = torch.tensor(theta, dtype=torch.float32)
        th64 = th.double().numpy()                       # the kernel reads the fp32 theta
        for arg in (th.view(1, nd, nd + 1).to(DEV), th.reshape(-1).to(DEV)):
            w = tr.affine_to_flow(arg, shape)
            assert w.shape == (1, nd) + shape and w.dtype == torch.float32
            _close(w[0].cpu().numpy(), compose_affine_ref(th64, zero, shape), affine_bound(th64, zero, shape), name)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_affine_to_flow_warps_like_the_affine_warp(shape):
    """warp_flow(m, affine_to_flow(theta)) against warp_affine(theta, m) on a smooth blob volume: both sample m at T(p),
    through different fp32 chains.  Position error along coordinate r: the affine kernel's, fewer than 16 roundings of
    at most (sum_c |theta_rc| + 1) S_r / 2 each; the flow chain's, affine_bound for w plus the flow warp's normalise /
    un-normalise round trip of p + w (at most 6 roundings of |p + w| <= S_r + |w|).  A bilinear sample moves by at most
    the largest step of the zero-padded m along r per voxel of position error; each blend adds 16 U (values in [0, 1])."""
    import torchregister_b200 as tr
    import torchregister_b200.functional as TF
    from torchregister_b200.synth import make_pair
    nd = len(shape)
    m = make_pair(shape, "identity", noise=0)[0]
    mm = m[0, 0].double().numpy()
    pad = np.pad(mm, 1)
    for name, theta in _thetas(nd).items():
        th = torch.tensor(theta, dtype=torch.float32)
        th64 = th.double().numpy()
        w = tr.affine_to_flow(th.view(1, nd, nd + 1).to(DEV), shape)
        got = TF.warp_flow(m.to(DEV), w)[0, 0].cpu().numpy()
        ref = TF.warp_affine(th.to(DEV), m.to(DEV))[0, 0].cpu().numpy()
        wref = compose_affine_ref(th64, np.zeros((nd,) + shape), shape)
        wb = affine_bound(th64, np.zeros((nd,) + shape), shape)
        tol = 32 * U
        for i in range(nd):
            r = nd - 1 - i
            S = shape[i]
            pos_err = 16 * U * (np.abs(th64[r]).sum() + 1) * S / 2 + wb[i].max() + 6 * U * (S + np.abs(wref[i]).max())
            tol += np.abs(np.diff(pad, axis=i)).max() * pos_err
        err = np.abs(got.astype(np.float64) - ref).max()
        assert err <= tol, "%s: %.3e > %.3e" % (name, err, tol)


# ------------------------------------------------------------------------------------------------------------------
# GPU: composition
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES + [BIG], ids=str)
def test_compose_theta_then_flow_matches_fp64(shape):
    import torchregister_b200 as tr
    nd = len(shape)
    u = _outward(shape)
    for name, theta in _thetas(nd).items():
        th = torch.tensor(theta, dtype=torch.float32)
        th64 = th.double().numpy()
        w = tr.compose_flow(th.view(1, nd, nd + 1).to(DEV), _cuda(u))
        _close(w[0].cpu().numpy(), compose_affine_ref(th64, u, shape), affine_bound(th64, u, shape), name)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES + [BIG], ids=str)
def test_compose_flow_then_flow_matches_fp64(shape):
    """Tolerance: sample_bound for f~ at q = p + u (|q_j| <= S_j + max|u_j|), plus the rounding of u + f~ (U |w|)."""
    import torchregister_b200 as tr
    from torchregister_b200.synth import smooth_flow
    nd = len(shape)
    u = _outward(shape)
    f = smooth_flow(shape[::-1], 3.0)[0].numpy()
    f = np.ascontiguousarray(np.stack([f[nd - 1 - i].T for i in range(nd)]))        # a field unlike u
    w = tr.compose_flow(_cuda(f), _cuda(u))[0].cpu().numpy()
    ref = compose_flows_ref(f, u)
    qmax = np.array(shape, np.float64) + np.abs(u).reshape(nd, -1).max(1)
    bound = sample_bound(f, qmax) + U * np.abs(ref).reshape(nd, -1).max(1)
    _close(w, ref, bound.reshape((nd,) + (1,) * nd), "flow then flow")
    # exact cases: p + 0 is a lattice point, where the blend returns the corner itself; a zero field samples to 0
    zero = torch.zeros((1, nd) + shape, device=DEV)
    assert torch.equal(tr.compose_flow(_cuda(f), zero), _cuda(f))
    assert torch.equal(tr.compose_flow(zero, _cuda(u)), _cuda(u))


# ------------------------------------------------------------------------------------------------------------------
# GPU: inverse
# ------------------------------------------------------------------------------------------------------------------
def _residual_bound(u, v):
    """Bound on |fp32 residual - fp64 residual| at v: sample_bound at q = p + v plus the roundings of v + s (U (|v| +
    |s|)) and of the max; twice that for the rounding of the bound's own terms."""
    nd = u.shape[0]
    vmax = np.nanmax(np.abs(v))
    qmax = np.array(u.shape[1:], np.float64) + vmax
    return 2 * (sample_bound(u, qmax).max() + 2 * U * (vmax + np.abs(u).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,amp", [((37, 50, 61), 1.0), ((97, 130), 3.0), (BIG, 1.0)], ids=str)
def test_invert_flow_converges_to_the_fp64_fixed_point(shape, amp):
    import torchregister_b200 as tr
    from torchregister_b200.synth import smooth_flow
    u = smooth_flow(shape, amp)[0].numpy()
    L = lipschitz(u)
    assert L < 0.8, L
    tol, max_iter = 1e-3, 50
    v_t, info = tr.invert_flow(_cuda(u), max_iter=max_iter, tol=tol)
    v = v_t[0].cpu().numpy().astype(np.float64)
    e = _residual_bound(u, v)
    assert info["n_not_converged"] == 0 and info["n_nonfinite"] == 0
    r64 = residual_ref(u, v)
    assert r64.max() <= tol + e, (r64.max(), tol, e)
    assert abs(info["max_residual"] - r64.max()) <= e
    vstar = fixed_point_ref(u)
    assert np.abs(v - vstar).max() <= (tol + e + 1e-12) / (1 - L)
    # the iteration count: the fp32 and fp64 iterates stay within e / (1 - L) of each other (the error of one step,
    # contracted), so their residuals within band; only voxels whose fp64 residual came that close to tol may stop at a
    # different iteration
    band = (2 + L) * e / (1 - L)
    _, _, k, bad, amb = invert_ref(u, max_iter, tol, band)
    assert not bad.any()
    n = k.size
    assert abs(info["mean_iterations"] * n - k.sum()) <= amb.sum() * max_iter, (info["mean_iterations"], k.mean(), amb.sum())
    assert info["mean_iterations"] >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(37, 50, 61), (97, 130)], ids=str)
def test_invert_flow_reports_a_folding_field(shape):
    """A field compressed past the fold (L > 1) in one region: the call returns within max_iter and counts the voxels
    whose residual stays above tol, which are those whose fp64 residual at the returned field exceeds tol up to the
    evaluation bound."""
    import torchregister_b200 as tr
    from torchregister_b200.synth import smooth_flow
    nd = len(shape)
    u = smooth_flow(shape, 1.0)[0].numpy().astype(np.float64)
    p = voxel_grid(shape)
    cen = [s / 2.0 for s in shape]
    sig = min(shape) / 6.0
    r2 = sum((p[j] - cen[j]) ** 2 for j in range(nd))
    u[nd - 1] += -4.0 * (p[nd - 1] - cen[nd - 1]) * np.exp(-r2 / (2 * sig * sig))
    u = u.astype(np.float32)
    assert lipschitz(u) > 1
    tol = 1e-3
    v_t, info = tr.invert_flow(_cuda(u), max_iter=30, tol=tol)
    v = v_t[0].cpu().numpy().astype(np.float64)
    assert info["n_not_converged"] > 0 and info["n_nonfinite"] == 0
    assert 1 <= info["mean_iterations"] <= 30
    e = _residual_bound(u, v)
    r64 = residual_ref(u, v)
    assert int((r64 > tol + e).sum()) <= info["n_not_converged"] <= int((r64 > tol - e).sum())
    assert abs(info["max_residual"] - r64.max()) <= e


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(12, 13, 14), (15, 17)], ids=str)
def test_nonfinite_input(shape):
    """u = 0.25 everywhere, so every sample position p + u (or p - 0.25 in the inverse) lies a quarter voxel from the
    lattice and the cells that read a given voxel are unambiguous; one NaN in u, and (composition of flows) one in f.
    NaN must appear exactly where the fp64 definition puts it, channel by channel; the inverse counts those voxels."""
    import torchregister_b200 as tr
    nd = len(shape)
    a = tuple(s // 2 for s in shape)
    b = tuple(s // 3 for s in shape)
    u = np.full((nd,) + shape, 0.25, np.float32)
    u[(1,) + a] = np.nan
    th = _thetas(nd)["affine_star"].astype(np.float32)
    w = tr.compose_flow(torch.from_numpy(th).to(DEV), _cuda(u))[0].cpu().numpy()
    ref = compose_affine_ref(th.astype(np.float64), u, shape)
    assert np.array_equal(np.isnan(w), np.isnan(ref)) and int(np.isnan(ref).any(0).sum()) == 1
    f = np.random.default_rng(0).uniform(-1, 1, (nd,) + shape).astype(np.float32)
    w = tr.compose_flow(_cuda(f), _cuda(u))[0].cpu().numpy()
    assert np.array_equal(np.isnan(w), np.isnan(compose_flows_ref(f, u)))
    f[(0,) + b] = np.nan
    u[(1,) + a] = 0.25
    w = tr.compose_flow(_cuda(f), _cuda(u))[0].cpu().numpy()
    ref = compose_flows_ref(f, u)
    assert np.array_equal(np.isnan(w), np.isnan(ref))
    assert int(np.isnan(ref[0]).sum()) == 2 ** nd and not np.isnan(ref[1:]).any()
    u[(1,) + a] = np.nan
    v, info = tr.invert_flow(_cuda(u))
    bad = np.isnan(v[0].cpu().numpy())
    _, _, _, bad_ref, _ = invert_ref(u, 50, 1e-3)
    assert np.array_equal(bad, np.broadcast_to(bad_ref, bad.shape))
    assert info["n_nonfinite"] == int(bad_ref.sum()) == 2 ** nd
    assert info["n_not_converged"] == 0 and info["max_residual"] == 0.0


@pytest.mark.gpu
def test_invert_flow_is_bit_reproducible():
    import torchregister_b200 as tr
    from torchregister_b200.synth import smooth_flow
    u = smooth_flow(BIG, 1.5).to(DEV)
    runs = [tr.invert_flow(u, max_iter=20, tol=1e-5) for _ in range(2)]
    assert torch.equal(runs[0][0], runs[1][0])
    assert runs[0][1] == runs[1][1]


# ------------------------------------------------------------------------------------------------------------------
# GPU: the pipeline end to end
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rigid_affine_flow_pipeline_composes_to_one_field():
    import torchregister_b200 as tr
    from torchregister_b200.synth import make_pair
    shape = (24, 28, 32)
    mov, tgt = make_pair(shape, "affine")
    rig = tr.Register(mode="rigid", device=DEV, weight=[0.5, 0.5, 0.0])
    rig.optim(mov, tgt, lr=1e-3, max_epochs=20, reg0=torch.tensor([0.02, -0.01, 0.03, 0.05, -0.05, 0.02], device=DEV))
    aff = tr.Register(mode="affine", device=DEV, weight=[0.5, 0.5, 0.0])
    aff.optim(mov, tgt, lr=1e-3, max_epochs=20, theta0=rig.theta)
    flo = tr.Register(mode="flow", device=DEV, weight=[0.5, 0.5, 0.0], flow_param="direct", smooth=2.0)
    flo.optim(tr.get_affine_warp(aff.theta, mov.to(DEV)).detach(), tgt, lr=0.05, max_epochs=20)
    theta, flow = aff.theta.detach(), flo.theta.detach()
    w = tr.compose_flow(theta, flow)
    th64 = theta.reshape(3, 4).double().cpu().numpy()
    u = flow[0].cpu().numpy()
    _close(w[0].cpu().numpy(), compose_affine_ref(th64, u, shape), affine_bound(th64, u, shape), "pipeline")
    jac = tr.jacobian_determinant(w)
    assert jac["n_nonfinite"] == 0 and jac["min"] > 0
    assert lipschitz(w[0].cpu().numpy()) < 0.8
    inv, info = tr.invert_flow(w)
    assert info["n_not_converged"] == 0 and info["n_nonfinite"] == 0 and info["max_residual"] <= 1e-3
