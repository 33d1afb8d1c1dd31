"""Label maps through a registration (nearest-neighbour forward warps) and the validity of a deformation (Jacobian
determinant of a flow), plus the Dice overlap.  CPU tests check the host surface; GPU tests compare the kernels with
torch's grid_sample and a numpy fp64 restatement."""
import inspect

import numpy as np
import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"


# ------------------------------------------------------------------------------------------------------------------
# CPU: the host surface
# ------------------------------------------------------------------------------------------------------------------
def test_reference_default_unet_and_nearest_transformer_construct():
    import torchregister_b200 as tr
    tr.Attention_UNet((160, 160))                      # the reference's default mode is 'nearest'
    st = tr.SpatialTransformer((8, 8, 8), "nearest")
    assert st.mode == "nearest"
    with pytest.raises(NotImplementedError):
        tr.SpatialTransformer((8, 8, 8), "bicubic")


def test_flow_register_trains_bilinear_only():
    import torchregister_b200 as tr
    with pytest.raises(NotImplementedError, match="bilinear"):
        tr.flow_register((64, 64), mode="nearest")


def test_new_keywords_are_keyword_only_with_bilinear_defaults():
    import torchregister_b200 as tr
    import torchregister_b200.functional as TF
    for fn, name, default in ((TF.warp_affine, "mode", "bilinear"), (TF.warp_flow, "mode", "bilinear"),
                              (tr.get_affine_warp, "mode", "bilinear"), (tr.Register.__call__, "mode", "bilinear"),
                              (tr.flow_register.deform, "mode", "bilinear"),
                              (tr.direct_flow_register.deform, "mode", "bilinear"),
                              (tr.jacobian_determinant, "return_field", False)):
        p = inspect.signature(fn).parameters[name]
        assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default == default, (fn, p)
    assert inspect.signature(tr.dice).parameters["n_labels"].default is None
    x = torch.zeros(1, 1, 8, 8, 8)
    with pytest.raises(ValueError, match="mode"):
        TF.warp_affine(torch.eye(3, 4), x, mode="bicubic")
    with pytest.raises(ValueError, match="mode"):
        TF.warp_flow(x, torch.zeros(1, 3, 8, 8, 8), mode="bicubic")


def test_label_and_jacobian_functions_have_no_cpu_fallback():
    import torchregister_b200 as tr
    import torchregister_b200.functional as TF
    x, flow = torch.zeros(1, 1, 8, 8, 8), torch.zeros(1, 3, 8, 8, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        TF.warp_affine(torch.eye(3, 4), x, mode="nearest")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        TF.warp_flow(x, flow, mode="nearest")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tr.get_affine_warp(torch.eye(3, 4).view(1, 3, 4), x, mode="nearest")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tr.SpatialTransformer((8, 8, 8), "nearest")(x, flow)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tr.jacobian_determinant(flow)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tr.dice(x.long(), x.long())


# ------------------------------------------------------------------------------------------------------------------
# GPU: nearest affine warps
# ------------------------------------------------------------------------------------------------------------------
def _block_labels(shape, n, block, seed):
    """Integer-valued label map [n, *shape] made of blocks of random labels 1..9."""
    g = torch.Generator().manual_seed(seed)
    coarse = torch.randint(1, 10, (n,) + tuple((s + block - 1) // block for s in shape), generator=g).float()
    for ax in range(len(shape)):
        coarse = coarse.repeat_interleave(block, dim=ax + 1)
    return coarse[(slice(None),) + tuple(slice(0, s) for s in shape)].contiguous()


def _nearest_reference(theta, labels, band=1e-3):
    """fp64 affine_grid coordinates (align_corners=False), rounded half to even.  -> (reference, compared mask,
    candidate values [2^nd, ...] for the voxels within `band` of a half-integer on some axis)."""
    N, C = labels.shape[:2]
    shape = labels.shape[2:]
    nd = len(shape)
    grid = F.affine_grid(theta.double().reshape(N, nd, nd + 1), list(labels.shape), align_corners=False)
    sizes = list(reversed(shape))                                   # grid components are (x, y[, z])
    coords = [((grid[..., k] + 1) * sizes[k] - 1) / 2 for k in range(nd)]
    near_half = [(c - torch.floor(c) - 0.5).abs() < band for c in coords]
    compared = ~torch.stack(near_half).any(0)

    def gather(idx):
        inside = torch.ones_like(idx[0], dtype=torch.bool)
        lin = torch.zeros_like(idx[0])
        stride = 1
        for k in range(nd):
            inside &= (idx[k] >= 0) & (idx[k] < sizes[k])
            lin = lin + idx[k].clamp(0, sizes[k] - 1) * stride
            stride *= sizes[k]
        flat = labels.reshape(N, C, -1)
        vals = torch.gather(flat, 2, lin.reshape(N, 1, -1).expand(N, C, -1)).reshape(labels.shape)
        return torch.where(inside.unsqueeze(1), vals, torch.zeros_like(vals))

    ref = gather([torch.round(c).long() for c in coords])           # torch.round: half to even
    cands = []
    for corner in range(2 ** nd):
        idx = []
        for k in range(nd):
            lo = torch.floor(coords[k]).long()
            pick = lo + ((corner >> k) & 1)
            idx.append(torch.where(near_half[k], pick, torch.round(coords[k]).long()))
        cands.append(gather(idx))
    return ref, compared.unsqueeze(1).expand_as(ref), torch.stack(cands)


def _check_nearest(out, labels, theta):
    ref, cmp, cands = _nearest_reference(theta, labels)
    assert cmp.float().mean().item() >= 0.98
    assert torch.equal(out[cmp], ref[cmp])
    assert bool((cands == out.unsqueeze(0)).any(0)[~cmp].all())
    values = torch.cat([labels.unique(), torch.zeros(1, device=labels.device)])
    assert bool(torch.isin(out, values).all())
    # torch's own fp32 nearest grid_sample on the same device, outside the same band
    nd = labels.dim() - 2
    grid = F.affine_grid(theta.reshape(-1, nd, nd + 1), list(labels.shape), align_corners=False)
    ts = F.grid_sample(labels, grid, mode="nearest", padding_mode="zeros", align_corners=False)
    assert torch.equal(out[cmp], ts[cmp])
    return cmp


@pytest.mark.gpu
def test_affine_nearest_3d_tma_and_gather_vs_grid_sample():
    import torchregister_b200.functional as TF
    import torchregister_b200 as tr
    shape = (37, 50, 68)                          # partial 32x16x16 tiles along every axis; W % 4 == 0 (TMA-eligible)
    labels = _block_labels(shape, 6, 5, seed=7).reshape(3, 2, *shape).to(DEV)
    small = torch.tensor([[1.01, .02, -.01, .01], [-.02, .99, .01, 0.], [.01, -.01, 1., .02]], device=DEV)
    big = torch.tensor([[0.7, -0.7, 0.1, .05], [0.7, 0.7, -0.1, 0.], [0.0, 0.14, 0.99, .02]], device=DEV)   # 45 deg
    ths = torch.stack([small, big, small * 0.98])
    tma = TF.warp_affine(ths, labels, mode="nearest")
    gather = TF.warp_affine(ths, labels, large_rotation=True, mode="nearest")
    cmp = _check_nearest(tma, labels, ths)
    _check_nearest(gather, labels, ths)
    assert torch.equal(tma[cmp], gather[cmp])
    # get_affine_warp: same values, no autograd graph
    th = small.clone().requires_grad_(True)
    out = tr.get_affine_warp(th.view(1, 3, 4), labels[:1], mode="nearest")
    assert out.grad_fn is None and torch.equal(out, TF.warp_affine(small, labels[:1], mode="nearest"))
    # bilinear stays the default
    assert torch.equal(TF.warp_affine(ths, labels), TF.warp_affine(ths, labels, mode="bilinear"))


@pytest.mark.gpu
def test_affine_nearest_2d_vs_grid_sample():
    import torchregister_b200.functional as TF
    shape = (45, 61)
    labels = _block_labels(shape, 6, 4, seed=11).reshape(3, 2, *shape).to(DEV)
    c, s = np.cos(np.pi / 4), np.sin(np.pi / 4)
    ths = torch.tensor([[[1.01, .02, .01], [-.02, .99, -.03]], [[c, -s, .05], [s, c, 0.]], [[.97, .05, 0.], [-.04, 1.02, .02]]],
                       dtype=torch.float32, device=DEV)
    out = TF.warp_affine(ths, labels, mode="nearest")
    _check_nearest(out, labels, ths)


# ------------------------------------------------------------------------------------------------------------------
# GPU: nearest flow warp, SpatialTransformer, Register round trips
# ------------------------------------------------------------------------------------------------------------------
def _reference_flow_nearest(src, flow):
    """The reference's SpatialTransformer grid (utils.py:343-365) built on the device, sampled with mode='nearest'."""
    shape = flow.shape[2:]
    vecs = [torch.arange(0, s, dtype=torch.float32, device=flow.device) for s in shape]
    locs = torch.stack(torch.meshgrid(*vecs, indexing="ij"))[None] + flow
    comps = [2 * (locs[:, i] / (s - 1) - 0.5) for i, s in enumerate(shape)]
    comps.reverse()
    return F.grid_sample(src, torch.stack(comps, dim=-1), mode="nearest", padding_mode="zeros", align_corners=True)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(33, 47), (19, 26, 35)])
def test_flow_nearest_equals_grid_sample_bitwise(shape):
    import torchregister_b200.functional as TF
    from torchregister_b200.synth import smooth_flow
    nd = len(shape)
    src = _block_labels(shape, 3, 3, seed=5).unsqueeze(0).to(DEV)
    flows = [smooth_flow(shape, 6.0).to(DEV),                          # displacements that leave the volume
             torch.full((1, nd) + shape, 0.5, device=DEV),             # exactly half a voxel: round half to even
             torch.full((1, nd) + shape, -0.5, device=DEV)]
    g = torch.Generator().manual_seed(3)
    flows.append((torch.randint(-4, 5, (1, nd) + shape, generator=g).float() * 0.5).to(DEV))
    for flow in flows:
        got = TF.warp_flow(src, flow, mode="nearest")
        assert torch.equal(got, _reference_flow_nearest(src, flow))


@pytest.mark.gpu
def test_spatial_transformer_nearest_forward_and_zero_gradient():
    import torchregister_b200 as tr
    import torchregister_b200.functional as TF
    from torchregister_b200.synth import smooth_flow
    shape = (20, 24, 28)
    src = _block_labels(shape, 2, 4, seed=9).unsqueeze(0).to(DEV)
    flow = smooth_flow(shape, 3.0).to(DEV).requires_grad_(True)
    out = tr.SpatialTransformer(shape, "nearest")(src, flow)
    assert torch.equal(out, TF.warp_flow(src, flow.detach(), mode="nearest"))
    (out * torch.rand_like(out)).sum().backward()
    assert flow.grad is not None and not bool(flow.grad.any())


@pytest.mark.gpu
def test_register_nearest_round_trips():
    import torchregister_b200 as tr
    import torchregister_b200.functional as TF
    from torchregister_b200.synth import make_pair
    shape = (24, 32, 40)
    mov, tgt = make_pair(shape, "rigid")
    labels = _block_labels(shape, 1, 4, seed=2).unsqueeze(0).to(DEV)
    reg = tr.Register(mode="rigid", device=DEV, weight=[0.5, 0.5, 0.0])
    reg.optim(mov, tgt, lr=1e-3, max_epochs=5, reg0=torch.tensor([0.02, -0.01, 0.03, 0.05, -0.05, 0.02], device=DEV))
    assert torch.equal(reg(labels, mode="nearest"), TF.warp_affine(reg.theta, labels, mode="nearest"))
    assert torch.equal(reg(mov), TF.warp_affine(reg.theta, mov.to(DEV)))
    mov, tgt = make_pair(shape, "flow")
    reg = tr.Register(mode="flow", device=DEV, weight=[0.5, 0.5, 0.0], flow_param="direct", smooth=2.0)
    reg.optim(mov, tgt, lr=0.05, max_epochs=10)
    two = torch.cat([labels, labels + 1], 1)
    assert torch.equal(reg(two, mode="nearest"), TF.warp_flow(two, reg.theta, mode="nearest"))
    assert torch.equal(reg._flowreg.deform(two, mode="nearest"), _reference_flow_nearest(two, reg.theta))


# ------------------------------------------------------------------------------------------------------------------
# GPU: Jacobian determinant
# ------------------------------------------------------------------------------------------------------------------
def _jacobian_np(u):
    """numpy fp64 restatement: J = I + np.gradient(u_i, axis=j), np.linalg.det."""
    u = u.astype(np.float64)
    nd = u.shape[0]
    J = np.empty(u.shape[1:] + (nd, nd))
    for i in range(nd):
        g = np.gradient(u[i])
        for j in range(nd):
            J[..., i, j] = g[j] + (1.0 if i == j else 0.0)
    return np.linalg.det(J)


def _folded_flow(shape, seed):
    """Smooth random flow plus a region compressed past the fold along the last axis."""
    from torchregister_b200.synth import smooth_flow
    nd = len(shape)
    u = smooth_flow(shape, 1.5).numpy()[0].astype(np.float64)
    rng = np.random.default_rng(seed)
    u += 0.05 * rng.standard_normal(u.shape)
    grids = np.meshgrid(*[np.arange(s, dtype=np.float64) for s in shape], indexing="ij")
    c = [s / 2.0 for s in shape]
    sig = max(1.0, min(shape) / 6.0)
    r2 = sum((g - cc) ** 2 for g, cc in zip(grids, c))
    u[nd - 1] += -3.0 * (grids[nd - 1] - c[nd - 1]) * np.exp(-r2 / (2 * sig * sig))
    return torch.from_numpy(u.astype(np.float32))[None]


def _check_jacobian(flow):
    import torchregister_b200 as tr
    det = _jacobian_np(flow[0].numpy())
    got = tr.jacobian_determinant(flow.to(DEV), return_field=True)
    field = got["field"].cpu().numpy()[0, 0].astype(np.float64)
    fin = np.isfinite(det)
    assert got["n_nonfinite"] == int((~fin).sum())
    assert np.array_equal(np.isfinite(field), fin)
    d = det[fin]
    assert np.all(np.abs(field[fin] - d) <= 1.2e-7 * np.abs(d) + 1e-12)
    assert got["n_folding"] == int((d <= 0).sum())
    assert got["fraction_folding"] == (d <= 0).sum() / det.size
    L = np.log(np.clip(d, 1e-9, 1e9))
    for key, ref, tol in (("mean", d.mean(), 1e-12), ("min", d.min(), 1e-12), ("max", d.max(), 1e-12),
                          ("std", d.std(), 1e-9), ("log_std", L.std(), 1e-9)):
        assert abs(got[key] - ref) <= tol * max(abs(ref), 1e-300), (key, got[key], ref)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 2), (37, 41), (2, 2, 2), (37, 41, 43), (160, 160, 160)])
def test_jacobian_vs_numpy(shape):
    flow = _folded_flow(shape, seed=len(shape))
    got = _check_jacobian(flow)
    if min(shape) > 8:
        assert got["n_folding"] > 0                   # the folded region is seen
    zero = __import__("torchregister_b200").jacobian_determinant(torch.zeros_like(flow).to(DEV), return_field=True)
    assert bool((zero["field"] == 1).all())
    assert zero["n_folding"] == 0 and zero["std"] == 0.0 and zero["mean"] == 1.0 and zero["log_std"] == 0.0


@pytest.mark.gpu
def test_jacobian_counts_nonfinite_and_is_bit_reproducible():
    import torchregister_b200 as tr
    import torchregister_b200.functional as TF
    from torchregister_b200 import _lib
    flow = _folded_flow((37, 41, 43), seed=1)
    flow[0, 1, 10, 11, 12] = float("nan")
    flow[0, 2, 0, 0, 0] = float("nan")
    got = _check_jacobian(flow)
    assert got["n_nonfinite"] > 0
    lib = _lib.load()
    f = flow.to(DEV).contiguous()
    ws = TF._flow_ws(f.device)
    runs = []
    for _ in range(2):
        stats = torch.empty(8, dtype=torch.float64, device=DEV)
        _lib.check(lib.trb_flow_jacobian(3, f.data_ptr(), 37, 41, 43, None, stats.data_ptr(), ws.data_ptr(), ws.numel(),
                                         TF._stream(f.device)), "flow_jacobian")
        runs.append(stats)
    assert torch.equal(runs[0], runs[1])
    with pytest.raises(ValueError):
        tr.jacobian_determinant(torch.zeros(1, 3, 1, 8, 8, device=DEV))       # an axis of size 1


# ------------------------------------------------------------------------------------------------------------------
# GPU: Dice
# ------------------------------------------------------------------------------------------------------------------
def _dice_np(a, b, n):
    out = np.full((a.shape[0], n), np.nan)
    for i in range(a.shape[0]):
        for l in range(n):
            sa, sb = (a[i] == l).sum(), (b[i] == l).sum()
            if sa + sb:
                out[i, l] = 2.0 * ((a[i] == l) & (b[i] == l)).sum() / (sa + sb)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.int64])
def test_dice_vs_numpy(dtype):
    import torchregister_b200 as tr
    g = torch.Generator().manual_seed(4)
    a = torch.randint(0, 5, (2, 1, 12, 14, 16), generator=g)
    b = a.clone()
    b[:, :, :6] = torch.randint(0, 5, (2, 1, 6, 14, 16), generator=g)
    got = tr.dice(a.to(DEV, dtype), b.to(DEV, dtype), n_labels=7)
    ref = _dice_np(a.numpy(), b.numpy(), 7)
    assert got.dtype == torch.float64 and got.shape == (2, 7)
    assert np.allclose(got.cpu().numpy(), ref, rtol=1e-15, atol=0, equal_nan=True)
    assert bool(torch.isnan(got[:, 5:]).all())                    # labels 5, 6 are in neither map
    same = tr.dice(a.to(DEV, dtype), a.to(DEV, dtype))
    assert same.shape == (2, 5) and bool((same == 1).all())
    with pytest.raises(ValueError):
        tr.dice(a.to(DEV, dtype), b.to(DEV, dtype), n_labels=3)
    with pytest.raises(ValueError):
        tr.dice(-a.to(DEV, dtype) - 1, b.to(DEV, dtype))
    if dtype.is_floating_point:
        with pytest.raises(ValueError):
            tr.dice(a.to(DEV, dtype) + 0.5, b.to(DEV, dtype))
