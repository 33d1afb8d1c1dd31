"""Algebra of registration transforms on the GPU: an affine result as a flow, composition of a theta or a flow with a
flow, and the inverse of a flow (csrc/transform.cu).  With them a rigid -> affine -> flow pipeline becomes ONE field:
volumes and label maps are resampled once, `jacobian_determinant` sees the whole mapping, and target-space labels can be
taken back to the moving volume.

Conventions: flows are fp32 [1, nd, (D,) H, W] in voxel units, channel i displacing spatial axis i ((z, y, x) in 3-D),
and a flow u stands for p -> p + u(p), the position `warp_flow(m, u)` samples m at.  A theta ([1, nd, nd+1] or its nd*(nd+1)
values) stands for the position `get_affine_warp(theta, m)` samples at.  No autograd: the results are plain tensors.
CUDA only, N == 1, every spatial axis >= 2."""
from __future__ import annotations

import torch

from . import _lib
from . import functional as TF
from ._lib import check

__all__ = ["affine_to_flow", "compose_flow", "invert_flow"]

INV_NSTATS = 4


def _flow_dims(flow: torch.Tensor, name: str):
    TF.require_cuda(flow, name)
    if flow.dim() not in (4, 5) or flow.shape[0] != 1 or flow.shape[1] != flow.dim() - 2:
        raise ValueError("%s must be a flow [1, nd, (D,) H, W] with nd spatial axes (got shape %s)"
                         % (name, tuple(flow.shape)))
    nd = flow.dim() - 2
    return nd, [1] * (3 - nd) + [int(s) for s in flow.shape[2:]]


def _theta(theta, nd: int, dev) -> torch.Tensor:
    """theta as nd*(nd+1) contiguous fp32 values on `dev`; no host synchronisation."""
    if not isinstance(theta, torch.Tensor):
        raise TypeError("theta must be a torch.Tensor")
    if not theta.is_cuda:
        raise RuntimeError("torchregister_b200 runs on CUDA (B200, sm_100a) only; theta is on %s. "
                           "There is no CPU fallback." % (theta.device,))
    if theta.numel() != nd * (nd + 1):
        raise ValueError("a %d-D theta has %d values ([1, %d, %d] or flat), got shape %s"
                         % (nd, nd * (nd + 1), nd, nd + 1, tuple(theta.shape)))
    return theta.detach().to(device=dev, dtype=torch.float32).reshape(-1).contiguous()


def affine_to_flow(theta: torch.Tensor, shape) -> torch.Tensor:
    """The flow w with warp_flow(m, w) = get_affine_warp(theta, m): w(p) = T(p) - p, T theta's map in voxel units.
    theta [1, nd, nd+1] or its nd*(nd+1) values (CUDA); shape: the spatial shape ((D,) H, W).  -> [1, nd, *shape]."""
    shape = tuple(int(s) for s in shape)
    if len(shape) not in (2, 3):
        raise ValueError("shape must be the 2 or 3 spatial sizes ((D,) H, W), got %s" % (shape,))
    nd = len(shape)
    th = _theta(theta, nd, getattr(theta, "device", None))
    dev = th.device
    dims = [1] * (3 - nd) + list(shape)
    out = torch.empty((1, nd) + shape, dtype=torch.float32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        check(lib.trb_compose_affine_flow(nd, th.data_ptr(), None, dims[0], dims[1], dims[2], out.data_ptr(),
                                          TF._stream(dev)), "compose_affine_flow")
    return out


def compose_flow(first: torch.Tensor, second: torch.Tensor) -> torch.Tensor:
    """The one flow w for "first, then second": warp_flow(m, w) = warp_flow(warp(m, first), second) up to the
    interpolation of the intermediate volume, which w avoids.  Name and order mirror `compose_theta`.
      first a theta ([1, nd, nd+1] or flat): w(p) = T(p + u(p)) - p, exact (T is affine);
      first a flow f of second's shape:      w(p) = u(p) + f~(p + u(p)), f~ bi/trilinear with border padding;
    u = second, a flow.  A non-finite position p + u(p) gives NaN at that voxel."""
    nd, dims = _flow_dims(second, "second")
    dev = second.device
    u = second.detach().contiguous()
    out = torch.empty_like(u)
    lib = _lib.load()
    if isinstance(first, torch.Tensor) and first.shape == second.shape:
        TF.require_cuda(first, "first")
        f = first.detach().contiguous()
        if f.device != dev:
            raise ValueError("first and second must be on the same device")
        with torch.cuda.device(dev):
            check(lib.trb_compose_flows(nd, f.data_ptr(), u.data_ptr(), dims[0], dims[1], dims[2], out.data_ptr(),
                                        TF._stream(dev)), "compose_flows")
        return out
    if isinstance(first, torch.Tensor) and first.numel() != nd * (nd + 1):
        raise ValueError("first must be a theta (%d values) or a flow of second's shape %s (got shape %s)"
                         % (nd * (nd + 1), tuple(second.shape), tuple(first.shape)))
    th = _theta(first, nd, dev)
    with torch.cuda.device(dev):
        check(lib.trb_compose_affine_flow(nd, th.data_ptr(), u.data_ptr(), dims[0], dims[1], dims[2], out.data_ptr(),
                                          TF._stream(dev)), "compose_affine_flow")
    return out


def invert_flow(flow: torch.Tensor, *, max_iter: int = 50, tol: float = 1e-3):
    """The inverse v of a flow u: p + v(p) + u(p + v(p)) = p, i.e. warp_flow(warp_flow(m, v), u) ~ m, by the per-voxel
    fixed point v = -u~(p + v) (u~ bi/trilinear with border padding), started at -u(p) and stopped when the residual
    |v + u~(p + v)|_inf <= tol (voxels) or after max_iter evaluations (1..1000).  It converges where u is a contraction
    (a mild, fold-free flow); otherwise it reports what did not converge.  -> (inverse [1, nd, ...], info), info read in
    one device-to-host copy:
      n_not_converged   finite voxels whose residual is still > tol;
      n_nonfinite       voxels that met a non-finite position or residual (NaN in the inverse);
      max_residual      over the finite voxels (NaN if there are none);
      mean_iterations   residual evaluations per voxel."""
    nd, dims = _flow_dims(flow, "flow")
    max_iter, tol = int(max_iter), float(tol)
    if not 1 <= max_iter <= 1000:
        raise ValueError("max_iter must lie in [1, 1000] (got %d)" % max_iter)
    if not (0.0 < tol < float("inf")):
        raise ValueError("tol must be finite and > 0 (got %r)" % tol)
    dev = flow.device
    u = flow.detach().contiguous()
    inv = torch.empty_like(u)
    stats = torch.empty(INV_NSTATS, dtype=torch.float64, device=dev)
    ws = TF._flow_ws(dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        check(lib.trb_invert_flow(nd, u.data_ptr(), dims[0], dims[1], dims[2], max_iter, tol, inv.data_ptr(),
                                  stats.data_ptr(), ws.data_ptr(), ws.numel(), TF._stream(dev)), "invert_flow")
    n_nc, n_bad, rmax, evals = stats.cpu().tolist()
    n = dims[0] * dims[1] * dims[2]
    info = {
        "n_not_converged": int(n_nc),
        "n_nonfinite": int(n_bad),
        "max_residual": rmax if n_bad < n else float("nan"),
        "mean_iterations": evals / n,
    }
    return inv, info
