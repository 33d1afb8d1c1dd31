"""Quality measures of a registration result: the Jacobian determinant of a flow (is the deformation valid?) and the
Dice overlap of label maps (do warped segmentations line up?).  CUDA only, like the rest of the package."""
from __future__ import annotations

import math
from typing import Optional

import torch

from . import _lib
from . import functional as TF
from ._lib import check

__all__ = ["jacobian_determinant", "dice"]

JAC_NSTATS = 8


def jacobian_determinant(flow: torch.Tensor, *, return_field: bool = False) -> dict:
    """Jacobian determinant of phi(p) = p + u(p) for a flow u [1, nd, (D,) H, W] in voxel units (channel i displaces
    spatial axis i, the layout of every flow here).  J = I + du/dp with numpy.gradient's differences (central inside,
    one-sided at the ends; every spatial axis must be >= 2), in fp64 on the device (csrc/jacobian.cu).

    Returns a dict of Python numbers, read from the device in one copy:
      n_folding, fraction_folding   voxels with det <= 0 (folded), and their share of all voxels;
      min, max, mean, std           of det (std: population);
      log_std                       std of log(clamp(det, 1e-9, 1e9)), the spread of local volume change;
      n_nonfinite                   voxels whose det is inf or NaN (a non-finite flow); every other entry is over the
                                    finite ones only;
    plus `field` (fp32 [1, 1, (D,) H, W]) with return_field=True."""
    TF.require_cuda(flow, "flow")
    if flow.dim() not in (4, 5) or flow.shape[0] != 1 or flow.shape[1] != flow.dim() - 2:
        raise ValueError("flow must be [1, nd, (D,) H, W] with nd spatial axes (got shape %s)" % (tuple(flow.shape),))
    ndim = flow.dim() - 2
    dims = [1] * (3 - ndim) + [int(s) for s in flow.shape[2:]]
    lib = _lib.load()
    dev = flow.device
    f = flow.detach().contiguous()
    field = torch.empty((1, 1) + tuple(flow.shape[2:]), dtype=torch.float32, device=dev) if return_field else None
    stats = torch.empty(JAC_NSTATS, dtype=torch.float64, device=dev)
    ws = TF._flow_ws(dev)
    with torch.cuda.device(dev):
        check(lib.trb_flow_jacobian(ndim, f.data_ptr(), dims[0], dims[1], dims[2], TF._ptr(field), stats.data_ptr(),
                                    ws.data_ptr(), ws.numel(), TF._stream(dev)), "flow_jacobian")
    n_fold, n_bad, lo, hi, s1, s2, l1, l2 = stats.cpu().tolist()
    n = dims[0] * dims[1] * dims[2]
    n_ok = n - int(n_bad)
    nan = float("nan")
    mean = s1 / n_ok if n_ok else nan
    lmean = l1 / n_ok if n_ok else nan
    out = {
        "n_folding": int(n_fold),
        "fraction_folding": n_fold / n,
        "min": lo if n_ok else nan,
        "max": hi if n_ok else nan,
        "mean": mean,
        "std": math.sqrt(max(s2 / n_ok - mean * mean, 0.0)) if n_ok else nan,
        "log_std": math.sqrt(max(l2 / n_ok - lmean * lmean, 0.0)) if n_ok else nan,
        "n_nonfinite": int(n_bad),
    }
    if return_field:
        out["field"] = field
    return out


def dice(a: torch.Tensor, b: torch.Tensor, n_labels: Optional[int] = None) -> torch.Tensor:
    """Dice overlap 2|A_l & B_l| / (|A_l| + |B_l|) of every label l of two label maps [N, 1, ...] of equal shape (integer
    values, or float values that hold integers, e.g. the output of a nearest warp).  Returns fp64 [N, n_labels], NaN
    where a label is absent from both maps.  n_labels=None: the largest label + 1.  A value that is not an integer in
    [0, n_labels) raises ValueError."""
    for t, name in ((a, "a"), (b, "b")):
        if not isinstance(t, torch.Tensor):
            raise TypeError("%s must be a torch.Tensor" % name)
        if not t.is_cuda:
            raise RuntimeError("torchregister_b200 runs on CUDA (B200, sm_100a) only; %s is on %s. "
                               "There is no CPU fallback." % (name, t.device))
    if a.shape != b.shape or a.dim() < 3 or a.shape[1] != 1:
        raise ValueError("a and b must be label maps [N, 1, ...] of equal shape (got %s and %s)"
                         % (tuple(a.shape), tuple(b.shape)))
    if a.is_floating_point() or b.is_floating_point():
        for t, name in ((a, "a"), (b, "b")):
            if t.is_floating_point() and not bool((t == torch.round(t)).all()):
                raise ValueError("%s holds values that are not integers" % name)
    la, lb = a.reshape(a.shape[0], -1).long(), b.reshape(b.shape[0], -1).long()
    lo = int(torch.minimum(la.min(), lb.min()))
    hi = int(torch.maximum(la.max(), lb.max()))
    if n_labels is None:
        n_labels = hi + 1
    if lo < 0 or hi >= n_labels:
        raise ValueError("labels must lie in [0, %d) (got values in [%d, %d])" % (n_labels, lo, hi))
    N, L = int(a.shape[0]), int(n_labels)
    base = torch.arange(N, device=a.device).unsqueeze(1) * L
    ia, ib = (la + base).reshape(-1), (lb + base).reshape(-1)
    size_a = torch.bincount(ia, minlength=N * L).reshape(N, L).double()
    size_b = torch.bincount(ib, minlength=N * L).reshape(N, L).double()
    inter = torch.bincount(ia[ia == ib], minlength=N * L).reshape(N, L).double()
    return 2.0 * inter / (size_a + size_b)          # 0 / 0 = NaN: label in neither map
