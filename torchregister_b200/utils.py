"""Host-side mirror of the reference's building blocks (TR/utils.py) for the hot path.

Same public names and call signatures as the reference so `from utils import ...`
style code keeps working; the arithmetic of the warp and of the similarity runs in
libtrb_b200.so (see functional.py).  The flow network (Attention_UNet) is a dense
conv stack outside the gather/stencil path and stays PyTorch/cuDNN, as SURVEY.md
§8a-9 scopes it; it is re-written here (not copied) with identical parameter names
so reference state_dicts load.
"""
from __future__ import annotations

from math import ceil

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as TF

EPSILON = 1E-10

__all__ = ["EPSILON", "NCCLoss", "LNCCLoss", "SSDLoss", "NMILoss", "norm", "padNd", "Theta", "Regressor", "SpatialTransformer",
           "attention_grid", "Attention_UNet", "Edge3D", "get_sobel_kernel3D"]


# --------------------------------------------------------------------------- #
# similarity modules (API parity).  Inside Register/rigid/affine/flow the MSE and
# NCC terms are recognised by type and evaluated by the fused CUDA kernels; the
# nn.Module forwards below exist for users who call the criteria directly.
# --------------------------------------------------------------------------- #
class NCCLoss(nn.Module):
    """Global normalised cross-correlation, loss = (1 - NCC) * alpha
    (reference utils.py:186-205; `grad_edges` and `device` are accepted and unused there too)."""

    def __init__(self, alpha=100, grad_edges=True, device='cpu'):
        super().__init__()
        self.NCC = None
        self.alpha = alpha

    def forward(self, y, yp):
        a = y - torch.mean(y)
        b = yp - torch.mean(yp)
        self.NCC = torch.sum(a * b) / ((torch.sum(a ** 2) * torch.sum(b ** 2) + EPSILON) ** 0.5)
        return (1 - self.NCC) * self.alpha


class LNCCLoss(nn.Module):
    """EXTENSION (no counterpart in the reference): local (windowed) normalised cross-correlation, VoxelMorph's NCC with
    the sign turned so the loss is >= 0: loss = 1 - mean over all voxels of cc, cc = A^2 / (B C + eps) over a win^nd box
    with zero padding (include/trb.h: trb_lncc_forward).  forward(y, yp) = crit(target, warped), the order of the
    reference's criteria; the gradient flows to yp only.  CUDA fp32 [N,1,(D,)H,W] only, on the kernels of csrc/lncc.cu.
    Recognised by type in direct flow mode, where it runs inside the epoch."""

    def __init__(self, win=9, eps=1e-5):
        super().__init__()
        self.win = TF.check_lncc_window(win)
        if not (float(eps) > 0 and float(eps) < float('inf')):
            raise ValueError("eps must be finite and > 0 (got %r)" % (eps,))
        self.eps = float(eps)

    def forward(self, y, yp):
        if isinstance(y, torch.Tensor) and y.requires_grad:
            raise ValueError("LNCCLoss differentiates w.r.t. the warped image yp only: y (the target) must not require grad")
        TF.check_lncc_pair(y, yp)
        return _LnccFn.apply(yp, y, self.win, self.eps)


class _LnccFn(torch.autograd.Function):
    """autograd node: forward = trb_lncc_forward (keeps alpha, beta, gamma), backward = trb_lncc_backward."""

    @staticmethod
    def forward(ctx, yp, y, win, eps):
        stats, coef = TF.lncc_forward(y, yp, win, eps)
        ctx.win = win
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(y, yp, coef)
        return stats[1].float()

    @staticmethod
    def backward(ctx, grad_out):
        y, yp, coef = ctx.saved_tensors
        return TF.lncc_backward(y, yp, coef, ctx.win) * grad_out, None, None, None


class SSDLoss(nn.Module):
    """Sum of squared differences times alpha (reference utils.py:208-221; unused by any loop)."""

    def __init__(self, alpha=3):
        super().__init__()
        self.SSD = None
        self.alpha = alpha

    def forward(self, y, yp):
        self.SSD = torch.sum((y - yp) ** 2)
        return self.SSD * self.alpha


class _KDEMutualInfoFn(torch.autograd.Function):
    """|NMI - 1| * alpha averaged over chunks, for chunked samples t_s, w_s of shape [n, P], differentiable in w_s.

    Same arithmetic as the reference's K_gauss / PDF_xis / get_pdf / NMI (utils.py:18-79), including the swapped
    min/max of the bin range (:45-49), the 1/(2*pi) kernel constant (:19) and the "joint" density being a 1-D KDE
    over the concatenation of both images (:62-63) — but evaluated in blocks of bins with the backward written
    out by hand, so the [n, P, 256] temporaries (8 GB each in 3-D) and their autograd copies never exist."""

    @staticmethod
    def _bins(sig, steps):
        hi, lo = torch.max(sig).item(), torch.min(sig).item()
        return torch.linspace(hi, lo, steps, dtype=torch.float, device=sig.device).to(sig.dtype)

    @staticmethod
    def _pdf(sig, xs, h, block):
        cols = []
        for i0 in range(0, xs.numel(), block):
            z = (sig.unsqueeze(-1) - xs[i0:i0 + block]) / h
            cols.append((1 / h) * torch.mean((1 / (2 * torch.pi)) * torch.exp(-(z ** 2) / 2), dim=1))
        return torch.cat(cols, dim=1)

    @staticmethod
    def forward(ctx, t_s, w_s, bins, h, alpha, block):
        with torch.no_grad():
            both = torch.cat((t_s, w_s), dim=1)
            x1, x2, xj = (_KDEMutualInfoFn._bins(v, bins) for v in (t_s, w_s, both))
            pdf1 = _KDEMutualInfoFn._pdf(t_s, x1, h, block)
            pdf2 = _KDEMutualInfoFn._pdf(w_s, x2, h, block)
            pdfj = 0.5 * (_KDEMutualInfoFn._pdf(t_s, xj, h, block) + _KDEMutualInfoFn._pdf(w_s, xj, h, block))
        with torch.enable_grad():                      # the [n, 256] tail of the graph is tiny: let autograd do it
            q2 = pdf2.detach().requires_grad_(True)
            qj = pdfj.detach().requires_grad_(True)
            p1 = pdf1 / torch.sum(pdf1, dim=1, keepdim=True)
            p2 = q2 / torch.sum(q2, dim=1, keepdim=True)
            pj = qj / torch.sum(qj, dim=1, keepdim=True)
            e1 = -torch.sum(p1 * -torch.log2(p1 + EPSILON), dim=1)
            e2 = -torch.sum(p2 * -torch.log2(p2 + EPSILON), dim=1)
            ej = -torch.sum(pj * -torch.log2(pj + EPSILON), dim=1)
            mi = e1 + e2 - ej
            loss = torch.mean(torch.abs(2 * mi / (e1 + e2) - 1.) * alpha)
            g2, gj = torch.autograd.grad(loss, (q2, qj))
        ctx.save_for_backward(w_s, x2, xj, g2, gj)
        ctx.h, ctx.block = h, block
        return loss.detach()

    @staticmethod
    def backward(ctx, grad_out):
        w_s, x2, xj, g2, gj = ctx.saved_tensors
        h, block = ctx.h, ctx.block
        n_s = w_s.shape[1]
        grad = torch.zeros_like(w_s)
        c = (1 / h) * (1 / (2 * torch.pi))
        for xs, g, cnt in ((x2, g2, n_s), (xj, gj, 2 * n_s)):
            for i0 in range(0, xs.numel(), block):
                z = (w_s.unsqueeze(-1) - xs[i0:i0 + block]) / h
                # d/dw of c * exp(-z^2/2) / cnt  =  -c * z / h * exp(-z^2/2) / cnt
                grad += torch.sum(g[:, None, i0:i0 + block] * (-(c / (h * cnt)) * z * torch.exp(-(z ** 2) / 2)), dim=-1)
        return None, grad * grad_out, None, None, None, None


class NMILoss(nn.Module):
    """Normalised-mutual-information term of the reference's default loss (utils.py:224-259): nearest-resample
    both images to (2*patch)^n, view as 2^n chunks of patch^n, 256-bin Gaussian KDE (bandwidth 3) of target,
    warped and their concatenation, loss = mean(|NMI - 1|) * alpha.  One fp32 CUDA pair with the default bins/patch
    runs on the kernels of csrc/nmi.cu (SURVEY.md §8 f-1); anything else (CPU tensors, batches, other bin counts)
    on the PyTorch restatement below (the GPU tests check the kernels against it)."""

    def __init__(self, alpha=1000, bins=256, patch_size=100, bandwidth=3, block=8):
        super().__init__()
        self.bins, self.alpha, self.patch, self.bandwidth, self.block = bins, alpha, patch_size, bandwidth, block

    def _chunks(self, v):
        nd = v.dim() - 2
        r = self.patch * 2
        v = F.interpolate(v, size=(r,) * nd, mode='nearest')
        return v.reshape((2 ** nd) * v.shape[0] * v.shape[1], -1)

    def _cuda_term(self, y):
        """CUDA kernels (csrc/nmi.cu) for one fp32 [1,1,...] pair with the default bins/patch; the target's resample
        and marginal are cached while the same target tensor comes back (every epoch of a registration)."""
        from . import functional as TF
        # The cache holds a REFERENCE to the target tensor and compares identity (+ in-place version): a different
        # tensor that the caching allocator happens to place at the same address can therefore never hit it.
        key = (y._version, tuple(y.shape), float(self.bandwidth), float(self.alpha))
        if getattr(self, "_term_target", None) is not y or getattr(self, "_term_key", None) != key:
            self._term = TF.NmiTerm(y, self.bandwidth, self.alpha)
            self._term_key = key
            self._term_target = y
        return self._term

    def forward(self, y, yp):
        if (y.is_cuda and yp.is_cuda and y.dtype == torch.float32 and yp.dtype == torch.float32 and y.shape == yp.shape
                and y.shape[0] == 1 and y.shape[1] == 1 and self.bins == 256 and self.patch == 100 and y.dim() in (4, 5)):
            return _NmiCudaFn.apply(yp, self._cuda_term(y))
        return _KDEMutualInfoFn.apply(self._chunks(y), self._chunks(yp), self.bins, float(self.bandwidth),
                                      float(self.alpha), self.block)


class _NmiCudaFn(torch.autograd.Function):
    """autograd node around trb_nmi_loss_grad: the backward w.r.t. the warped image is produced with the forward."""

    @staticmethod
    def forward(ctx, yp, term):
        loss, gout = term.loss_grad(yp, 1.0, want_grad=yp.requires_grad)
        ctx.save_for_backward(gout if gout is not None else torch.empty(0, device=yp.device))
        return loss[0].float().clone()

    @staticmethod
    def backward(ctx, grad_out):
        (gout,) = ctx.saved_tensors
        return gout * grad_out, None


def get_sobel_kernel3D(n1=1, n2=2, n3=2):
    """The nine 3x3x3 Sobel-type kernels of the reference (utils.py:82-127): axis kernels Sx, Sy, Sz, then six diagonal
    ones derived from two base diagonals by transposition.  Returned as a list of [3,3,3] float64 tensors in the
    reference's order [Sx, Sy, Sz, Sd11, Sd12, Sd21, Sd22, Sd31, Sd32]."""
    a, b, c = float(n1), float(n2), float(n2 * n3)
    plane = torch.tensor([[a, b, a], [b, c, b], [a, b, a]], dtype=torch.float64)        # smoothing across the two other axes
    d = torch.tensor([-1.0, 0.0, 1.0], dtype=torch.float64)
    # the reference indexes its literals [i][j][k]: Sx differentiates along k, Sy along j, Sz along i
    Sx = plane[:, :, None] * d[None, None, :]
    Sy = plane[:, None, :] * d[None, :, None]
    Sz = d[:, None, None] * plane[None, :, :]
    row = torch.tensor([a, b, a], dtype=torch.float64)                                  # weights of the three [i] slabs
    diag1 = torch.tensor([[0, 1, 2], [-1, 0, 1], [-2, -1, 0]], dtype=torch.float64)     # pattern of Sd11 for n1=1, n2=2
    diag2 = torch.tensor([[-2, -1, 0], [-1, 0, 1], [0, 1, 2]], dtype=torch.float64)     # pattern of Sd12

    def slab(pattern, lo, hi):
        # |1| entries -> lo, |2| entries -> hi, signs kept
        return torch.sign(pattern) * torch.where(pattern.abs() == 2, torch.tensor(hi, dtype=torch.float64),
                                                 torch.where(pattern.abs() == 1, torch.tensor(lo, dtype=torch.float64),
                                                             torch.tensor(0.0, dtype=torch.float64)))
    Sd11 = torch.stack([slab(diag1, a, b), slab(diag1, b, c), slab(diag1, a, b)])
    Sd12 = torch.stack([slab(diag2, a, b), slab(diag2, b, c), slab(diag2, a, b)])
    Sd21 = Sd11.permute(2, 1, 0)                 # numpy .T of a 3-D array reverses the axes
    Sd22 = Sd12.permute(2, 1, 0)
    Sd31 = torch.stack([-m.t() for m in Sd21])   # [-S.T for S in Sd11.T]
    Sd32 = torch.stack([m.t() for m in Sd22])    # [S.T for S in Sd12.T]
    del row
    return [Sx, Sy, Sz, Sd11, Sd12, Sd21, Sd22, Sd31, Sd32]


class Edge3D():
    """Sobel edge pre-filter of the reference (utils.py:130-183), as one CUDA stencil pass + one threshold pass
    (csrc/edge.cu) instead of 9*C conv3d calls on a padded copy.  Same constructor and call signature.

    Deviation, deliberate: the reference's default pad `a=5000` makes its reflect padding raise for every volume smaller
    than 5001 voxels per axis (SURVEY.md §2 #12), i.e. the filter cannot be used at its defaults.  Any pad `a >= 1`
    smaller than the volume gives the same output (the pad is cropped again and the stencil reaches one voxel), so the
    default here is `a=1`; `a >= min(shape)` raises like torch's reflect padding does."""

    def __init__(self, n1=1, n2=2, n3=2, device='cpu'):
        self.device = device
        ks = get_sobel_kernel3D(n1, n2, n3)
        self.weights = torch.stack(ks).to(torch.float32).reshape(9, 27).contiguous()      # host copy, (x,y,z) order

    def __call__(self, img, a=1, thresh=[0.2, 0.9], return_norm=False):
        import ctypes as C
        from . import _lib
        TF.require_cuda(img, "img")
        if img.dim() != 5:
            raise ValueError("Edge3D expects a 5-D tensor (b, c, x, y, z)")
        B, Cc, X, Y, Z = (int(v) for v in img.shape)
        if a < 1 or a >= min(X, Y, Z):
            raise RuntimeError("Padding size should be less than the corresponding input dimension (reflect pad %d, "
                               "volume %dx%dx%d); pass 1 <= a < min(shape)" % (a, X, Y, Z))
        src = img.detach().contiguous()
        out = torch.empty(B, 1, X, Y, Z, dtype=torch.float32, device=src.device)
        nrm = torch.empty_like(out) if return_norm else None
        minmax = torch.empty(2, dtype=torch.int32, device=src.device)
        w = (C.c_float * (9 * 27))(*self.weights.reshape(-1).tolist())
        self._keep = w                                  # the async upload reads it until the stream gets there
        with torch.cuda.device(src.device):
            _lib.check(_lib.load().trb_edge3d(src.data_ptr(), out.data_ptr(), B, Cc, X, Y, Z, w, float(thresh[0]), float(thresh[1]),
                                              minmax.data_ptr(), None if nrm is None else nrm.data_ptr(),
                                              torch.cuda.current_stream(src.device).cuda_stream), "edge3d")
        return (out, nrm) if return_norm else out


def norm(x):
    """Min-max normalisation (reference utils.py:262-267)."""
    try:
        lo = torch.min(x)
        return (x - lo) / ((torch.max(x) - lo) + 1E-9)
    except Exception:
        print('WARNING: Input could not be normalized!')


def padNd(input_, target, device='cpu', mode='constant', value=0):
    """Centre-pad `input_` to the spatial size of `target` (reference utils.py:271-277)."""
    dims = input_.dim() - 2
    pads = []
    for i in reversed(range(dims)):
        delta = target.shape[2 + i] - input_.shape[2 + i]
        hi = ceil(delta / 2)             # the reference puts the larger half AFTER the data
        pads += [delta - hi, hi]
    return F.pad(input_, tuple(pads), mode=mode, value=value).to(dtype=torch.float, device=device)


# --------------------------------------------------------------------------- #
# rigid parametrisation (API parity; the optimisation loop evaluates it on device
# inside the fused kernel's epilogue)
# --------------------------------------------------------------------------- #
class Theta(nn.Module):
    """6 -> 12 (ZYX Euler + 0.25*tanh translation) or 3 -> 6 (reference utils.py:280-310)."""

    def forward(self, x, max_translate=0.25):
        if len(x) > 3:
            cps, sps = torch.cos(x[0]), torch.sin(x[0])
            cth, sth = torch.cos(x[1]), torch.sin(x[1])
            cph, sph = torch.cos(x[2]), torch.sin(x[2])
            t = max_translate * torch.tanh(x[3:6])
            return torch.stack((cps * cth, sph * sps * cth - cph * sth, cph * sps * cth + sph * sth, t[0],
                                cps * sth, sph * sps * sth + cph * cth, cph * sps * sth - sph * cth, t[1],
                                -sps, sph * cps, cph * cps, t[2])).flatten()
        c, s = torch.cos(x[0]), torch.sin(x[0])
        return torch.stack((c, -s, x[1], s, c, x[2])).flatten()


class Regressor(nn.Module):
    """Rigid parameters, initialised with torch.rand on `device` (reference utils.py:313-330)."""

    def __init__(self, moving, device):
        super().__init__()
        self.reg = nn.Parameter(torch.rand(6 if moving.dim() == 5 else 3, device=device), requires_grad=True)
        self.thetas = Theta()

    def forward(self):
        theta = self.thetas(self.reg)
        return theta.view(1, 3, 4) if theta.shape[-1] == 12 else theta.view(1, 2, 3)


# --------------------------------------------------------------------------- #
# flow warp
# --------------------------------------------------------------------------- #
class _WarpFlowFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, flow, mode='bilinear'):
        ctx.save_for_backward(src, flow)
        ctx.mode = mode
        return TF.warp_flow(src, flow, mode=mode)

    @staticmethod
    def backward(ctx, grad_out):
        src, flow = ctx.saved_tensors
        if ctx.mode == 'nearest':
            # a nearest sample is piecewise constant in the position: d/d flow is 0 (torch's nearest grid_sample gives
            # the grid the same zero gradient)
            return None, torch.zeros_like(flow) if ctx.needs_input_grad[1] else None, None
        if src.shape[1] != 1:
            raise NotImplementedError("gradient of the flow warp is implemented for single-channel src")
        dflow = TF.warp_flow_vjp(src, flow, grad_out.contiguous()) if ctx.needs_input_grad[1] else None
        return None, dflow, None       # no gradient to `src`: the moving image is constant on this path


class SpatialTransformer(nn.Module):
    """N-D spatial transformer: samples `src` at voxel index + flow (voxel units, channel i
    displaces spatial axis i), zeros padding (reference utils.py:333-365), bilinear or nearest
    (grid_sample's modes; 'nearest' carries label maps and gives the flow a zero gradient).
    The identity index grid the reference keeps as a buffer is computed in the kernel."""

    def __init__(self, size, mode='bilinear'):
        super().__init__()
        if mode not in ('bilinear', 'nearest'):
            raise NotImplementedError("mode must be 'bilinear' or 'nearest' (got %r)" % (mode,))
        self.mode = mode
        self.size = tuple(int(s) for s in size)

    def forward(self, src, flow):
        return _WarpFlowFn.apply(src, flow, self.mode)


# --------------------------------------------------------------------------- #
# flow network: PyTorch/cuDNN host code (SURVEY.md §8a-9), same topology and
# parameter names as reference utils.py:368-559
# --------------------------------------------------------------------------- #
class _InstanceNormFn(torch.autograd.Function):
    """y = InstanceNorm(relu?(x)) on the CUDA kernels of csrc/instnorm.cu (forward keeps x and (mean, rstd))."""

    @staticmethod
    def forward(ctx, x, eps, relu):
        from . import functional as TF
        y, stats = TF.instance_norm_forward(x, eps, relu)
        ctx.save_for_backward(x, stats)
        ctx.relu = relu
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        from . import functional as TF
        x, stats = ctx.saved_tensors
        return TF.instance_norm_backward(x, dy, stats, ctx.relu), None, None


class _GatedInstanceNormFn(torch.autograd.Function):
    """y = InstanceNorm(x * gate), gate [1,1,*spatial] shared by the channels of one sample (the attention gate's bnorm(x * w))."""

    @staticmethod
    def forward(ctx, x, gate, eps):
        from . import functional as TF
        x, gate = x.contiguous(), gate.contiguous()
        y, stats = TF.instance_norm_forward(x, eps, False, gate)
        ctx.save_for_backward(x, gate, stats)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        from . import functional as TF
        x, gate, stats = ctx.saved_tensors
        dx, dgate = TF.instance_norm_backward(x, dy, stats, False, gate)
        return dx, dgate, None


class _InstanceNormB200:
    """Mixin over nn.InstanceNorm{2,3}d: float32 CUDA inputs of a plain instance norm (affine=False, no running statistics:
    the reference's configuration, utils.py:368-520) run on csrc/instnorm.cu — PyTorch parallelises instance norm over
    N*C only, which leaves a 2..32-channel U-Net on a handful of thread blocks (391 ms of a 492 ms epoch at 256^3).
    `fuse_relu`: the module also applies the ReLU that precedes it in the reference's blocks (one pass fewer each way)."""

    fuse_relu = False

    def forward(self, x):
        plain = not self.affine and not self.track_running_stats
        if plain and x.is_cuda and x.dtype == torch.float32 and x.dim() >= 3:
            return _InstanceNormFn.apply(x, float(self.eps), bool(self.fuse_relu))
        return super().forward(F.relu(x) if self.fuse_relu else x)


class InstanceNorm3dB200(_InstanceNormB200, nn.InstanceNorm3d):
    pass


class InstanceNorm2dB200(_InstanceNormB200, nn.InstanceNorm2d):
    pass


class _ThinConv3dFn(torch.autograd.Function):
    """conv3d (kernel 3, stride 1, valid) with <= 4 channels each way on csrc/thinconv.cu."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        from . import functional as TF
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return TF.thin_conv3d_forward(x, weight, bias)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        from . import functional as TF
        x, weight = ctx.saved_tensors
        gx, gw, gb = TF.thin_conv3d_backward(x, weight, gy, ctx.needs_input_grad[0], ctx.needs_input_grad[1],
                                             ctx.has_bias and ctx.needs_input_grad[2])
        return gx, gw, gb


class _PointConv3dFn(torch.autograd.Function):
    """1x1x1 conv3d (uniform stride, no padding) with <= 4 channels each way on csrc/thinconv.cu."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride):
        from . import functional as TF
        ctx.save_for_backward(x, weight)
        ctx.has_bias, ctx.stride = bias is not None, stride
        return TF.point_conv3d_forward(x, weight, bias, stride)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        from . import functional as TF
        x, weight = ctx.saved_tensors
        gx, gw, gb = TF.point_conv3d_backward(x, weight, gy, ctx.stride, ctx.needs_input_grad[0], ctx.needs_input_grad[1],
                                              ctx.has_bias and ctx.needs_input_grad[2])
        return gx, gw, gb, None


class Conv3dB200(nn.Conv3d):
    """nn.Conv3d whose thin 3x3x3 valid layers (<= 4 channels each way: the full-resolution layers of the flow U-Net at the
    reference's n = 32) run on csrc/thinconv.cu instead of cuDNN's tensor-core GEMMs, whose tiles are 64..256 output
    channels wide (74 ms of a 106 ms epoch at 256^3); likewise the 1x1x1 layers of the attention gates (uniform stride).  Same
    parameters, same state_dict; everything else is nn.Conv3d."""

    def _thin(self, x):
        from .functional import THIN_CONV_MAX_CHANNELS as M
        return (x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and self.weight.dtype == torch.float32
                and tuple(self.kernel_size) == (3, 3, 3) and tuple(self.stride) == (1, 1, 1) and tuple(self.dilation) == (1, 1, 1)
                and self.groups == 1 and self.padding in ((0, 0, 0), 0, 'valid') and min(x.shape[2:]) >= 3
                and ((self.in_channels <= M and self.out_channels <= M) or (self.in_channels, self.out_channels) in ((8, 4), (4, 8), (8, 8))))

    def _point(self, x):
        from .functional import THIN_CONV_MAX_CHANNELS as M
        return (x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.shape[0] == 1 and self.weight.dtype == torch.float32
                and tuple(self.kernel_size) == (1, 1, 1) and len(set(self.stride)) == 1 and tuple(self.dilation) == (1, 1, 1)
                and self.groups == 1 and self.padding in ((0, 0, 0), 0, 'valid') and self.in_channels <= M and self.out_channels <= M)

    def forward(self, x):
        if self._thin(x):
            return _ThinConv3dFn.apply(x, self.weight, self.bias)
        if self._point(x):
            return _PointConv3dFn.apply(x, self.weight, self.bias, int(self.stride[0]))
        return super().forward(x)


class _UpConv3dFn(torch.autograd.Function):
    """conv_transpose3d (kernel 2, stride 2) with <= 4 channels each way on csrc/thinconv.cu."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        from . import functional as TF
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return TF.up_conv3d_forward(x, weight, bias)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        from . import functional as TF
        x, weight = ctx.saved_tensors
        return TF.up_conv3d_backward(x, weight, gy, ctx.needs_input_grad[0], ctx.needs_input_grad[1],
                                     ctx.has_bias and ctx.needs_input_grad[2])


class ConvTranspose3dB200(nn.ConvTranspose3d):
    """nn.ConvTranspose3d whose thin 2x2x2 stride-2 layers (<= 4 channels each way: the U-Net's last up-sampling at n = 32) run
    as a streaming kernel of csrc/thinconv.cu — every output voxel has one source voxel.  Same parameters, same state_dict."""

    def _thin(self, x):
        from .functional import THIN_CONV_MAX_CHANNELS as M
        return (x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.shape[0] == 1 and self.weight.dtype == torch.float32
                and tuple(self.kernel_size) == (2, 2, 2) and tuple(self.stride) == (2, 2, 2) and tuple(self.dilation) == (1, 1, 1)
                and tuple(self.padding) == (0, 0, 0) and tuple(self.output_padding) == (0, 0, 0) and self.groups == 1
                and self.in_channels <= M and self.out_channels <= M)

    def forward(self, x, output_size=None):
        if output_size is None and self._thin(x):
            return _UpConv3dFn.apply(x, self.weight, self.bias)
        return super().forward(x, output_size)


def _relu_inorm(inorm, channels):
    """The reference's `nn.ReLU(), nn.InstanceNorm(co)` pair with the ReLU folded into the norm; an Identity keeps the
    positions (and therefore the parameter names of the convolutions) of the reference's nn.Sequential."""
    m = inorm(channels)
    m.fuse_relu = True
    return [nn.Identity(), m]


def _nd(dims):
    return (Conv3dB200, ConvTranspose3dB200, InstanceNorm3dB200, nn.MaxPool3d) if dims == 3 else \
           (nn.Conv2d, nn.ConvTranspose2d, InstanceNorm2dB200, nn.MaxPool2d)


class attention_grid(nn.Module):
    """Additive attention gate with a stride-3 1x1 projection of the skip (reference utils.py:368-406)."""

    def __init__(self, x_c, g_c, i_c, stride=3, mode='nearest', dims=3):
        super().__init__()
        conv, _, inorm, _ = _nd(dims)
        self.input_filter = conv(x_c, i_c, kernel_size=1, stride=stride, bias=False)
        self.gate_filter = conv(g_c, i_c, kernel_size=1, stride=1, bias=True)
        self.psi = conv(i_c, 1, kernel_size=1, stride=1, bias=True)
        self.bnorm = inorm(i_c)
        self.mode = mode

    def forward(self, x, g, device):
        a, b = self.input_filter(x), self.gate_filter(g)
        if a.shape[-1] < b.shape[-1]:
            a = padNd(a, b, device)
        elif a.shape[-1] > b.shape[-1]:
            b = padNd(b, a, device)
        w = torch.sigmoid(self.psi(F.relu(a + b)))
        w = F.interpolate(w, size=x.shape[2:], mode=self.mode)
        b = self.bnorm
        if (isinstance(b, _InstanceNormB200) and not b.affine and not b.track_running_stats and not b.fuse_relu and x.is_cuda
                and x.dtype == torch.float32 and w.dtype == torch.float32 and x.shape[0] == 1 and w.shape[1] == 1
                and x.shape[1] <= 64 and tuple(w.shape[2:]) == tuple(x.shape[2:])):
            return _GatedInstanceNormFn.apply(x, w, float(b.eps)), w       # the product x * w is never materialised
        return self.bnorm(x * w), w


class Attention_UNet(nn.Module):
    """5-level valid-convolution attention U-Net whose 1x1 head emits the flow, followed by the
    warp of its own input (reference utils.py:409-559).  Widths 64/n .. 1024/n."""

    def __init__(self, img_size, mode='nearest', in_c=1, n=1):
        super().__init__()
        dims = len(img_size)
        conv, convT, inorm, pool = _nd(dims)
        w = [int(c / n) for c in (64, 128, 256, 512, 1024)]

        def double(ci, co, up_to=None):
            mods = [conv(ci, co, kernel_size=3), *_relu_inorm(inorm, co),
                    conv(co, co, kernel_size=3), *_relu_inorm(inorm, co)]
            if up_to is not None:
                mods += [convT(co, up_to, kernel_size=2, stride=2), *_relu_inorm(inorm, up_to)]
            return nn.Sequential(*mods)

        self.layer1 = double(in_c, w[0])
        self.skip1 = attention_grid(w[0], w[0], w[0], dims=dims)
        self.layer2 = double(w[0], w[1])
        self.skip2 = attention_grid(w[1], w[1], w[1], dims=dims)
        self.layer3 = double(w[1], w[2])
        self.skip3 = attention_grid(w[2], w[2], w[2], dims=dims)
        self.layer4 = double(w[2], w[3])
        self.skip4 = attention_grid(w[3], w[3], w[3], dims=dims)
        self.layer5 = double(w[3], w[4], up_to=w[3])
        self.layer6 = double(w[4], w[3], up_to=w[2])
        self.layer7 = double(w[3], w[2], up_to=w[1])
        self.layer8 = double(w[2], w[1], up_to=w[0])
        self.layer9 = double(w[1], w[0])
        self.out = conv(w[0], dims, kernel_size=1)
        self.maxpool = pool(kernel_size=2, stride=2)
        self.warp = SpatialTransformer(img_size, mode)

    def features(self, x, device):
        """Decoder output BEFORE the final zero padding and the 1x1 `out` convolution (reference utils.py:523-551):
        [1, w0, ...] at the valid-convolution size.  flow_field(x) == out(padNd(features(x), x))."""
        y1 = self.layer1(x)
        y2 = self.layer2(self.maxpool(y1))
        y3 = self.layer3(self.maxpool(y2))
        y4 = self.layer4(self.maxpool(y3))
        y = self.layer5(self.maxpool(y4))
        for skip, enc, dec in ((self.skip4, y4, self.layer6), (self.skip3, y3, self.layer7),
                               (self.skip2, y2, self.layer8), (self.skip1, y1, self.layer9)):
            gated, _ = skip(enc, y, device=device)
            y = dec(torch.cat((gated, padNd(y, gated, device=device)), dim=1))
        return y

    def flow_field(self, x, device):
        """The network part only: x -> flow (no warp)."""
        return self.out(padNd(self.features(x, device), x, device=device))

    def forward(self, x, device, out_att=False):
        flow = self.flow_field(x, device)
        return self.warp(x, flow), flow
