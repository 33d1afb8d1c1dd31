"""Tensor-level wrappers over the C ABI (include/trb.h).

PyTorch is used for device memory, streams and (elsewhere) torch.distributed
only; all arithmetic of the hot path runs in libtrb_b200.so.  Every function
requires CUDA tensors and raises otherwise — there is no CPU path.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import check

STATE_FLOATS = 64
S_PARAMS, S_THETA, S_BEST_THETA, S_BEST_LOSS, S_LAST_LOSS = 0, 12, 24, 36, 37
MOMENTS = 41
MODE = {"rigid": 0, "affine": 1}
OPT = {"sgd": 0, "adam": 1}


def set_kernel_path(path: str = "auto") -> None:
    """'auto': persistent multi-epoch TMA kernel when shape/alignment allow, else the direct-gather kernel;
    'direct': always the direct-gather kernel; 'tma': the per-epoch TMA kernel instead of the persistent one
    (tests / A-B timing)."""
    check(_lib.load().trb_set_kernel_path({"auto": 0, "direct": 1, "tma": 2}[path]), "set_kernel_path")


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError(
            "torchregister_b200 runs on CUDA (B200, sm_100a) only; %s is on %s. "
            "There is no CPU fallback — use the reference TorchRegister for device='cpu'." % (name, t.device))
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32 (got %s)" % (name, t.dtype))


def _vol_dims(t: torch.Tensor):
    """[N, C, (D,) H, W] -> (ndim, D, H, W)."""
    if t.dim() == 5:
        return 3, int(t.shape[2]), int(t.shape[3]), int(t.shape[4])
    if t.dim() == 4:
        return 2, 1, int(t.shape[2]), int(t.shape[3])
    raise ValueError("expected a 4-D [N,C,H,W] or 5-D [N,C,D,H,W] tensor, got shape %s" % (tuple(t.shape),))


# --------------------------------------------------------------------------- #
# base coordinates
# --------------------------------------------------------------------------- #
_TABLES = {}


def base_coords(size: int, device) -> torch.Tensor:
    """linspace(-1, 1, S) * (S - 1) / S — the per-axis base grid F.affine_grid builds
    for align_corners=False (reference call site warpings.py:24).  Computed with
    torch on the host so the values are bit-identical to the CPU reference, then
    cached on the device: three 1-D tables replace the materialised [N,D,H,W,3] grid."""
    key = (int(size), str(device))
    t = _TABLES.get(key)
    if t is None:
        if size <= 1:
            h = torch.zeros(max(size, 1), dtype=torch.float32)
        else:
            h = torch.linspace(-1, 1, size, dtype=torch.float32) * (size - 1) / size
        t = h.to(device)
        _TABLES[key] = t
    return t


# --------------------------------------------------------------------------- #
# rigid / affine registration
# --------------------------------------------------------------------------- #
class AffineProblem:
    """Device-resident state for `n_pairs` independent rigid/affine registrations
    of equally shaped volume pairs (one fused launch per epoch covers the batch)."""

    def __init__(self, moving: torch.Tensor, target: torch.Tensor, mode: str, params0: torch.Tensor,
                 max_epochs: int, large_rotation: Optional[bool] = None):
        require_cuda(moving, "moving")
        require_cuda(target, "target")
        if moving.shape != target.shape:
            raise ValueError("moving %s and target %s shapes differ" % (tuple(moving.shape), tuple(target.shape)))
        if moving.shape[1] != 1:
            raise ValueError("registration expects single-channel volumes [N,1,...]; got C=%d" % moving.shape[1])
        if mode not in MODE:
            raise ValueError("mode must be 'rigid' or 'affine'")
        self.lib = _lib.load()
        self.device = moving.device
        self.mode = mode
        self.ndim, self.D, self.H, self.W = _vol_dims(moving)
        self.n_pairs = int(moving.shape[0])
        self.moving = moving.contiguous()
        self.target = target.contiguous()
        self.pair_stride = self.D * self.H * self.W
        self.nt = self.ndim * (self.ndim + 1)
        self.np = (6 if self.ndim == 3 else 3) if mode == "rigid" else self.nt
        self.xb = base_coords(self.W, self.device)
        self.yb = base_coords(self.H, self.device)
        self.zb = base_coords(self.D, self.device) if self.ndim == 3 else None
        # the kernel-variant hint below needs the start parameters on the host: take them before the upload when the
        # caller passed host data (no device round trip, no stream synchronisation)
        p0_src = torch.as_tensor(params0, dtype=torch.float32)
        p0_host = p0_src.detach().reshape(-1, self.np).contiguous() if not p0_src.is_cuda else None
        self.state = torch.zeros(self.n_pairs, STATE_FLOATS, dtype=torch.float32, device=self.device)
        if p0_host is not None:
            # host parameters go up as kernel arguments: a pageable H2D copy would block the caller until everything
            # already queued on the stream (e.g. the previous stage's epochs) has finished
            if p0_host.shape[0] not in (1, self.n_pairs):
                raise ValueError("params0 must have %d rows" % self.n_pairs)
            with torch.cuda.device(self.device):
                check(self.lib.trb_affine_set_params(self.state.data_ptr(), self.n_pairs, self.np, p0_host.data_ptr(),
                                                     int(p0_host.shape[0]), _stream(self.device)), "affine_set_params")
            p0 = None
        else:
            p0 = p0_src.to(self.device).reshape(-1, self.np)
            if p0.shape[0] == 1 and self.n_pairs > 1:
                p0 = p0.expand(self.n_pairs, self.np)
            if p0.shape[0] != self.n_pairs:
                raise ValueError("params0 must have %d rows" % self.n_pairs)
            self.state[:, : self.np] = p0
        self.max_epochs = int(max_epochs)
        self.loss_log = torch.zeros(self.n_pairs, max(self.max_epochs, 1), dtype=torch.float32, device=self.device)
        ws_bytes = int(self.lib.trb_affine_workspace_bytes(self.n_pairs))
        self.workspace = torch.zeros(ws_bytes, dtype=torch.uint8, device=self.device)   # zero: tickets start at 0
        self.epoch = 0
        self._default_scratch = None          # run_default: warped volumes + d term / d warped
        with torch.cuda.device(self.device):
            check(self.lib.trb_affine_init_state(self.ndim, MODE[mode], self.state.data_ptr(), self.n_pairs,
                                                 _stream(self.device)), "affine_init_state")
        # Kernel variant for the fused 3-D loop: TMA-staged boxes when the start theta keeps an output tile's source
        # footprint inside the staged box (rotations up to ~5 degrees), the L1-gather variant otherwise (e.g. the
        # reference's own torch.rand(6) start).  Decided ONCE from the initial parameters (one small D2H read if they
        # live on the device); both variants compute the same values.
        self.flags = 0
        if self.ndim == 3:
            if large_rotation is None:
                large_rotation = self._start_needs_gather(p0 if p0_host is None else p0_host)
            self.flags = 1 if large_rotation else 0
        # gather variant: a pair volume (x neighbours side by side) halves the number of gathers; it costs 2x the moving
        # volumes in memory and one pass to build
        self.moving_pairs = None
        import os
        force = os.environ.get("TRB_PAIRS")           # test / A-B hook: "0" scalar gathers, "1" pair volume, "2" quad volume
        if self.flags & 1 and self.pair_stride == self.D * self.H * self.W and force != "0":
            qbytes = int(self.lib.trb_affine_quads_bytes(self.n_pairs, self.D, self.H, self.W))
            pbytes = int(self.lib.trb_affine_pairs_bytes(self.n_pairs, self.D, self.H, self.W))
            quad = pbytes > PAIR_VOLUME_L2_BYTES if force is None else force == "2"
            nbytes = qbytes if quad else pbytes
            if nbytes <= PAIR_VOLUME_MAX_BYTES:
                self.moving_pairs = torch.empty(nbytes // 4, dtype=torch.float32, device=self.device)
                build = self.lib.trb_affine_build_quads if quad else self.lib.trb_affine_build_pairs
                with torch.cuda.device(self.device):
                    check(build(self.moving.data_ptr(), self.moving_pairs.data_ptr(), self.n_pairs, self.D, self.H, self.W,
                                _stream(self.device)), "affine_build_pairs")
                    check(self.lib.trb_affine_attach_pairs(self.workspace.data_ptr(), self.workspace.numel(), self.n_pairs,
                                                           self.moving_pairs.data_ptr(), _stream(self.device)), "affine_attach_pairs")
                self.flags |= 4 if quad else 2          # TRB_FLAG_QUAD_VOLUME / TRB_FLAG_PAIR_VOLUME

    def _start_needs_gather(self, p0: torch.Tensor) -> bool:
        import ctypes as C
        ph = p0.detach().to("cpu", torch.float64)
        if self.mode == "rigid":
            c, s_, t = torch.cos(ph[:, :3]), torch.sin(ph[:, :3]), 0.25 * torch.tanh(ph[:, 3:6])
            cps, cth, cph = c[:, 0], c[:, 1], c[:, 2]
            sps, sth, sph = s_[:, 0], s_[:, 1], s_[:, 2]
            th = torch.stack([cps * cth, sph * sps * cth - cph * sth, cph * sps * cth + sph * sth, t[:, 0],
                              cps * sth, sph * sps * sth + cph * cth, cph * sps * sth - sph * cth, t[:, 1],
                              -sps, sph * cps, cph * cps, t[:, 2]], dim=1)          # utils.py:290-305
        else:
            th = ph
        th = th.to(torch.float32).contiguous()
        misfit = 0
        for i in range(th.shape[0]):
            row = (C.c_float * 12)(*th[i].tolist())
            misfit += 0 if self.lib.trb_affine_tile_fits(self.D, self.H, self.W, row) else 1
        return 2 * misfit > th.shape[0]

    def run(self, n_epochs: int, lr: float, w_mse: float, w_ncc: float, optimiser: str = "sgd",
            betas=(0.9, 0.999), eps: float = 1e-8) -> None:
        """Enqueue `n_epochs` fused epochs (asynchronous; no host sync)."""
        if n_epochs <= 0:
            return
        if self.epoch + n_epochs > self.max_epochs:
            raise ValueError("max_epochs exceeded")
        with torch.cuda.device(self.device):
            check(self.lib.trb_affine_optim_ex(
                self.ndim, MODE[self.mode], self.moving.data_ptr(), self.target.data_ptr(), self.pair_stride,
                self.n_pairs, self.D, self.H, self.W, self.xb.data_ptr(), self.yb.data_ptr(), _ptr(self.zb),
                self.state.data_ptr(), self.loss_log.data_ptr(), self.loss_log.shape[1], self.epoch, n_epochs,
                float(w_mse), float(w_ncc), float(lr), OPT[optimiser], float(betas[0]), float(betas[1]), float(eps),
                int(self.flags), self.workspace.data_ptr(), self.workspace.numel(), _stream(self.device)), "affine_optim")
        self.epoch += n_epochs

    def run_default(self, n_epochs: int, lr: float, w_mse: float, w_ncc: float, w_nmi: float, term: "NmiSourceTerm",
                    optimiser: str = "sgd", betas=(0.9, 0.999), eps: float = 1e-8) -> None:
        """Enqueue `n_epochs` epochs of the reference's DEFAULT loss [MSE, NCC, NMI] (warpings.py:36-40,123-159) with one
        C-ABI call: the NMI term runs in its source-space form (`term`, built on this problem's targets)."""
        if n_epochs <= 0:
            return
        if self.epoch + n_epochs > self.max_epochs:
            raise ValueError("max_epochs exceeded")
        if term.n_pairs != self.n_pairs or term.ndim != self.ndim:
            raise ValueError("run_default needs a term built on the same batch")
        if self._default_scratch is None:
            self._default_scratch = torch.empty((2,) + tuple(self.target.shape), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.trb_affine_optim_nmi(
                self.ndim, MODE[self.mode], self.moving.data_ptr(), self.target.data_ptr(), self.n_pairs, self.D, self.H, self.W,
                self.xb.data_ptr(), self.yb.data_ptr(), _ptr(self.zb), self.state.data_ptr(), self.loss_log.data_ptr(),
                self.loss_log.shape[1], self.epoch, n_epochs, float(w_mse), float(w_ncc), float(w_nmi), float(lr),
                OPT[optimiser], float(betas[0]), float(betas[1]), float(eps), int(self.flags), term.bandwidth, term.alpha,
                term.lo, term.hi, self._default_scratch[0].data_ptr(), self._default_scratch[1].data_ptr(),
                term.workspace.data_ptr(), term.workspace.numel(), self.workspace.data_ptr(), self.workspace.numel(),
                _stream(self.device)), "affine_optim_nmi")
        self.epoch += n_epochs

    # -- sharded (z-slab) form, fused: the epoch kernel all-reduces the moments itself through peer memory
    def run_peer(self, n_epochs: int, s_begin: int, s_end: int, mailbox_ptrs, rank: int, world: int, seq0: int,
                 lr: float, w_mse: float, w_ncc: float, optimiser: str = "sgd", betas=(0.9, 0.999), eps: float = 1e-8) -> None:
        """`mailbox_ptrs[r]`: rank r's mailbox (2*8*48+8 float64, zeroed) as mapped into this process.  Every rank makes
        the same calls; `seq0` >= 1 advances by n_epochs per call (parallel.PeerMailbox keeps it).  n_epochs == 0 only
        validates (raises if this shape / slab cannot take the fused path)."""
        if n_epochs < 0:
            return
        if self.ndim != 3 or self.n_pairs != 1:
            raise ValueError("the fused sharded epoch handles one 3-D pair")
        if self.epoch + n_epochs > self.max_epochs:
            raise ValueError("max_epochs exceeded")
        import ctypes
        arr = (ctypes.c_void_p * world)(*[int(v) for v in mailbox_ptrs])
        with torch.cuda.device(self.device):
            check(self.lib.trb_affine_optim_peer(
                self.moving.data_ptr(), self.target.data_ptr(), self.D, self.H, self.W, int(s_begin), int(s_end),
                self.xb.data_ptr(), self.yb.data_ptr(), _ptr(self.zb), MODE[self.mode],
                self.state.data_ptr(), self.loss_log.data_ptr(), self.loss_log.shape[1], self.epoch, n_epochs,
                float(w_mse), float(w_ncc), float(lr), OPT[optimiser], float(betas[0]), float(betas[1]), float(eps),
                arr, int(rank), int(world), int(seq0), self.workspace.data_ptr(), self.workspace.numel(),
                _stream(self.device)), "affine_optim_peer")
        self.epoch += n_epochs

    # -- sharded (z-slab) form: moments -> [all-reduce by the caller] -> apply
    def moments(self, s_begin: int, s_end: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if out is None:
            out = torch.empty(self.n_pairs, MOMENTS, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.trb_affine_moments_ex(
                self.ndim, self.moving.data_ptr(), self.target.data_ptr(), self.pair_stride, self.n_pairs,
                self.D, self.H, self.W, int(s_begin), int(s_end), self.xb.data_ptr(), self.yb.data_ptr(),
                _ptr(self.zb), self.state.data_ptr(), out.data_ptr(), int(self.flags), self.workspace.data_ptr(),
                self.workspace.numel(), _stream(self.device)), "affine_moments")
        return out

    def apply(self, moments: torch.Tensor, lr: float, w_mse: float, w_ncc: float, optimiser: str = "sgd",
              betas=(0.9, 0.999), eps: float = 1e-8, extra: Optional[torch.Tensor] = None) -> None:
        """extra: optional [n_pairs, 13] float64 — an additional loss term and its d/dtheta per pair."""
        if self.epoch + 1 > self.max_epochs:
            raise ValueError("max_epochs exceeded")
        with torch.cuda.device(self.device):
            check(self.lib.trb_affine_apply(
                self.ndim, MODE[self.mode], moments.data_ptr(), self.n_pairs, self.D, self.H, self.W,
                self.state.data_ptr(), self.loss_log.data_ptr(), self.loss_log.shape[1], self.epoch,
                float(w_mse), float(w_ncc), float(lr), OPT[optimiser], float(betas[0]), float(betas[1]), float(eps),
                _ptr(extra), _stream(self.device)), "affine_apply")
        self.epoch += 1

    # -- results (device tensors; reading them on the host is the only sync)
    def _theta(self, off: int) -> torch.Tensor:
        return self.state[:, off: off + self.nt].reshape(self.n_pairs, self.ndim, self.ndim + 1).clone()

    @property
    def theta(self) -> torch.Tensor:
        """theta the next epoch samples with (== final theta once the loop is over)."""
        return self._theta(S_THETA)

    @property
    def final_theta(self) -> torch.Tensor:
        return self._theta(S_THETA)

    @property
    def best_theta(self) -> torch.Tensor:
        return self._theta(S_BEST_THETA)

    @property
    def params(self) -> torch.Tensor:
        return self.state[:, : self.np].clone()

    @property
    def losses(self) -> torch.Tensor:
        return self.loss_log[:, : self.epoch]


TRB_FLAG_NEAREST = 8


def _mode_flag(mode: str) -> int:
    """Sampling mode of the forward warps -> C-ABI flag: 'bilinear' (the reference's) or 'nearest' (label maps)."""
    if mode == 'bilinear':
        return 0
    if mode == 'nearest':
        return TRB_FLAG_NEAREST
    raise ValueError("mode must be 'bilinear' or 'nearest' (got %r)" % (mode,))


def warp_affine(theta: torch.Tensor, moving: torch.Tensor, out: Optional[torch.Tensor] = None,
                large_rotation: bool = False, *, mode: str = 'bilinear') -> torch.Tensor:
    """out[n, c] = grid_sample(moving[n, c], affine_grid(theta[n])), align_corners=False, zeros padding (reference
    get_affine_warp, warpings.py:18-26).  theta: 12|6 values per pair; moving [N,C,...] with N pairs (N == 1 is the
    reference's case, N > 1 the batch extension: every pair its own theta, ONE launch for all pairs and channels).
    `out`: optional contiguous fp32 destination of moving's shape.  `large_rotation`: theta is known to rotate by more
    than a few degrees (3-D: take the gather kernel instead of the TMA-staged one; same values either way).
    `mode='nearest'`: grid_sample(mode='nearest') for label maps — the source coordinate rounded half to even, so only
    values of `moving` and 0 appear in the output (labels travel as fp32, exact up to 2^24)."""
    flag = _mode_flag(mode)
    require_cuda(moving, "moving")
    ndim, D, H, W = _vol_dims(moving)
    lib = _lib.load()
    dev = moving.device
    n = int(moving.shape[0])
    nt = ndim * (ndim + 1)
    th = torch.as_tensor(theta, dtype=torch.float32, device=dev).detach().reshape(-1).contiguous()
    if th.numel() == nt and n > 1:
        th = th.repeat(n)
    if th.numel() != n * nt:
        raise ValueError("theta has %d values, expected %d per pair (%d pair(s))" % (th.numel(), nt, n))
    src = moving.detach().contiguous()
    if out is None:
        out = torch.empty_like(src)
    elif out.shape != src.shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != dev:
        raise ValueError("out must be a contiguous fp32 tensor of moving's shape on moving's device")
    xb, yb = base_coords(W, dev), base_coords(H, dev)
    zb = base_coords(D, dev) if ndim == 3 else None
    with torch.cuda.device(dev):
        check(lib.trb_warp_affine_batch(ndim, src.data_ptr(), out.data_ptr(), n, int(src.shape[1]), D, H, W, th.data_ptr(),
                                        xb.data_ptr(), yb.data_ptr(), _ptr(zb), (1 if large_rotation else 0) | flag,
                                        _stream(dev)), "warp_affine")
    return out


def warp_affine_vjp(theta: torch.Tensor, moving: torch.Tensor, grad_out: torch.Tensor, large_rotation: bool = False) -> torch.Tensor:
    """d theta (fp64 [ndim, ndim+1]) = sum_v grad_out_v * d warped_v / d theta; single channel."""
    require_cuda(moving, "moving")
    require_cuda(grad_out, "grad_out")
    ndim, D, H, W = _vol_dims(moving)
    if moving.shape[0] != 1 or moving.shape[1] != 1:
        raise ValueError("warp_affine_vjp expects [1,1,...]")
    lib = _lib.load()
    dev = moving.device
    th = torch.as_tensor(theta, dtype=torch.float32, device=dev).detach().reshape(-1).contiguous()
    ws_bytes = int(lib.trb_affine_workspace_bytes(1)) + MOMENTS * 8
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device=dev)
    out = torch.empty(ndim * (ndim + 1), dtype=torch.float64, device=dev)
    xb, yb = base_coords(W, dev), base_coords(H, dev)
    zb = base_coords(D, dev) if ndim == 3 else None
    with torch.cuda.device(dev):
        check(lib.trb_warp_affine_vjp_ex(ndim, moving.contiguous().data_ptr(), grad_out.contiguous().data_ptr(),
                                         D, H, W, th.data_ptr(), xb.data_ptr(), yb.data_ptr(), _ptr(zb),
                                         out.data_ptr(), 1 if large_rotation else 0, ws.data_ptr(), ws.numel(), _stream(dev)),
              "warp_affine_vjp")
    return out.reshape(ndim, ndim + 1)


# --------------------------------------------------------------------------- #
# flow field
# --------------------------------------------------------------------------- #
_FLOW_WS = {}


def _flow_ws(dev):
    key = str(dev)
    ws = _FLOW_WS.get(key)
    if ws is None:
        ws = torch.zeros(int(_lib.load().trb_flow_workspace_bytes()), dtype=torch.uint8, device=dev)
        _FLOW_WS[key] = ws
    return ws


def flow_head_forward(moving, target, feat, weight, bias, w_mse, w_ncc):
    """U-Net head fused with the node (SURVEY.md §8 f-3): flow = out(padNd(feat)) evaluated inside the kernel, then warp +
    similarity.  feat [1,C,(d,)h,w] un-padded decoder output (C <= 8), weight [nd,C,1,(1,)1], bias [nd] the 1x1 `out`
    convolution.  -> (loss [1], flow [1,nd,...]).  Leaves the loss coefficients in the per-device workspace for
    flow_head_backward, which must follow on the same stream."""
    require_cuda(moving, "moving"); require_cuda(target, "target"); require_cuda(feat, "feat")
    ndim, D, H, W = _vol_dims(moving)
    lib = _lib.load()
    dev = moving.device
    C = int(feat.shape[1])
    fdims = [1] * (3 - ndim) + [int(v) for v in feat.shape[2:]]
    f, wt, b = feat.detach().contiguous(), weight.detach().reshape(ndim, C).contiguous(), bias.detach().contiguous()
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    flow = torch.empty((1, ndim) + tuple(moving.shape[2:]), dtype=torch.float32, device=dev)
    ws = _flow_ws(dev)
    with torch.cuda.device(dev):
        check(lib.trb_flow_head_forward(ndim, moving.detach().contiguous().data_ptr(), target.detach().contiguous().data_ptr(),
                                        f.data_ptr(), C, fdims[0], fdims[1], fdims[2], wt.data_ptr(), b.data_ptr(), D, H, W,
                                        float(w_mse), float(w_ncc), loss.data_ptr(), flow.data_ptr(), ws.data_ptr(), ws.numel(),
                                        _stream(dev)), "flow_head_forward")
    return loss, flow


def flow_head_backward(moving, target, flow, feat, weight):
    """-> (d loss / d feat, d loss / d weight [nd,C], d loss / d bias [nd]) for the loss of the preceding flow_head_forward."""
    ndim, D, H, W = _vol_dims(moving)
    lib = _lib.load()
    dev = moving.device
    C = int(feat.shape[1])
    fdims = [1] * (3 - ndim) + [int(v) for v in feat.shape[2:]]
    f, wt = feat.detach().contiguous(), weight.detach().reshape(ndim, C).contiguous()
    dfeat = torch.empty_like(f)
    dwb = torch.empty(ndim * C + ndim, dtype=torch.float32, device=dev)
    ws = _flow_ws(dev)
    with torch.cuda.device(dev):
        check(lib.trb_flow_head_backward(ndim, moving.detach().contiguous().data_ptr(), target.detach().contiguous().data_ptr(),
                                         flow.detach().contiguous().data_ptr(), f.data_ptr(), C, fdims[0], fdims[1], fdims[2],
                                         wt.data_ptr(), D, H, W, dfeat.data_ptr(), dwb.data_ptr(), ws.data_ptr(), ws.numel(),
                                         _stream(dev)), "flow_head_backward")
    return dfeat, dwb[: ndim * C].reshape(ndim, C), dwb[ndim * C:]

def _check_flow(src: torch.Tensor, flow: torch.Tensor):
    require_cuda(src, "src")
    require_cuda(flow, "flow")
    ndim, D, H, W = _vol_dims(src)
    if src.shape[0] != 1 or flow.shape[0] != 1:
        raise ValueError("flow warp expects N == 1")
    if tuple(flow.shape[1:]) != (ndim,) + tuple(src.shape[2:]):
        raise ValueError("flow shape %s does not match src %s" % (tuple(flow.shape), tuple(src.shape)))
    return ndim, D, H, W


def warp_flow(src: torch.Tensor, flow: torch.Tensor, *, mode: str = 'bilinear') -> torch.Tensor:
    """SpatialTransformer.forward (reference utils.py:350-365), all channels of `src`.  `mode='nearest'`:
    grid_sample(mode='nearest', align_corners=True) on the reference's grid, bit for bit (label maps)."""
    flag = _mode_flag(mode)
    ndim, D, H, W = _check_flow(src, flow)
    lib = _lib.load()
    dev = src.device
    s, f = src.detach().contiguous(), flow.detach().contiguous()
    out = torch.empty_like(s)
    with torch.cuda.device(dev):
        check(lib.trb_warp_flow_ex(ndim, s.data_ptr(), f.data_ptr(), out.data_ptr(), int(s.shape[1]), D, H, W, flag,
                                   _stream(dev)), "warp_flow")
    return out


def warp_flow_vjp(src: torch.Tensor, flow: torch.Tensor, grad_out: torch.Tensor) -> torch.Tensor:
    """d flow = J^T grad_out for the single-channel warp."""
    ndim, D, H, W = _check_flow(src, flow)
    if src.shape[1] != 1:
        raise ValueError("warp_flow_vjp expects a single channel")
    require_cuda(grad_out, "grad_out")
    lib = _lib.load()
    dev = src.device
    s, f, g = src.detach().contiguous(), flow.detach().contiguous(), grad_out.detach().contiguous()
    dflow = torch.empty_like(f)
    with torch.cuda.device(dev):
        check(lib.trb_warp_flow_vjp(ndim, s.data_ptr(), f.data_ptr(), g.data_ptr(), dflow.data_ptr(), D, H, W,
                                    _stream(dev)), "warp_flow_vjp")
    return dflow




def flow_loss_grad(moving: torch.Tensor, target: torch.Tensor, flow: torch.Tensor, w_mse: float, w_ncc: float,
                   want_warped: bool = False):
    """-> (loss [1] float32 dev, dflow, warped or None): fused warp + w_mse*MSE + w_ncc*100(1-NCC)
    + gradient w.r.t. the flow (reference utils.py:350-365 + warpings.py:213-215)."""
    ndim, D, H, W = _check_flow(moving, flow)
    require_cuda(target, "target")
    if moving.shape[1] != 1 or target.shape != moving.shape:
        raise ValueError("moving/target must both be [1,1,...] of equal shape")
    lib = _lib.load()
    dev = moving.device
    key = str(dev)
    ws = _FLOW_WS.get(key)
    if ws is None:
        ws = torch.zeros(int(lib.trb_flow_workspace_bytes()), dtype=torch.uint8, device=dev)
        _FLOW_WS[key] = ws
    m, t, f = moving.detach().contiguous(), target.detach().contiguous(), flow.detach().contiguous()
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    dflow = torch.empty_like(f)
    warped = torch.empty_like(m) if want_warped else None
    with torch.cuda.device(dev):
        check(lib.trb_flow_loss_grad(ndim, m.data_ptr(), t.data_ptr(), f.data_ptr(), D, H, W, float(w_mse),
                                     float(w_ncc), loss.data_ptr(), dflow.data_ptr(), _ptr(warped),
                                     ws.data_ptr(), ws.numel(), _stream(dev)), "flow_loss_grad")
    return loss, dflow, warped


# --------------------------------------------------------------------------- #
# EXTENSION: local normalised cross-correlation (csrc/lncc.cu; no reference counterpart)
# --------------------------------------------------------------------------- #
LNCC_MAX_WIN = 15
_LNCC_WS = {}


def check_lncc_window(win: int) -> int:
    if isinstance(win, bool) or int(win) != win or win < 3 or win > LNCC_MAX_WIN or win % 2 == 0:
        raise ValueError("the LNCC window must be an odd integer in [3, %d] (got %r)" % (LNCC_MAX_WIN, win))
    return int(win)


def check_lncc_pair(target: torch.Tensor, warped: torch.Tensor):
    """CUDA fp32 [N,1,(D,)H,W] pairs of one shape -> (ndim, N, D, H, W); raises otherwise (there is no CPU path)."""
    for t, name in ((target, "target"), (warped, "warped")):
        if isinstance(t, torch.Tensor) and t.dtype != torch.float32:
            raise TypeError("%s must be float32 (got %s)" % (name, t.dtype))
    require_cuda(target, "target")
    require_cuda(warped, "warped")
    ndim, D, H, W = _vol_dims(warped)
    if warped.shape[1] != 1 or target.shape != warped.shape:
        raise ValueError("LNCC expects target and warped of one [N,1,...] shape (got %s and %s)"
                         % (tuple(target.shape), tuple(warped.shape)))
    return ndim, int(warped.shape[0]), D, H, W


def _lncc_ws(dev):
    ws = _LNCC_WS.get(str(dev))
    if ws is None:
        ws = torch.zeros(int(_lib.load().trb_lncc_workspace_bytes()), dtype=torch.uint8, device=dev)
        _LNCC_WS[str(dev)] = ws
    return ws


def lncc_forward(target: torch.Tensor, warped: torch.Tensor, win: int = 9, eps: float = 1e-5):
    """-> (stats [2] fp64 device tensor (sum of cc, loss), coef [3, N*D*H*W] = alpha, beta, gamma) for
    loss = 1 - mean(cc) of the windowed NCC (include/trb.h: trb_lncc_forward)."""
    win = check_lncc_window(win)
    ndim, n, D, H, W = check_lncc_pair(target, warped)
    dev = warped.device
    t, w = target.detach().contiguous(), warped.detach().contiguous()
    coef = torch.empty(3, t.numel(), dtype=torch.float32, device=dev)
    stats = torch.empty(2, dtype=torch.float64, device=dev)
    ws = _lncc_ws(dev)
    with torch.cuda.device(dev):
        check(_lib.load().trb_lncc_forward(ndim, t.data_ptr(), w.data_ptr(), n, D, H, W, win, float(eps), coef.data_ptr(),
                                           stats.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)), "lncc_forward")
    return stats, coef


def lncc_backward(target: torch.Tensor, warped: torch.Tensor, coef: torch.Tensor, win: int = 9, scale: float = 1.0) -> torch.Tensor:
    """scale * d loss / d warped for the coef of lncc_forward on the same pair and window."""
    win = check_lncc_window(win)
    ndim, n, D, H, W = check_lncc_pair(target, warped)
    dev = warped.device
    t, w = target.detach().contiguous(), warped.detach().contiguous()
    grad = torch.empty_like(w)
    with torch.cuda.device(dev):
        check(_lib.load().trb_lncc_backward(ndim, t.data_ptr(), w.data_ptr(), coef.data_ptr(), n, D, H, W, win, float(scale),
                                            None, 0.0, 0.0, grad.data_ptr(), _stream(dev)), "lncc_backward")
    return grad


def lncc_loss_grad(warped: torch.Tensor, target: torch.Tensor, win: int = 9, eps: float = 1e-5):
    """-> (loss, d loss / d warped): loss = 1 - mean(cc) of the windowed NCC of (target, warped) as a 0-dim fp32 device
    tensor, and its gradient (two kernels, no host synchronisation)."""
    stats, coef = lncc_forward(target, warped, win, eps)
    return stats[1].float(), lncc_backward(target, warped, coef, win)


# --------------------------------------------------------------------------- #
# EXTENSION: direct per-voxel flow optimisation (no reference counterpart)
# --------------------------------------------------------------------------- #
class NmiTerm:
    """NMI/KDE term of the reference's default loss for ONE pair, on CUDA kernels (trb_nmi_prepare once per target,
    trb_nmi_loss_grad per call).  Reference: NMILoss.forward utils.py:224-259 + NMI/get_pdf utils.py:18-79 with the
    module's default bins=256, patch_size=100."""

    def __init__(self, target: torch.Tensor, bandwidth: float = 3.0, alpha: float = 1000.0):
        require_cuda(target, "target")
        self.lib = _lib.load()
        self.ndim, self.D, self.H, self.W = _vol_dims(target)
        if target.shape[0] != 1 or target.shape[1] != 1:
            raise ValueError("NmiTerm expects a [1,1,...] target")
        self.device = target.device
        self.bandwidth, self.alpha = float(bandwidth), float(alpha)
        n = int(self.lib.trb_nmi_workspace_bytes(self.ndim, self.D, self.H, self.W))
        self.workspace = torch.empty(n, dtype=torch.uint8, device=self.device)
        self.loss = torch.zeros(1, dtype=torch.float64, device=self.device)
        t = target.detach().contiguous().float()
        with torch.cuda.device(self.device):
            check(self.lib.trb_nmi_prepare(self.ndim, t.data_ptr(), self.D, self.H, self.W, self.bandwidth,
                                           self.workspace.data_ptr(), self.workspace.numel(), _stream(self.device)), "nmi_prepare")

    def loss_grad(self, warped: torch.Tensor, weight: float = 1.0, want_grad: bool = True):
        """-> (weight*loss as a [1] fp64 device tensor (overwritten by the next call), weight * d loss / d warped or None)."""
        require_cuda(warped, "warped")
        if tuple(warped.shape[2:]) != ((self.D, self.H, self.W) if self.ndim == 3 else (self.H, self.W)) or warped.shape[0] != 1 or warped.shape[1] != 1:
            raise ValueError("warped must have the target's [1,1,...] shape")
        w = warped.detach().contiguous().float()
        gout = torch.empty_like(w) if want_grad else None
        with torch.cuda.device(self.device):
            check(self.lib.trb_nmi_loss_grad(self.ndim, w.data_ptr(), self.D, self.H, self.W, self.bandwidth, self.alpha,
                                             float(weight), self.loss.data_ptr(), _ptr(gout), self.workspace.data_ptr(),
                                             self.workspace.numel(), _stream(self.device)), "nmi_loss_grad")
        return self.loss, gout


class NmiSourceTerm:
    """The same term for a BATCH of 2-D or 3-D pairs, evaluated in source-voxel space (csrc/nmi_src.cu): no resampled arrays, one
    pass over the warped volumes + one pass writing the gradient.  Needs all values of the targets and of every warped
    volume inside [lo, hi] with hi - lo <= 0.6 * bandwidth (`bounds()` derives them; images normalised to [0,1] qualify
    with the default bandwidth 3); the loss is NaN if a value leaves the bounds."""

    MAX_RANGE = 0.6          # in bandwidths (Hermite-moment regime of the KDE)

    @staticmethod
    def bounds(moving: torch.Tensor, target: torch.Tensor):
        """Value bounds that hold for the targets and for ANY warp of the moving volumes (a trilinear sample with zero
        padding is a convex combination of voxel values and 0).  One host synchronisation."""
        v = torch.stack([moving.amin(), target.amin(), moving.amax(), target.amax()]).tolist()
        return min(0.0, v[0], v[1]), max(0.0, v[2], v[3])

    @classmethod
    def eligible(cls, moving: torch.Tensor, lo: float, hi: float, bandwidth: float = 3.0) -> bool:
        return moving.dim() in (4, 5) and moving.shape[1] == 1 and (hi - lo) <= cls.MAX_RANGE * bandwidth and lo <= hi

    def __init__(self, target: torch.Tensor, lo: float, hi: float, bandwidth: float = 3.0, alpha: float = 1000.0):
        require_cuda(target, "target")
        self.lib = _lib.load()
        if target.dim() not in (4, 5) or target.shape[1] != 1:
            raise ValueError("NmiSourceTerm expects [N,1,(D,)H,W] targets")
        self.device = target.device
        self.ndim, self.D, self.H, self.W = _vol_dims(target)
        self.n_pairs = int(target.shape[0])
        self.shape = tuple(target.shape)
        self.vol = self.D * self.H * self.W
        self.bandwidth, self.alpha, self.lo, self.hi = float(bandwidth), float(alpha), float(lo), float(hi)
        n = int(self.lib.trb_nmi_src_workspace_bytes(self.ndim, self.n_pairs, self.D, self.H, self.W))
        self.workspace = torch.empty(n, dtype=torch.uint8, device=self.device)
        self.loss = torch.zeros(self.n_pairs, dtype=torch.float64, device=self.device)
        t = target.detach().contiguous().float()
        with torch.cuda.device(self.device):
            check(self.lib.trb_nmi_src_prepare(self.ndim, t.data_ptr(), self.vol, self.n_pairs, self.D, self.H, self.W,
                                               self.bandwidth, self.lo, self.hi, self.workspace.data_ptr(),
                                               self.workspace.numel(), _stream(self.device)), "nmi_src_prepare")

    def loss_grad(self, warped: torch.Tensor, weight: float = 1.0, want_grad: bool = True):
        """-> (weight*loss per pair, [N] fp64 device tensor overwritten by the next call; weight * d loss / d warped or None)."""
        require_cuda(warped, "warped")
        if tuple(warped.shape) != self.shape:
            raise ValueError("warped must have the targets' shape %s" % (self.shape,))
        w = warped.detach().contiguous().float()
        gout = torch.empty_like(w) if want_grad else None
        with torch.cuda.device(self.device):
            check(self.lib.trb_nmi_src_loss_grad(self.ndim, w.data_ptr(), self.vol, self.n_pairs, self.D, self.H, self.W,
                                                 self.bandwidth, self.alpha, float(weight), self.lo, self.hi,
                                                 self.loss.data_ptr(), 1, _ptr(gout), self.workspace.data_ptr(),
                                                 self.workspace.numel(), _stream(self.device)), "nmi_src_loss_grad")
        return self.loss, gout


# --------------------------------------------------------------------------- #
# InstanceNorm of the flow U-Net
# --------------------------------------------------------------------------- #
_IN_WS = {}


def _instnorm_ws(device, n_inst: int, S: int) -> torch.Tensor:
    need = int(_lib.load().trb_instnorm_workspace_bytes(n_inst, S))
    ws = _IN_WS.get(str(device))
    if ws is None or ws.numel() < need:
        ws = torch.empty(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _IN_WS[str(device)] = ws
    return ws


def instance_norm_forward(x: torch.Tensor, eps: float = 1e-5, relu: bool = False, gate: Optional[torch.Tensor] = None):
    """y = InstanceNorm(relu?(x)) for x [N,C,*spatial] (affine=False, no running statistics) -> (y, stats [N*C,2]).
    gate ([1,1,*spatial], N == 1, no ReLU): y = InstanceNorm(x * gate) without the product tensor."""
    require_cuda(x, "x")
    x = x.contiguous()
    n_inst = int(x.shape[0] * x.shape[1])
    S = x.numel() // n_inst
    if gate is not None:
        gate = gate.contiguous()
        if x.shape[0] != 1 or gate.numel() != S or relu:
            raise ValueError("gated instance norm: one sample, gate [1,1,*spatial], no ReLU")
    y = torch.empty_like(x)
    stats = torch.empty(n_inst, 2, dtype=torch.float32, device=x.device)
    ws = _instnorm_ws(x.device, n_inst, S)
    with torch.cuda.device(x.device):
        check(_lib.load().trb_instnorm_forward(x.data_ptr(), _ptr(gate), y.data_ptr(), n_inst, S, float(eps), int(bool(relu)),
                                               stats.data_ptr(), ws.data_ptr(), ws.numel(), _stream(x.device)), "instnorm_forward")
    return y, stats


def instance_norm_backward(x: torch.Tensor, dy: torch.Tensor, stats: torch.Tensor, relu: bool = False,
                           gate: Optional[torch.Tensor] = None):
    """-> d/dx, or (d/dx, d/dgate) with a gate."""
    require_cuda(dy, "dy")
    x, dy = x.contiguous(), dy.contiguous()
    n_inst = int(x.shape[0] * x.shape[1])
    S = x.numel() // n_inst
    dx = torch.empty_like(x)
    dgate = torch.empty_like(gate) if gate is not None else None
    coef = torch.empty(n_inst, 2, dtype=torch.float32, device=x.device)
    ws = _instnorm_ws(x.device, n_inst, S)
    with torch.cuda.device(x.device):
        check(_lib.load().trb_instnorm_backward(x.data_ptr(), _ptr(gate), dy.data_ptr(), dx.data_ptr(), _ptr(dgate), n_inst, S,
                                                int(bool(relu)), stats.data_ptr(), coef.data_ptr(), ws.data_ptr(), ws.numel(),
                                                _stream(x.device)), "instnorm_backward")
    return dx if gate is None else (dx, dgate)


# --------------------------------------------------------------------------- #
# thin 3x3x3 convolutions of the flow U-Net
# --------------------------------------------------------------------------- #
THIN_CONV_MAX_CHANNELS = 4
# the pair volume of the gather variant costs 2x the moving volumes in memory (measured gain: one 192x192x160 pair 55 -> 36 us,
# 256^3 144 -> 117, a batch of 8 389 -> 287); beyond this size the scalar gathers are used
PAIR_VOLUME_MAX_BYTES = 16 << 30
# Measured (same box, us/epoch, scalar / pair / quad): one 192x192x160 pair 56.6 / 37.0 / 41.8; 256^3 143 / 146 / 115; 8 pairs
# 388 / 358 / 286.  While the pair volume sits in L2 the four 8-byte gathers win; once it streams from HBM the quad volume
# (x and y neighbours in one 16-byte record, 2 gathers per voxel, 4x the memory) touches half as many sectors per voxel
PAIR_VOLUME_L2_BYTES = 64 << 20


def thin_conv3d_forward(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """conv3d(x, weight, bias) for kernel 3, stride 1, no padding, <= 4 channels each way (csrc/thinconv.cu)."""
    require_cuda(x, "x")
    x, weight = x.contiguous(), weight.contiguous()
    n, ci, D, H, W = (int(v) for v in x.shape)
    co = int(weight.shape[0])
    y = torch.empty(n, co, D - 2, H - 2, W - 2, dtype=torch.float32, device=x.device)
    b = bias.contiguous() if bias is not None else None
    with torch.cuda.device(x.device):
        check(_lib.load().trb_thinconv3_forward(x.data_ptr(), weight.data_ptr(), _ptr(b), y.data_ptr(), n, ci, co, D, H, W,
                                                _stream(x.device)), "thinconv3_forward")
    return y


def thin_conv3d_backward(x: torch.Tensor, weight: torch.Tensor, gy: torch.Tensor, need_gx: bool, need_gw: bool, need_gb: bool):
    """-> (d/dx or None, d/dweight or None, d/dbias or None)."""
    require_cuda(gy, "gy")
    x, weight, gy = x.contiguous(), weight.contiguous(), gy.contiguous()
    n, ci, D, H, W = (int(v) for v in x.shape)
    co = int(weight.shape[0])
    lib = _lib.load()
    gx = torch.empty_like(x) if need_gx else None
    want_w = need_gw or need_gb
    gw = torch.empty_like(weight) if want_w else None
    gb = torch.empty(co, dtype=torch.float32, device=x.device) if want_w else None
    ws = torch.empty(max(int(lib.trb_thinconv3_workspace_bytes(ci, co)), 8), dtype=torch.uint8, device=x.device) if want_w else None
    with torch.cuda.device(x.device):
        if n == 1 or not want_w:
            check(lib.trb_thinconv3_backward(x.data_ptr(), weight.data_ptr(), gy.data_ptr(), _ptr(gx), _ptr(gw), _ptr(gb), n, ci, co,
                                             D, H, W, _ptr(ws), ws.numel() if ws is not None else 0, _stream(x.device)), "thinconv3_backward")
        else:
            check(lib.trb_thinconv3_backward(x.data_ptr(), weight.data_ptr(), gy.data_ptr(), _ptr(gx), None, None, n, ci, co,
                                             D, H, W, None, 0, _stream(x.device)), "thinconv3_backward")
            gw.zero_(); gb.zero_()
            for i in range(n):            # the weight gradient handles one sample per call
                gwi, gbi = torch.empty_like(gw), torch.empty_like(gb)
                check(lib.trb_thinconv3_backward(x[i].data_ptr(), weight.data_ptr(), gy[i].data_ptr(), None, gwi.data_ptr(), gbi.data_ptr(),
                                                 1, ci, co, D, H, W, ws.data_ptr(), ws.numel(), _stream(x.device)), "thinconv3_backward")
                gw += gwi; gb += gbi
    return gx, (gw if need_gw else None), (gb if need_gb else None)


def point_conv3d_forward(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], stride: int) -> torch.Tensor:
    """conv3d(x, weight, bias, stride) for a 1x1x1 kernel, no padding, <= 4 channels each way, x [1,CI,D,H,W]."""
    require_cuda(x, "x")
    x, weight = x.contiguous(), weight.contiguous()
    _, ci, D, H, W = (int(v) for v in x.shape)
    co = int(weight.shape[0])
    od, oh, ow = (D - 1) // stride + 1, (H - 1) // stride + 1, (W - 1) // stride + 1
    y = torch.empty(1, co, od, oh, ow, dtype=torch.float32, device=x.device)
    b = bias.contiguous() if bias is not None else None
    with torch.cuda.device(x.device):
        check(_lib.load().trb_pointconv_forward(x.data_ptr(), weight.data_ptr(), _ptr(b), y.data_ptr(), ci, co, D, H, W, int(stride),
                                                _stream(x.device)), "pointconv_forward")
    return y


def point_conv3d_backward(x: torch.Tensor, weight: torch.Tensor, gy: torch.Tensor, stride: int, need_gx: bool, need_gw: bool,
                          need_gb: bool):
    require_cuda(gy, "gy")
    x, weight, gy = x.contiguous(), weight.contiguous(), gy.contiguous()
    _, ci, D, H, W = (int(v) for v in x.shape)
    co = int(weight.shape[0])
    lib = _lib.load()
    want_w = need_gw or need_gb
    gx = torch.empty_like(x) if need_gx else None
    gw = torch.empty_like(weight) if want_w else None
    gb = torch.empty(co, dtype=torch.float32, device=x.device) if want_w else None
    ws = torch.empty(max(int(lib.trb_pointconv_workspace_bytes(ci, co)), 8), dtype=torch.uint8, device=x.device) if want_w else None
    with torch.cuda.device(x.device):
        check(lib.trb_pointconv_backward(x.data_ptr(), weight.data_ptr(), gy.data_ptr(), _ptr(gx), _ptr(gw), _ptr(gb), ci, co, D, H, W,
                                         int(stride), _ptr(ws), ws.numel() if ws is not None else 0, _stream(x.device)), "pointconv_backward")
    return gx, (gw if need_gw else None), (gb if need_gb else None)


def up_conv3d_forward(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """conv_transpose3d(x, weight, bias, stride=2) for a 2x2x2 kernel, <= 4 channels each way, x [1,CI,D,H,W]."""
    require_cuda(x, "x")
    x, weight = x.contiguous(), weight.contiguous()
    _, ci, D, H, W = (int(v) for v in x.shape)
    co = int(weight.shape[1])
    y = torch.empty(1, co, 2 * D, 2 * H, 2 * W, dtype=torch.float32, device=x.device)
    b = bias.contiguous() if bias is not None else None
    with torch.cuda.device(x.device):
        check(_lib.load().trb_upconv2_forward(x.data_ptr(), weight.data_ptr(), _ptr(b), y.data_ptr(), ci, co, D, H, W,
                                              _stream(x.device)), "upconv2_forward")
    return y


def up_conv3d_backward(x: torch.Tensor, weight: torch.Tensor, gy: torch.Tensor, need_gx: bool, need_gw: bool, need_gb: bool):
    require_cuda(gy, "gy")
    x, weight, gy = x.contiguous(), weight.contiguous(), gy.contiguous()
    _, ci, D, H, W = (int(v) for v in x.shape)
    co = int(weight.shape[1])
    lib = _lib.load()
    want_w = need_gw or need_gb
    gx = torch.empty_like(x) if need_gx else None
    gw = torch.empty_like(weight) if want_w else None
    gb = torch.empty(co, dtype=torch.float32, device=x.device) if want_w else None
    ws = torch.empty(max(int(lib.trb_upconv2_workspace_bytes(ci, co)), 8), dtype=torch.uint8, device=x.device) if want_w else None
    with torch.cuda.device(x.device):
        check(lib.trb_upconv2_backward(x.data_ptr(), weight.data_ptr(), gy.data_ptr(), _ptr(gx), _ptr(gw), _ptr(gb), ci, co, D, H, W,
                                       _ptr(ws), ws.numel() if ws is not None else 0, _stream(x.device)), "upconv2_backward")
    return gx, (gw if need_gw else None), (gb if need_gb else None)


class DirectFlowProblem:
    """Per-voxel flow field optimised with SGD or Adam on
    loss = w_mse*MSE + w_ncc*100*(1-NCC) + smooth * mean_axes(mean(forward_diff(flow)^2)).

    Holds a z-slab [z_off, z_off+Ds) of the target/flow (the whole volume by default); `moving` is always the
    full volume.  One epoch = stats pass -> (all-reduce hook) -> update pass, ping-ponging two flow buffers.
    """

    def __init__(self, moving, target_slab, max_epochs, z_off=0, flow0=None, optimiser="sgd", flow_buffers=None):
        require_cuda(moving, "moving")
        require_cuda(target_slab, "target")
        self.lib = _lib.load()
        self.device = moving.device
        self.ndim, self.D, self.H, self.W = _vol_dims(moving)
        if moving.shape[0] != 1 or moving.shape[1] != 1:
            raise ValueError("direct flow expects [1,1,...] volumes")
        self.moving = moving.contiguous()
        self.target = target_slab.contiguous()
        self.Ds = int(target_slab.shape[2]) if self.ndim == 3 else 1
        self.z_off = int(z_off) if self.ndim == 3 else 0
        if tuple(target_slab.shape[-2:]) != (self.H, self.W):
            raise ValueError("target slab must share H, W with moving")
        shape = (1, self.ndim) + tuple(self.target.shape[2:])
        if flow_buffers is not None:
            # caller-owned ping-pong buffers (parallel.ShardedDirectFlow puts them in symmetric memory so the neighbour
            # ranks can read the boundary slices in place)
            self.flow, self._other = (b.view(shape) for b in flow_buffers)
            if flow0 is None:
                self.flow.zero_()
            else:
                self.flow.copy_(flow0.detach().to(self.device, torch.float32))
        else:
            self.flow = (torch.zeros(shape, dtype=torch.float32, device=self.device) if flow0 is None
                         else flow0.detach().to(self.device, torch.float32).contiguous().clone())
            if tuple(self.flow.shape) != shape:
                raise ValueError("flow0 must have shape %s" % (shape,))
            self._other = torch.empty_like(self.flow)
        self.optimiser = optimiser
        self.adam_m = torch.zeros_like(self.flow) if optimiser == "adam" else None
        self.adam_v = torch.zeros_like(self.flow) if optimiser == "adam" else None
        self.moments = torch.zeros(6, dtype=torch.float64, device=self.device)
        self.loss_log = torch.zeros(max(int(max_epochs), 1), dtype=torch.float32, device=self.device)
        self.workspace = torch.zeros(int(self.lib.trb_flow_direct_workspace_bytes()), dtype=torch.uint8, device=self.device)
        self.max_epochs = int(max_epochs)
        self.epoch = 0
        self._pending = False          # a fused step whose loss entry is not complete yet (see `finish`)
        self._sums_epoch = -1          # epoch whose (all-reduced) similarity sums `moments` holds

    def boundary_slices(self):
        """(first, last) z-slices of the current flow, [ndim, H, W] each — what the neighbours need as halos."""
        return self.flow[0, :, 0].contiguous(), self.flow[0, :, -1].contiguous()

    def stats(self, smooth, halo_lo=None, halo_hi=None):
        with torch.cuda.device(self.device):
            check(self.lib.trb_flow_direct_stats(
                self.ndim, self.moving.data_ptr(), self.target.data_ptr(), self.flow.data_ptr(), _ptr(halo_lo), _ptr(halo_hi),
                self.D, self.H, self.W, self.z_off, self.Ds, float(smooth), self.moments.data_ptr(),
                self.workspace.data_ptr(), self.workspace.numel(), _stream(self.device)), "flow_direct_stats")
        return self.moments

    def update(self, lr, w_mse, w_ncc, smooth, halo_lo=None, halo_hi=None, betas=(0.9, 0.999), eps=1e-8):
        if self.epoch >= self.max_epochs:
            raise ValueError("max_epochs exceeded")
        with torch.cuda.device(self.device):
            check(self.lib.trb_flow_direct_update(
                self.ndim, self.moving.data_ptr(), self.target.data_ptr(), self.flow.data_ptr(), self._other.data_ptr(),
                _ptr(halo_lo), _ptr(halo_hi), self.D, self.H, self.W, self.z_off, self.Ds, self.moments.data_ptr(),
                float(w_mse), float(w_ncc), float(smooth), float(lr), OPT[self.optimiser], float(betas[0]), float(betas[1]),
                float(eps), self.epoch + 1, _ptr(self.adam_m), _ptr(self.adam_v), self.loss_log.data_ptr(), self.epoch,
                _stream(self.device)), "flow_direct_update")
        self.flow, self._other = self._other, self.flow
        self.epoch += 1

    @property
    def fused(self):
        """3-D volumes below 2^31/3 voxels take the one-pass-per-epoch kernel (trb_flow_direct_step)."""
        return self.ndim == 3 and 3 * self.Ds * self.H * self.W < 2 ** 31 and self.D * self.H * self.W < 2 ** 31

    def step(self, lr, w_mse, w_ncc, smooth, halo_lo=None, halo_hi=None, betas=(0.9, 0.999), eps=1e-8):
        """One fused epoch.  `self.moments` must hold the (all-reduced) similarity sums of the current flow when
        w_ncc != 0 (see `prime`); on return it holds this slab's sums for the next call."""
        if self.epoch >= self.max_epochs:
            raise ValueError("max_epochs exceeded")
        with torch.cuda.device(self.device):
            check(self.lib.trb_flow_direct_step(
                self.moving.data_ptr(), self.target.data_ptr(), self.flow.data_ptr(), self._other.data_ptr(),
                _ptr(halo_lo), _ptr(halo_hi), self.D, self.H, self.W, self.z_off, self.Ds, self.moments.data_ptr(),
                float(w_mse), float(w_ncc), float(smooth), float(lr), OPT[self.optimiser], float(betas[0]), float(betas[1]),
                float(eps), self.epoch + 1, _ptr(self.adam_m), _ptr(self.adam_v), self.loss_log.data_ptr(), self.epoch,
                int(self._pending), self.workspace.data_ptr(), self.workspace.numel(), _stream(self.device)), "flow_direct_step")
        self.flow, self._other = self._other, self.flow
        self.epoch += 1
        self._pending = True

    def step_peer(self, lr, w_mse, w_ncc, smooth, halo_lo_ptr, halo_lo_cs, halo_hi_ptr, halo_hi_cs, mailbox_ptrs, rank, world, seq,
                  betas=(0.9, 0.999), eps=1e-8):
        """One fused epoch of a z-slab with the neighbours' boundary slices read in place (raw device pointers into their
        flow buffers) and the 6 sums all-reduced inside the kernel (include/trb.h: trb_flow_direct_step_peer)."""
        if self.epoch >= self.max_epochs:
            raise ValueError("max_epochs exceeded")
        import ctypes
        arr = (ctypes.c_void_p * world)(*[int(v) for v in mailbox_ptrs])
        with torch.cuda.device(self.device):
            check(self.lib.trb_flow_direct_step_peer(
                self.moving.data_ptr(), self.target.data_ptr(), self.flow.data_ptr(), self._other.data_ptr(),
                halo_lo_ptr, int(halo_lo_cs), halo_hi_ptr, int(halo_hi_cs), self.D, self.H, self.W, self.z_off, self.Ds,
                self.moments.data_ptr(), float(w_mse), float(w_ncc), float(smooth), float(lr), OPT[self.optimiser],
                float(betas[0]), float(betas[1]), float(eps), self.epoch + 1, _ptr(self.adam_m), _ptr(self.adam_v),
                self.loss_log.data_ptr(), self.epoch, int(self._pending), arr, int(rank), int(world), int(seq),
                self.workspace.data_ptr(), self.workspace.numel(), _stream(self.device)), "flow_direct_step_peer")
        self.flow, self._other = self._other, self.flow
        self.epoch += 1
        self._pending = True

    def prime(self, w_ncc):
        """Similarity sums of the current flow (this slab) into `self.moments` — what the first fused epoch of an
        NCC-weighted run reads.  Returns True if the caller has to all-reduce them."""
        self._pending = False
        if w_ncc == 0 or self._sums_epoch == self.epoch:
            return False
        self.stats(0.0)
        return True

    def finish(self, w_mse, w_ncc, smooth):
        """Complete the loss log of the last fused epoch from the (all-reduced) moments."""
        with torch.cuda.device(self.device):
            check(self.lib.trb_flow_direct_finish(
                self.moments.data_ptr(), self.D, self.H, self.W, float(w_mse), float(w_ncc), float(smooth),
                self.loss_log.data_ptr(), self.epoch, self.workspace.data_ptr(), self.workspace.numel(),
                _stream(self.device)), "flow_direct_finish")
        self._pending = False
        self._sums_epoch = self.epoch if w_ncc != 0 else -1      # moments[0..4] describe the current flow

    def run(self, n_epochs, lr, w_mse, w_ncc, smooth=0.0, betas=(0.9, 0.999), eps=1e-8, *, w_lncc=0.0, lncc_win=9,
            lncc_eps=1e-5):
        """Single-GPU epochs (whole volume in this problem): no host synchronisation.  w_lncc != 0 adds the local NCC
        term (window lncc_win) and runs `run_lncc`'s epochs."""
        if w_lncc != 0:
            self.run_lncc(n_epochs, lr, w_mse, w_ncc, w_lncc, lncc_win, lncc_eps, smooth, betas, eps)
            return
        if self.fused and n_epochs > 0:
            self.prime(w_ncc)
            for _ in range(n_epochs):
                self.step(lr, w_mse, w_ncc, smooth, betas=betas, eps=eps)
            self.finish(w_mse, w_ncc, smooth)
            return
        for _ in range(n_epochs):
            self.stats(smooth)
            self.update(lr, w_mse, w_ncc, smooth, betas=betas, eps=eps)

    def run_lncc(self, n_epochs, lr, w_mse, w_ncc, w_lncc, win=9, lncc_eps=1e-5, smooth=0.0, betas=(0.9, 0.999), eps=1e-8):
        """Epochs of loss = w_lncc * (1 - mean cc) + w_mse*MSE + w_ncc*100*(1-NCC) + smooth * R(flow), whole volume on one
        GPU, no host synchronisation.  Per epoch: the stats pass (MSE / NCC moments and the smoothness sum; skipped when
        all three weights are 0), the flow warp J, trb_lncc_forward, trb_lncc_backward (dL/dJ, with the pointwise MSE /
        NCC terms) and trb_flow_direct_update_lncc.  loss_log[e] is the loss of flow_e, before its step."""
        win = check_lncc_window(win)
        if self.ndim == 3 and (self.z_off != 0 or self.Ds != self.D):
            raise ValueError("the LNCC epoch runs on the whole volume (no z-slab)")
        if self.epoch + n_epochs > self.max_epochs:
            raise ValueError("max_epochs exceeded")
        if getattr(self, "_lncc", None) is None:
            # J, alpha / beta / gamma and dL/dJ: 5 volumes (335 MB at 256^3), kept for the problem's lifetime
            self._lncc = (torch.empty_like(self.target), torch.empty(3, self.target.numel(), dtype=torch.float32, device=self.device),
                          torch.empty_like(self.target), torch.zeros(2, dtype=torch.float64, device=self.device),
                          torch.zeros(int(self.lib.trb_lncc_workspace_bytes()), dtype=torch.uint8, device=self.device))
        warped, coef, resid, lstats, lws = self._lncc
        need_stats = w_mse != 0 or w_ncc != 0 or smooth != 0
        if not need_stats:
            self.moments.zero_()
        lib, s = self.lib, _stream(self.device)
        with torch.cuda.device(self.device):
            for _ in range(n_epochs):
                if need_stats:
                    self.stats(smooth)
                check(lib.trb_warp_flow(self.ndim, self.moving.data_ptr(), self.flow.data_ptr(), warped.data_ptr(), 1,
                                        self.D, self.H, self.W, s), "warp_flow")
                check(lib.trb_lncc_forward(self.ndim, self.target.data_ptr(), warped.data_ptr(), 1, self.D, self.H, self.W,
                                           win, float(lncc_eps), coef.data_ptr(), lstats.data_ptr(), lws.data_ptr(),
                                           lws.numel(), s), "lncc_forward")
                check(lib.trb_lncc_backward(self.ndim, self.target.data_ptr(), warped.data_ptr(), coef.data_ptr(), 1,
                                            self.D, self.H, self.W, win, float(w_lncc),
                                            self.moments.data_ptr() if (w_mse != 0 or w_ncc != 0) else None,
                                            float(w_mse), float(w_ncc), resid.data_ptr(), s), "lncc_backward")
                check(lib.trb_flow_direct_update_lncc(
                    self.ndim, self.moving.data_ptr(), self.flow.data_ptr(), self._other.data_ptr(), resid.data_ptr(),
                    self.D, self.H, self.W, self.moments.data_ptr(), lstats.data_ptr(), float(w_mse), float(w_ncc),
                    float(w_lncc), float(smooth), float(lr), OPT[self.optimiser], float(betas[0]), float(betas[1]),
                    float(eps), self.epoch + 1, _ptr(self.adam_m), _ptr(self.adam_v), self.loss_log.data_ptr(), self.epoch,
                    s), "flow_direct_update_lncc")
                self.flow, self._other = self._other, self.flow
                self.epoch += 1
        self._pending = False
        self._sums_epoch = -1          # moments describe the flow before the last step

    def run_two_pass(self, n_epochs, lr, w_mse, w_ncc, smooth=0.0, betas=(0.9, 0.999), eps=1e-8):
        """The stats + update form of `run` (2-D, very large slabs, and the cross-check of the fused kernel)."""
        for _ in range(n_epochs):
            self.stats(smooth)
            self.update(lr, w_mse, w_ncc, smooth, betas=betas, eps=eps)

    @property
    def losses(self):
        return self.loss_log[: self.epoch]
