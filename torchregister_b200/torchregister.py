"""`Register` — drop-in for the reference's user API (TR/torchregister.py:11-129).

Same constructor, `optim`, `__call__` and attributes; the work is done by the fused
sm_100a kernels behind warpings.py.  CUDA only.
"""
from __future__ import annotations

from torch import cat

from .warpings import flow_register, direct_flow_register, affine_register, rigid_register, get_affine_warp


class Register():
    def __init__(self, mode='rigid', device='cpu', criterion=None, weight=None, grad_edges=False, debug=False, *,
                 flow_param='unet', smooth=0.0, optm='SGD'):
        '''
        B200 registration with the reference's interface (torchregister.py:12-44).

        Parameters
        ----------
        mode : 'rigid' | 'affine' | 'flow'. The default is 'rigid'.
        device : device the optimisation runs on. The default 'cpu' is accepted for signature
            compatibility, but this implementation has no CPU path: `optim` raises unless the
            device is a CUDA device.
        criterion, weight : as in the reference — (criterion and weight) are passed through,
            weight alone re-weights the default [MSE, NCC, NMI] terms. NOTE the reference ignores a
            user criterion in rigid/affine mode and uses MSE (warpings.py:38-40,125-127); so do we.
        grad_edges, debug : as in the reference.
        flow_param, smooth, optm : keyword-only EXTENSIONS with reference-preserving defaults. flow_param='direct'
            optimises the dense flow itself with a smoothness weight `smooth` instead of the reference's U-Net
            parametrisation ('unet'). optm='ADAM' (default 'SGD', the reference's optimiser) selects torch.optim.Adam
            semantics, fused into the epoch kernel: on theta for rigid/affine, on the flow for flow_param='direct'.
        '''
        self.criterion = criterion
        self.weight = weight
        self.mode = mode
        self.warp = None if mode == 'flow' else get_affine_warp
        self.device = device
        self.debug = debug
        self.theta = None
        self.grad_edges = grad_edges
        self.losses = None
        self.flow_param, self.smooth, self.optm = flow_param, smooth, optm

    def _check_device(self):
        import torch
        if torch.device(self.device).type != 'cuda':
            raise RuntimeError(
                "torchregister_b200.Register runs on CUDA only (got device=%r); there is no CPU fallback. "
                "Use Register(device='cuda')." % (self.device,))

    def optim(self, moving, target, lr=1E-5, max_epochs=1000, n=32, per=0.1, *, reg0=None, theta0=None):
        '''
        Optimisation loop (reference torchregister.py:46-106). Sets `self.theta` to the best
        (lowest-loss, pre-step) theta for rigid/affine, or to the last flow field for flow.
        `reg0` (keyword-only extension): initial rigid parameters instead of the torch.rand draw.
        `theta0` (keyword-only extension, affine mode): start theta instead of identity — e.g. the theta of a preceding
        rigid stage together with the ORIGINAL moving volume, so that the pipeline needs no intermediate resampling.
        '''
        self._check_device()
        # the reference works in float32 throughout (dtype=torch.float, warpings.py:48,55; utils.py:347)
        moving = moving.to(device=self.device, dtype=__import__('torch').float32)
        target = target.to(device=self.device, dtype=__import__('torch').float32)
        if self.mode == 'flow' and moving.shape[0] != 1:
            raise ValueError("flow mode registers one pair per call (moving must be [1,1,...])")
        both = self.criterion is not None and self.weight is not None
        if self.mode == 'flow' and self.flow_param == 'direct':
            kw = dict(lr=lr, max_epochs=max_epochs, smooth=self.smooth, optimiser=self.optm)
            if both:
                kw.update(criterions=self.criterion, weights=self.weight)
            elif self.weight is not None:
                kw.update(weights=self.weight)
            flowreg = direct_flow_register(target.shape[2:], **kw)
            flowreg.optimize(moving, target, self.device, self.debug)
            self.theta = flowreg.flow
            self.warp = flowreg.deform
            self.losses = flowreg.losses
            self._flowreg = flowreg
        elif self.mode == 'flow':
            kw = dict(mode='bilinear', n=n, lr=lr, max_epochs=max_epochs)
            if both:
                kw.update(criterions=self.criterion, weights=self.weight)
            elif self.weight is not None:
                kw.update(weights=self.weight)
            flowreg = flow_register(target.shape[2:], **kw).to(self.device)
            flowreg.optimize(moving, target, self.device, self.debug)
            self.theta = flowreg.flow
            self.warp = flowreg.deform
            self.losses = flowreg.losses
            self._flowreg = flowreg
        else:
            fn = affine_register if self.mode == 'affine' else rigid_register
            probs = []
            kw = dict(lr=lr, epochs=max_epochs, per=per, device=self.device, debug=self.debug,
                      grad_edges=self.grad_edges, optm=self.optm, _want_warped=False, _problem_out=probs)
            if both:
                kw.update(criterions=self.criterion, weights=self.weight)
            elif self.weight is not None:
                kw.update(weights=self.weight)
            if reg0 is not None and self.mode == 'rigid':
                kw.update(reg0=reg0)
            if theta0 is not None and self.mode == 'affine':
                kw.update(theta0=theta0)
            _, theta = fn(moving, target, **kw)
            self.theta = theta[-1]                    # best theta, [1,nd,nd+1] ([N,nd,nd+1] for a batch: extension)
            self.losses = probs[0].losses[0] if moving.shape[0] == 1 else probs[0].losses   # device tensor(s): loss log
            self._last_problem = probs[0]             # final theta / params / best theta of the run (device state)

    def __call__(self, moving, *, mode='bilinear'):
        '''
        Warp `moving` [1,c,...] with the deformation found by `optim` (reference torchregister.py:108-129).
        `mode` (keyword-only extension): 'bilinear' (the reference's) or 'nearest', for label maps such as a
        segmentation or an atlas — only values of `moving` and 0 appear in the result.
        '''
        moving = moving.to(device=self.device, dtype=__import__('torch').float32)
        if self.mode == 'flow':
            return self.warp(moving, mode=mode)      # all channels in one launch
        return self.warp(self.theta, moving, mode=mode)
