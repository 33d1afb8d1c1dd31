"""torchregister_b200 — B200-native (sm_100a) implementation of the iterative registration
hot path of AgamChopra/TorchRegister, behind the reference's own API:

    import torchregister_b200 as tr
    warping = tr.Register(mode='rigid', device='cuda', weight=[0.5, 0.5, 0.])
    warping.optim(moving, target, max_epochs=500, lr=1e-5)
    warped = warping(moving);  theta = warping.theta
"""
from .utils import *            # noqa: F401,F403   (mirrors TR/__init__.py:1-3 star exports)
from .warpings import *         # noqa: F401,F403
from .torchregister import Register   # noqa: F401
from .metrics import jacobian_determinant, dice   # noqa: F401
from .transforms import affine_to_flow, compose_flow, invert_flow   # noqa: F401
from . import functional, synth, metrics, transforms      # noqa: F401

__version__ = '0.1.0'
