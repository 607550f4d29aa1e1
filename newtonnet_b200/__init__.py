"""newtonnet_b200 - B200-native (sm_100a) energy / force / stress path of NewtonNet.

Drop-in for the hot path of THGLab/NewtonNet v2.1.0: `NewtonNet.forward(z, pos, cell, batch)` and
`MLAseCalculator`.  Hand-written CUDA kernels behind a C ABI (include/newtonnet_b200.h); PyTorch is
used for device memory, streams and torch.distributed only.  No CPU fallback.
"""
__version__ = '0.1.0'

from newtonnet_b200.models.newtonnet import NewtonNet  # noqa: F401
from newtonnet_b200.hessian import hessian  # noqa: F401,E402  (the function; the module is newtonnet_b200.hessian)
