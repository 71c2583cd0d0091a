"""b2n -- host binding of the B200 ray-marching kernels (libb2nerf.so).

Importing this package loads the CUDA extension and raises ImportError if it
has not been built: there is deliberately no CPU fallback.
"""
from . import _lib  # noqa: F401  (fails loudly when the .so is missing)
from .ops import (HashGeometry, check_errors, composite, fourier_encode, fused_mlp, hash_encode, instant_mlp, instant_sigma, linear,  # noqa: F401
                  mlp_precision,
                  set_mlp_precision, sigma_head)
from . import checkpoint, graphs, importance, march, mesh, ops, optim, render  # noqa: F401
from .importance import Hierarchical, render_image_hierarchical, render_rays_hierarchical  # noqa: F401
from .render import Rendered, render_image_fast, render_rays_fast  # noqa: F401
