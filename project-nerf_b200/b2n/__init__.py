"""b2n -- host binding of the B200 ray-marching kernels (libb2nerf.so).

Importing this package loads the CUDA extension and raises ImportError if it
has not been built: there is deliberately no CPU fallback.
"""
from . import _lib  # noqa: F401  (fails loudly when the .so is missing)
from . import checkpoint, distortion as _distortion, errormap, graphs, importance, march, mesh, ops, optim, pose, render  # noqa: F401
# after the submodules: loading b2n/distortion.py sets the attribute ``b2n.distortion`` to the module, and the name
# belongs to the op
from .ops import (HashGeometry, check_errors, composite, distortion, fourier_encode, fused_mlp, hash_encode, instant_mlp, instant_sigma, linear,  # noqa: F401
                  mlp_precision,
                  set_mlp_precision, sigma_head)
from .distortion import render_rays_distortion  # noqa: F401
from .errormap import ErrorMap  # noqa: F401
from .importance import Hierarchical, render_image_hierarchical, render_rays_hierarchical  # noqa: F401
from .pose import PoseRefinement  # noqa: F401
from .render import Rendered, render_image_fast, render_rays_fast  # noqa: F401
