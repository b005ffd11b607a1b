"""gfnerf_b200 -- B200-native (sm_100a) implementation of GF-NeRF's per-ray hot path.

The directory is named `gf-nerf_b200`; import it as `gfnerf_b200` (the repo-root shim
package of that name points its __path__ here).
"""
from . import _lib  # noqa: F401
from .hash_3d_anchored import Hash3DAnchored, Hash3DAnchoredCore  # noqa: F401
from .perssampler import PersSampler, PersSamplerCore  # noqa: F401
from .engine import GFNeRFEngine  # noqa: F401
from .field import FieldHeadNames, GFNeRFField  # noqa: F401
from .metrics import image_metrics  # noqa: F401
from .mlp import MLPNetwork  # noqa: F401
from .model import GFNeRFModel  # noqa: F401
from .cameras import Cameras  # noqa: F401
from .pixel_samplers import ErrorPixelSampler, update_error_map  # noqa: F401
from .rays import Frustums, RayBundle, RaySamples, WarpedSamples  # noqa: F401
from .renderers import AccumulationRenderer, DepthRenderer, RGBRenderer  # noqa: F401

__version__ = "0.1.0"
