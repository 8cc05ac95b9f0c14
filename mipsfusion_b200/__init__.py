"""mipsfusion_b200: B200-native (sm_100a CUDA) implementation of MIPSFusion's per-frame neural-field
hot path behind the reference's Python call surface.

    from mipsfusion_b200 import JointEncoding, get_encoder, MLP_reg, RandomOptimizer

The compute lives in ``libmipsfusion_b200.so`` (C ABI, include/mipsfusion_b200.h); importing this
package does not load it, the first kernel call does -- and raises if it has not been built."""
from ._lib import MipsFusionB200Error, lib, load_library  # noqa: F401
from ._lib import set_deterministic, get_deterministic  # noqa: F401
from .encodings import get_encoder, HashGridEncoding, FrequencyEncoding, IdentityEncoding  # noqa: F401
from .decoder import MLP_reg  # noqa: F401
from .scene_rep import JointEncoding  # noqa: F401
from .optim import FusedAdam, create_map_optimizer  # noqa: F401
from .random_optimizer import RandomOptimizer  # noqa: F401
from .joint_query import JointSubmapQuery, get_grid_uniform  # noqa: F401
from .keyframe_store import KeyframeRayStore, sample_without_replacement  # noqa: F401
from .render_full import render_full_img  # noqa: F401
from .tracker import FusedPoseRefiner, FusedTracker  # noqa: F401
from .submap_parallel import SubmapParallel  # noqa: F401
from .overlap import OverlapSDF  # noqa: F401
from . import sampling_helper  # noqa: F401
from .manager import SubmapContainment, pts_in_bbox  # noqa: F401
from . import marching_cubes  # noqa: F401  (module, like the reference's `marching_cubes` package: marching_cubes.marching_cubes(volume, isovalue, truncation))
from .marching_cubes import marching_cubes_device  # noqa: F401
from .mesher import MeshVisibility  # noqa: F401
from .mesh_utils import extract_mesh2, getVoxels  # noqa: F401
