"""cpuvox_b200 — B200-native raybuffer renderer (the hot path of pipliz/cpuvox) behind a C ABI.

The product is cpuvox_b200/libcpuvox_b200.so (CUDA, sm_100a); this package is the thin host mirror of the
reference's RenderManager/World/Camera surface used by tests and bench.py. Importing fails loudly if the
shared library has not been built — there is no CPU or Python fallback.
"""
from .native import LIB_PATH, CvxError, FrameSetup, LOD_LEVELS  # noqa: F401
from .host import (  # noqa: F401
    BOX_DTYPE,
    RAY_DTYPE,
    RAY_HIT_DTYPE,
    SKYBOX_ARGB,
    CameraPose,
    RenderManager,
    World,
    algorithmic_bytes,
    alloc_pinned,
    benchmark_length,
    benchmark_path,
    benchmark_pose,
    frame_setup,
    make_boxes,
    make_rays,
    screen_ray,
    setup_lods,
    write_bmp,
)
from .parallel import ShardedRenderManager, broadcast_world, partition_rays, partition_views, ray_weights  # noqa: F401,E402
