"""datum_b200 — B200-native image-based-lighting bake behind pniekamp/datum's tools/ibl.h API.

The compute path is libdatum_ibl_cuda (hand-written sm_100a kernels behind the
C ABI of include/datum_ibl_cuda.h).  This package is the Python host side used
by the tests, the benchmark and the multi-GPU driver; the C++ host shim that
keeps the reference's tools/ibl.h signatures lives in datum_b200/host/.

There is no CPU implementation in this package: importing it works anywhere,
but every compute entry point raises if the CUDA library or a GPU is missing.
"""

from .ibl import (  # noqa: F401
    IblContext,
    MultiContext,
    IblError,
    FORMAT_RGBE,
    FORMAT_F32,
    FORMAT_F16,
    default_context,
    image_datasize,
    image_maxlevels,
    level_offsets,
    image_buildmips_cube_ibl,
    image_pack_cube_ibl,
    image_pack_envbrdf,
    image_pack_watercolor,
    project_sh9,
)
