"""vloam-noted_b200: B200-native lidar registration hot path (scanRegistration ->
laserOdometry -> laserMapping of liuzm-slam/VLOAM-NOTED) behind a C ABI.

The directory name carries a hyphen; import it with
    importlib.import_module("vloam-noted_b200")
(tests/conftest.py and bench.py do)."""
from . import _build  # noqa: F401
from .api import (Context, Params, VloamError, load_lib, EXPORTS, ScanRegistration, LaserOdometry, LaserMapping,  # noqa: F401
                  LidarOdometryMapping, CLOUD_FULL, CLOUD_SHARP, CLOUD_LESS_SHARP, CLOUD_FLAT, CLOUD_LESS_FLAT,
                  CLOUD_CORNER_LAST, CLOUD_SURF_LAST, CLOUD_FULL_RES, FLAG_DISTORTION, FLAG_TRANSFORM_TO_END)
from . import synth  # noqa: F401
from . import kitti_io  # noqa: F401
from . import parallel  # noqa: F401
