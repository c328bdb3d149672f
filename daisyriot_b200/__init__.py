"""daisyriot_b200 -- B200-native form-factor build + radiosity/fluorescence gather behind DaisyRiot's entry points.

``libdaisy_b200.so`` (hand-written sm_100a CUDA, C-ABI in ``include/daisy_b200.h``) is the product; this package is
the host-side mirror of the reference's classes for that path.  There is no CPU fallback."""
from ._lib import DaisyError, FF_DEVICE, FF_HOST, build, lib  # noqa: F401
from .api import (BWLightning, DeviceGroup, GroupSolver, Lightning, MeshS, OptixPrimeFunctionality, RadMat, RGBLightning,  # noqa: F401
                  SpectralLightning, cie1931WavelengthToXYZFit, deserialize_mat, remap_bands, serialize_mat)
from .scenes import RAYS_PER_PATCH, Scene, cornell_box, load_obj, load_scene_npz, msvc_sample_pattern, save_scene_npz  # noqa: F401
