"""taichi_image_b200 -- B200-native (sm_100a) camera ISP hot path with the public API of
uc-vision/taichi_image's ``packed``, ``bayer``, ``tonemap``, ``color``, ``interpolate`` and
``camera_isp`` modules.  Python is only the host layer: every pixel operation is a hand-written CUDA
kernel in ``csrc/`` reached through the C ABI of ``include/b200isp.h`` (``libb200isp.so``); there is
no Taichi, no Triton, no backend dispatch and no CPU fallback.

    import taichi_image_b200 as ti_image
    from taichi_image_b200 import bayer, packed, camera_isp, u8, f16
"""
from . import _lib  # noqa: F401  (fails loudly if libb200isp.so is missing)
from .dtypes import (u8, u16, i16, f16, f32, uint8, uint16, int16, float16, float32, as_dtype)  # noqa: F401
from . import types, util, packed, bayer, tonemap, interpolate, color, camera_isp, distributed  # noqa: F401
from .camera_isp import Camera16, Camera32  # noqa: F401

__version__ = "0.1.1"
