"""pathtracercuda_b200 — B200-native (sm_100a) trace path behind the reference's `Pathtracer` interface.

The product is the C-ABI shared library `libpt_b200.so` (include/pt_b200.h) built from csrc/ by `make -C
pathtracercuda_b200/csrc`; this package is a thin ctypes mirror of the reference's host class so tests and the bench
read like the reference's call sites (reference: PathtracerCUDA/src/main.cpp:263-294, SceneLoader.cpp:124-348).
There is no CPU fallback: importing works anywhere, but creating a Pathtracer without the library or without a CUDA
device raises.
"""
from .abi import (ASSETS, MATERIALS, REPO_ROOT, SHAPES, CameraDesc, MaterialDesc, ObjectDesc, Stats, make_camera,
                  make_object, object_array, parse_scene_py)
from .api import LIB_PATH, Pathtracer, PtError, camera_rotate, camera_translate, env_distribution, light_distribution, load_library, parse_scene_file, read_image, write_hdr, write_png

__all__ = ["Pathtracer", "PtError", "camera_rotate", "camera_translate", "load_library", "env_distribution", "light_distribution", "parse_scene_file", "read_image", "write_hdr", "write_png", "LIB_PATH",
           "make_object", "make_camera", "object_array", "parse_scene_py", "ObjectDesc", "MaterialDesc", "CameraDesc", "Stats",
           "SHAPES", "MATERIALS", "ASSETS", "REPO_ROOT"]
