"""ctypes wrapper of tests/device_probe.cu (the trace kernels' device routines, one call per thread) and the module-scoped `probe`
fixture that builds it; test modules import the fixture from here"""
import ctypes as C
import functools
import os
import subprocess
import tempfile

import numpy as np
import pytest

import pathtracercuda_b200 as pt
from tests.helpers import ROOT

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(ROOT, "pathtracercuda_b200", "csrc")
NVCC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
# the product's flags (csrc/Makefile) plus -shared; -fopenmp / -lgomp for scene_compile.cpp's parallel sort
NVFLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC,-fopenmp,-ffp-contract=off"]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Probe:
    def __init__(self, path, ptxas_log):
        self.log = ptxas_log
        L = self.L = C.CDLL(path)
        vp, u32 = C.c_void_p, C.c_uint32
        L.probe_material.argtypes = [u32, vp, vp]
        L.probe_scene_create.restype = vp
        L.probe_scene_create.argtypes = [C.c_size_t, vp]
        L.probe_scene_destroy.argtypes = [vp]
        L.probe_scene_info.restype = u32
        L.probe_scene_info.argtypes = [vp, vp]
        L.probe_hit.argtypes = [vp, C.c_int, u32, vp, vp, vp, C.c_float, vp, vp]
        L.probe_light.argtypes = [vp, u32, vp, vp, vp]
        L.probe_env.argtypes = [u32, u32, C.c_int, vp, C.c_int, u32, vp, vp]
        L.probe_tex.argtypes = [u32, u32, C.c_int, vp, C.c_int, u32, vp, vp]
        L.probe_angles.argtypes = [u32, vp, vp]

    def tex(self, img, u, v, unit):
        """texLookup at (u, v) on an (H, W, 4) uint8 or float32 texture; unit 1 = through a texture object -> (n, 3) rgb"""
        img = np.ascontiguousarray(img)
        uv = np.ascontiguousarray(np.stack([u, v], 1), np.float32)
        out = np.zeros((len(uv), 3), np.float32)
        assert self.L.probe_tex(img.shape[1], img.shape[0], int(img.dtype == np.float32), _p(img), int(unit), len(uv), _p(uv), _p(out)) == 0
        return out

    def angles(self, y, x, c, p):
        """-> (n, 4): fastAtan2(y, x), fastAtan2Inline(y, x), fastAcos(c), fastPow(p, 2.2f)"""
        inp = np.ascontiguousarray(np.stack([y, x, c, p], 1), np.float32)
        out = np.zeros((len(inp), 4), np.float32)
        assert self.L.probe_angles(len(inp), _p(inp), _p(out)) == 0
        return out

    def material(self, inp):
        inp = np.ascontiguousarray(inp, np.float32)
        out = np.zeros((len(inp), 32), np.float32)
        assert self.L.probe_material(len(inp), _p(inp), _p(out)) == 0
        return out

    def env(self, img, q, mode=0):
        img = np.ascontiguousarray(img, np.float32)
        q = np.ascontiguousarray(q, np.uint32 if mode == 0 else np.float32)
        out = np.zeros((len(q), 8) if mode == 0 else len(q), np.float32)
        assert self.L.probe_env(img.shape[1], img.shape[0], 1, _p(img), mode, len(q), _p(q), _p(out)) == 0
        return out


class ProbeScene:
    """a scene compiled and given its emitter table by the product's host code, uploaded as the render kernels see it"""

    def __init__(self, probe, objects):
        self.L = probe.L
        self._arr = pt.abi.object_array(objects)
        self.h = self.L.probe_scene_create(len(objects), C.byref(self._arr))
        assert self.h
        self.prim_of = np.zeros(len(objects), np.int32)
        self.emitters = self.L.probe_scene_info(self.h, _p(self.prim_of))
        self.object_of = np.argsort(self.prim_of)

    def __del__(self):
        try:
            self.L.probe_scene_destroy(self.h)
        except Exception:
            pass

    def hit(self, obj, o, d, tmax, exact, clip, tmin=0.001):
        n = len(o)
        prim = np.ascontiguousarray(self.prim_of[np.asarray(obj)], np.int32)
        o, d, tmax = (np.ascontiguousarray(x, np.float32) for x in (o, d, tmax))
        out = np.zeros((n, 12), np.float32)
        assert self.L.probe_hit(self.h, int(exact) | 2 * int(clip), n, _p(prim), _p(o), _p(d), tmin, _p(tmax), _p(out)) == 0
        return out

    def light(self, q, p):
        q, p = np.ascontiguousarray(q, np.uint32), np.ascontiguousarray(p, np.float32)
        out = np.zeros((len(q), 8), np.float32)
        assert self.L.probe_light(self.h, len(q), _p(q), _p(p), _p(out)) == 0
        return out


@functools.cache
def _build():
    """nvcc the probe once per test process -> (library path, nvcc output with the ptxas report)"""
    out = os.path.join(tempfile.mkdtemp(prefix="device_probe_"), "libdevice_probe.so")
    srcs = [os.path.join(HERE, "device_probe.cu")] + [os.path.join(CSRC, f) for f in ("scene_compile.cpp", "light_sampling.cpp", "env_sampling.cpp")]
    r = subprocess.run([NVCC] + NVFLAGS + ["-Xptxas", "-v", "-shared", "-o", out] + srcs + ["-lgomp"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return out, r.stdout + r.stderr


@pytest.fixture(scope="module")
def probe():
    return Probe(*_build())


def _rng(tag):
    return np.random.default_rng(sum(map(ord, tag)))
