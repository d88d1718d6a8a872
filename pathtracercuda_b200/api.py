"""ctypes binding of libpt_b200.so + a Python mirror of the reference's `class Pathtracer`
(reference: PathtracerCUDA/src/pathtracer/Pathtracer.h:12-69)."""
import ctypes as C
import os

import numpy as np

from .abi import CameraDesc, ObjectDesc, Stats, object_array

LIB_PATH = os.environ.get("PT_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libpt_b200.so")
_lib = None


class PtError(RuntimeError):
    pass


def load_library():
    """Load libpt_b200.so (fails loudly when it has not been built; there is no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PtError(f"{LIB_PATH} is missing: build it with `make -C pathtracercuda_b200/csrc` (or __graft_entry__.build())")
    L = C.CDLL(LIB_PATH)
    vp, u32, i32, f32, sz, cp = C.c_void_p, C.c_uint32, C.c_int, C.c_float, C.c_size_t, C.c_char_p
    sig = {
        "pt_create": (i32, [u32, u32, i32, C.POINTER(vp)]),
        "pt_create_multi": (i32, [u32, u32, u32, C.POINTER(vp)]),
        "pt_get_multi_info": (i32, [vp, vp, vp, vp, vp]),
        "pt_destroy": (None, [vp]),
        "pt_set_scene": (i32, [vp, sz, vp]),
        "pt_set_scene_xform": (i32, [vp, sz, vp]),
        "pt_render_vectors": (i32, [vp, vp, u32, i32]),
        "pt_load_texture": (u32, [vp, cp]),
        "pt_load_texture_mem": (u32, [vp, u32, u32, i32, vp]),
        "pt_set_skybox": (i32, [vp, u32]),
        "pt_render": (i32, [vp, vp, u32, i32]),
        "pt_get_timing_ms": (f32, [vp]),
        "pt_get_hdr": (vp, [vp]),
        "pt_get_hdr_mean": (vp, [vp]),
        "pt_get_hdr_sum": (vp, [vp]),
        "pt_get_ldr": (vp, [vp]),
        "pt_set_option": (i32, [vp, cp, C.c_double]),
        "pt_get_stats": (i32, [vp, vp]),
        "pt_camera_rotate": (None, [vp, f32, f32, f32]),
        "pt_camera_translate": (None, [vp, f32, f32, f32]),
        "pt_primary_pass": (i32, [vp, vp, vp, vp]),
        "pt_trace_rays": (i32, [vp, sz, vp, vp, f32, vp, vp, vp]),
        "pt_get_first_hit": (i32, [vp, vp, vp]),
        "pt_accum_device_ptr": (vp, [vp]),
        "pt_set_accum_device_ptr": (i32, [vp, vp]),
        "pt_load_scene_file": (i32, [vp, cp, vp]),
        "pt_parse_scene_file": (i32, [cp, vp, sz, vp, f32, vp, sz, vp]),
        "pt_write_png": (i32, [cp, u32, u32, vp]),
        "pt_write_hdr": (i32, [cp, u32, u32, vp]),
        "pt_env_distribution": (i32, [u32, u32, i32, vp, vp, vp, vp, vp]),
        "pt_light_distribution": (i32, [sz, vp, vp, vp, vp]),
        "pt_read_image": (i32, [cp, vp, vp, vp, vp]),
        "pt_free": (None, [vp]),
        "pt_last_error": (cp, []),
        "pt_version": (cp, []),
    }
    for name, (res, args) in sig.items():
        if os.environ.get("PT_B200_LIB") and not hasattr(L, name):
            continue  # (an experiment build of an older revision, tools/exp.py: it may lack the newest entry points)
        fn = getattr(L, name)  # AttributeError here = the library does not export what include/pt_b200.h declares
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTS = ["pt_create", "pt_create_multi", "pt_get_multi_info", "pt_destroy", "pt_set_scene", "pt_set_scene_xform", "pt_render_vectors", "pt_load_texture", "pt_load_texture_mem", "pt_set_skybox", "pt_render",
           "pt_get_timing_ms", "pt_get_hdr", "pt_get_hdr_mean", "pt_get_hdr_sum", "pt_get_ldr", "pt_set_option", "pt_get_stats", "pt_camera_rotate", "pt_camera_translate", "pt_primary_pass",
           "pt_trace_rays", "pt_get_first_hit", "pt_accum_device_ptr", "pt_set_accum_device_ptr", "pt_load_scene_file", "pt_parse_scene_file",
           "pt_write_png", "pt_write_hdr", "pt_env_distribution", "pt_light_distribution", "pt_read_image", "pt_free", "pt_last_error", "pt_version"]


def _err(L):
    return (L.pt_last_error() or b"").decode(errors="replace")


def _check(L, rc, what):
    if rc != 0:
        raise PtError(f"{what} failed ({rc}): {_err(L)}")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def camera_rotate(cam, pitch, yaw, roll=0.0):
    """Camera::rotate (reference Camera.inl:30-48) on a pt_camera_desc, in place; radians"""
    load_library().pt_camera_rotate(C.byref(cam), pitch, yaw, roll)
    return cam


def camera_translate(cam, x, y, z):
    """Camera::translate (reference Camera.inl:50-52) on a pt_camera_desc, in place; along the camera's right / up / backward axes"""
    load_library().pt_camera_translate(C.byref(cam), x, y, z)
    return cam


def parse_scene_file(path, width, height, capacity=None):
    """pt_parse_scene_file: JSON -> (objects, texture_paths, skybox_index, camera); host only, no GPU needed."""
    L = load_library()
    cam = CameraDesc()
    sky = C.c_int32(0)
    n = L.pt_parse_scene_file(os.fsencode(path), None, 0, C.byref(cam), np.float32(width) / np.float32(height), None, 0, C.byref(sky))
    if n < 0:
        raise PtError(f"pt_parse_scene_file failed ({n}): {_err(L)}")
    arr = (ObjectDesc * max(n, 1))()
    buf = C.create_string_buffer(1 << 16)
    n2 = L.pt_parse_scene_file(os.fsencode(path), C.byref(arr), n, C.byref(cam), np.float32(width) / np.float32(height), buf, len(buf), C.byref(sky))
    assert n2 == n
    paths = buf.value.decode().split("\n") if buf.value else []
    return [arr[i] for i in range(n)], paths, sky.value, cam


def env_distribution(img):
    """pt_env_distribution: (cols, rows, q, alias, density) of the sky distribution option "env_is" samples; host only"""
    L = load_library()
    img = np.ascontiguousarray(img)
    is_hdr = img.dtype == np.float32
    assert img.ndim == 3 and img.shape[2] == 4 and (is_hdr or img.dtype == np.uint8)
    cols, rows = C.c_uint32(), C.c_uint32()
    n = L.pt_env_distribution(img.shape[1], img.shape[0], int(is_hdr), _p(img), C.byref(cols), C.byref(rows), None, None)
    if n < 0:
        raise PtError(f"pt_env_distribution failed ({n}): {_err(L)}")
    table, dens = np.zeros(2 * n, np.uint32), np.zeros(n, np.float32)
    L.pt_env_distribution(img.shape[1], img.shape[0], int(is_hdr), _p(img), None, None, _p(table), _p(dens))
    return cols.value, rows.value, table[0::2].copy().view(np.float32), table[1::2].copy(), dens


def light_distribution(objects):
    """pt_light_distribution: (scene_index, probability, q, alias) of the emitter table option "light_is" samples; host only"""
    L = load_library()
    arr = object_array(objects)
    n = L.pt_light_distribution(len(objects), C.byref(arr), None, None, None)
    if n < 0:
        raise PtError(f"pt_light_distribution failed ({n}): {_err(L)}")
    idx, prob, table = np.zeros(n, np.uint32), np.zeros(n, np.float32), np.zeros(2 * n, np.uint32)
    if n:
        L.pt_light_distribution(len(objects), C.byref(arr), _p(idx), _p(prob), _p(table))
    return idx, prob, table[0::2].copy().view(np.float32), table[1::2].copy()


def write_png(path, rgba):
    L = load_library()
    rgba = np.ascontiguousarray(rgba, np.uint8)
    _check(L, L.pt_write_png(os.fsencode(path), rgba.shape[1], rgba.shape[0], _p(rgba)), "pt_write_png")


def write_hdr(path, rgba):
    L = load_library()
    rgba = np.ascontiguousarray(rgba, np.float32)
    _check(L, L.pt_write_hdr(os.fsencode(path), rgba.shape[1], rgba.shape[0], _p(rgba)), "pt_write_hdr")


def read_image(path):
    """pt_read_image: decode PNG (-> uint8 RGBA) or Radiance HDR (-> float32 RGBA), top row first."""
    L = load_library()
    w, h, hdr, ptr = C.c_uint32(), C.c_uint32(), C.c_int(), C.c_void_p()
    _check(L, L.pt_read_image(os.fsencode(path), C.byref(w), C.byref(h), C.byref(hdr), C.byref(ptr)), "pt_read_image")
    try:
        n = w.value * h.value * 4
        if hdr.value:
            out = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_float)), (n,)).copy().reshape(h.value, w.value, 4)
        else:
            out = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), (n,)).copy().reshape(h.value, w.value, 4)
    finally:
        L.pt_free(ptr)
    return out


class Pathtracer:
    """Mirror of the reference's `class Pathtracer` (Pathtracer.h:12-69).  Reference-named methods (setScene, render,
    getTiming, loadTexture, setSkyboxTextureHandle, getHDRImageData, getImageData) keep the reference's argument
    meaning; the rest are the extensions of include/pt_b200.h."""

    def __init__(self, width, height, device=0, device_mask=0):
        """device_mask != 0: a multi-GPU context over these CUDA ordinals (pt_create_multi) - same methods"""
        self.L = load_library()
        self.width, self.height = int(width), int(height)
        h = C.c_void_p()
        if device_mask:
            _check(self.L, self.L.pt_create_multi(self.width, self.height, int(device_mask), C.byref(h)), "pt_create_multi")
        else:
            _check(self.L, self.L.pt_create(self.width, self.height, int(device), C.byref(h)), "pt_create")
        self.h = h
        self._objs = None

    def multiInfo(self):
        """(devices, peer_to_peer, trace_ms, exchange_ms) of the last render (pt_get_multi_info)"""
        n, p2p, tr, ex = C.c_int(), C.c_int(), C.c_float(), C.c_float()
        _check(self.L, self.L.pt_get_multi_info(self.h, C.byref(n), C.byref(p2p), C.byref(tr), C.byref(ex)), "pt_get_multi_info")
        return n.value, bool(p2p.value), tr.value, ex.value

    def close(self):
        if getattr(self, "h", None):
            self.L.pt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- reference interface -------------------------------------------------------------------------------------
    def setScene(self, objects):
        arr = object_array(objects)
        _check(self.L, self.L.pt_set_scene(self.h, len(objects), C.byref(arr)), "pt_set_scene")

    def loadTexture(self, path):
        return self.L.pt_load_texture(self.h, os.fsencode(path))

    def loadTextureMem(self, img):
        img = np.ascontiguousarray(img)
        is_hdr = img.dtype == np.float32
        assert img.ndim == 3 and img.shape[2] == 4 and (is_hdr or img.dtype == np.uint8)
        return self.L.pt_load_texture_mem(self.h, img.shape[1], img.shape[0], int(is_hdr), _p(img))

    def setSkyboxTextureHandle(self, handle):
        _check(self.L, self.L.pt_set_skybox(self.h, int(handle)), "pt_set_skybox")

    def render(self, camera, spp, ignoreHistory):
        _check(self.L, self.L.pt_render(self.h, C.byref(camera), int(spp), int(bool(ignoreHistory))), "pt_render")

    def getTiming(self):
        return self.L.pt_get_timing_ms(self.h)

    def _img(self, ptr, dtype):
        if not ptr:
            raise PtError("image readback failed: " + _err(self.L))
        ct = C.c_float if dtype == np.float32 else C.c_uint8
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), (self.height, self.width, 4))

    def getHDRImageData(self, copy=True):
        a = self._img(self.L.pt_get_hdr(self.h), np.float32)
        return a.copy() if copy else a

    def getImageData(self, copy=True):
        a = self._img(self.L.pt_get_ldr(self.h), np.uint8)
        return a.copy() if copy else a

    # ---- extensions ----------------------------------------------------------------------------------------------
    def getHDRMean(self, copy=True):
        a = self._img(self.L.pt_get_hdr_mean(self.h), np.float32)
        return a.copy() if copy else a

    def getHDRSum(self, copy=True):
        """the raw accumulation buffer (per-pixel sums, alpha = 1)"""
        a = self._img(self.L.pt_get_hdr_sum(self.h), np.float32)
        return a.copy() if copy else a

    def setOption(self, key, value):
        _check(self.L, self.L.pt_set_option(self.h, key.encode(), float(value)), "pt_set_option")

    def stats(self):
        s = Stats()
        _check(self.L, self.L.pt_get_stats(self.h, C.byref(s)), "pt_get_stats")
        return s

    def primaryPass(self, camera):
        idx = np.zeros(self.width * self.height, np.int32)
        t = np.zeros(self.width * self.height, np.float32)
        _check(self.L, self.L.pt_primary_pass(self.h, C.byref(camera), _p(idx), _p(t)), "pt_primary_pass")
        return idx, t

    def firstHit(self):
        """(index, t) per pixel of the camera rays' closest hits as found by the last render (option first_hit = 1)"""
        idx = np.zeros(self.width * self.height, np.int32)
        t = np.zeros(self.width * self.height, np.float32)
        _check(self.L, self.L.pt_get_first_hit(self.h, _p(idx), _p(t)), "pt_get_first_hit")
        return idx, t

    def traceRays(self, origins, directions, t_min=0.001, normals=True):
        o = np.ascontiguousarray(origins, np.float32)
        d = np.ascontiguousarray(directions, np.float32)
        n = o.shape[0]
        idx = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        nrm = np.zeros((n, 3), np.float32) if normals else None
        _check(self.L, self.L.pt_trace_rays(self.h, n, _p(o), _p(d), t_min, _p(idx), _p(t), _p(nrm) if normals else None), "pt_trace_rays")
        return idx, t, nrm

    def loadSceneFile(self, path, cwd=None):
        """loadScene(pathtracer, params) (SceneLoader.cpp:124-348); texture paths resolve against `cwd` (default: CWD)."""
        cam = CameraDesc()
        old = os.getcwd()
        try:
            if cwd:
                os.chdir(cwd)
            _check(self.L, self.L.pt_load_scene_file(self.h, os.fsencode(path), C.byref(cam)), "pt_load_scene_file")
        finally:
            os.chdir(old)
        return cam

    def accumDevicePtr(self):
        return self.L.pt_accum_device_ptr(self.h)

    def setAccumDevicePtr(self, ptr):
        _check(self.L, self.L.pt_set_accum_device_ptr(self.h, C.c_void_p(int(ptr))), "pt_set_accum_device_ptr")
