"""ctypes loaders for the CHECKERS: oracle/_build/libpt_oracle.so (our CPU restatement) and
oracle/_ref/libref_host.so (the reference's own host math).  TEST INFRASTRUCTURE ONLY — imported by tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs, never by pathtracercuda_b200/."""
import ctypes as C
import os
import subprocess

import numpy as np

from pathtracercuda_b200.abi import CameraDesc, MaterialDesc, ObjectDesc, object_array

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "_build", "libpt_oracle.so")
REF_HOST_SO = os.path.join(HERE, "_ref", "libref_host.so")
REF_PT = os.path.join(HERE, "_ref", "ref_pt")
REF_PT_SEEDB = os.path.join(HERE, "_ref", "ref_pt_seedB")
REF_GPU = os.path.join(HERE, "_ref", "ref_gpu")


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    """our CPU restatement (oracle/pt_oracle.c)"""

    def __init__(self, objects):
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        L = C.CDLL(ORACLE_SO)
        self.L = L
        L.orc_scene_create.restype = C.c_void_p
        L.orc_scene_create.argtypes = [C.c_size_t, C.c_void_p]
        L.orc_scene_destroy.argtypes = [C.c_void_p]
        L.orc_add_texture.restype = C.c_uint32
        L.orc_add_texture.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
        L.orc_set_skybox.argtypes = [C.c_void_p, C.c_uint32]
        L.orc_bvh_info.argtypes = [C.c_void_p] * 4
        L.orc_object_info.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.orc_camera_ray.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_void_p]
        L.orc_hit_object.restype = C.c_int
        L.orc_hit_object.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p]
        L.orc_material_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p]
        L.orc_primary_pass.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_trace_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_render.restype = C.c_uint64
        L.orc_render.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_void_p]
        L.orc_tonemap.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]
        L.orc_philox.argtypes = [C.c_uint32] * 6 + [C.c_void_p]
        L.orc_uniform.restype = C.c_float
        L.orc_uniform.argtypes = [C.c_uint32]
        L.orc_texture_lookup.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_void_p]
        self.n = len(objects)
        self.env_is = self.light_is = False
        self._arr = object_array(objects)
        self.s = L.orc_scene_create(self.n, C.byref(self._arr))

    def __del__(self):
        try:
            self.L.orc_scene_destroy(self.s)
        except Exception:
            pass

    def add_texture(self, img):
        img = np.ascontiguousarray(img)
        is_hdr = img.dtype == np.float32
        assert img.ndim == 3 and img.shape[2] == 4 and (is_hdr or img.dtype == np.uint8)
        return self.L.orc_add_texture(self.s, img.shape[1], img.shape[0], int(is_hdr), _p(img))

    def set_skybox(self, h):
        self.L.orc_set_skybox(self.s, h)

    def set_env_is(self, on):
        """the product's option "env_is" (not the reference): sky importance sampling + multiple importance sampling"""
        if on and self.light_is:
            raise ValueError("env_is and light_is cannot be combined (pt_render refuses it too)")
        self.L.orc_set_env_is.argtypes = [C.c_void_p, C.c_int]
        self.L.orc_set_env_is(self.s, int(on))
        self.env_is = bool(on)

    def env_tables(self):
        """(cols, rows, q, alias, density) of the sky distribution built by set_env_is(1)"""
        self.L.orc_env_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        self.L.orc_env_tables.restype = C.c_uint32
        cols, rows = C.c_uint32(), C.c_uint32()
        n = self.L.orc_env_tables(self.s, C.byref(cols), C.byref(rows), None, None, None)
        q, alias, dens = np.zeros(n, np.float32), np.zeros(n, np.uint32), np.zeros(n, np.float32)
        self.L.orc_env_tables(self.s, None, None, _p(q), _p(alias), _p(dens))
        return cols.value, rows.value, q, alias, dens

    def env_sample(self, r):
        """r: (n, 3) uint32 random words -> (n, 6): direction, u, v, pdf"""
        self.L.orc_env_sample.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        r = np.ascontiguousarray(r, np.uint32)
        out = np.zeros((r.shape[0], 6), np.float32)
        row = np.zeros(6, np.float32)
        for i in range(r.shape[0]):
            self.L.orc_env_sample(self.s, int(r[i, 0]), int(r[i, 1]), int(r[i, 2]), _p(row))
            out[i] = row
        return out

    def set_light_is(self, on):
        """the product's option "light_is" (not the reference): emitter importance sampling + multiple importance sampling"""
        if on and self.env_is:
            raise ValueError("env_is and light_is cannot be combined (pt_render refuses it too)")
        self.L.orc_set_light_is.argtypes = [C.c_void_p, C.c_int]
        self.L.orc_set_light_is(self.s, int(on))
        self.light_is = bool(on)

    def light_table(self):
        """(scene_index, prob, q, alias) of the emitter table built by set_light_is(1)"""
        self.L.orc_light_table.argtypes = [C.c_void_p] * 5
        self.L.orc_light_table.restype = C.c_uint32
        n = self.L.orc_light_table(self.s, None, None, None, None)
        idx, prob, q, alias = np.zeros(n, np.uint32), np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.uint32)
        self.L.orc_light_table(self.s, _p(idx), _p(prob), _p(q), _p(alias))
        return idx, prob, q, alias

    def light_sample_points(self, q):
        """q: (n, 4) uint32 random words -> (n, 8): world point, area pdf without the selection probability, emitter, local point"""
        self.L.orc_light_sample_point.argtypes = [C.c_void_p] * 3
        q = np.ascontiguousarray(q, np.uint32)
        out = np.zeros((q.shape[0], 8), np.float32)
        row = np.zeros(8, np.float32)
        for i in range(q.shape[0]):
            self.L.orc_light_sample_point(self.s, _p(q[i]), _p(row))
            out[i] = row
        return out

    def bvh_info(self):
        n, d, v = C.c_uint32(), C.c_uint32(), C.c_int32()
        self.L.orc_bvh_info(self.s, C.byref(n), C.byref(d), C.byref(v))
        return n.value, d.value, bool(v.value)

    def object_info(self, i):
        rows = np.zeros(12, np.float32)
        box = np.zeros(6, np.float32)
        self.L.orc_object_info(self.s, i, _p(rows), _p(box))
        return rows, box

    def camera_ray(self, cam, s, t):
        out = np.zeros(6, np.float32)
        self.L.orc_camera_ray(C.byref(cam), s, t, _p(out))
        return out

    def hit_object(self, i, o, d, tmin=0.001, tmax=3.4028234663852886e38):
        o = np.asarray(o, np.float32)
        d = np.asarray(d, np.float32)
        out = np.zeros(10, np.float32)
        ok = self.L.orc_hit_object(self.s, i, _p(o), _p(d), tmin, tmax, _p(out))
        return (out if ok else None)

    def decision_margin(self, i, o, d):
        """how far the ray is from flipping a decision of object i's intersection routine, in units of float32 rounding noise"""
        o = np.asarray(o, np.float32)
        d = np.asarray(d, np.float32)
        self.L.orc_decision_margin.restype = C.c_double
        self.L.orc_decision_margin.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        return float(self.L.orc_decision_margin(self.s, i, _p(o), _p(d)))

    def material_sample(self, mat, N, in_dir, rnd0, rnd1):
        N = np.asarray(N, np.float32)
        in_dir = np.asarray(in_dir, np.float32)
        out = np.zeros(9, np.float32)
        self.L.orc_material_sample(C.byref(mat), _p(N), _p(in_dir), rnd0, rnd1, _p(out))
        return out

    def primary_pass(self, cam, w, h):
        idx = np.zeros(w * h, np.int32)
        t = np.zeros(w * h, np.float32)
        st = np.zeros(2, np.uint64)
        self.L.orc_primary_pass(self.s, C.byref(cam), w, h, _p(idx), _p(t), _p(st))
        return idx, t, st

    def trace_rays(self, o, d, tmin=0.001):
        o = np.ascontiguousarray(o, np.float32)
        d = np.ascontiguousarray(d, np.float32)
        n = o.shape[0]
        idx = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        nrm = np.zeros((n, 3), np.float32)
        self.L.orc_trace_rays(self.s, n, _p(o), _p(d), tmin, _p(idx), _p(t), _p(nrm))
        return idx, t, nrm

    def render(self, cam, w, h, spp, seed=1984, sample_offset=0, sample_stride=1, accum=None, max_bounces=5, stratify=None):
        """stratify: the product's first-bounce stratification (include/pt_b200.h option "stratify"); None = the product's
        default, on from 128 spp"""
        self.L.orc_set_stratify(int(spp >= 128 if stratify is None else stratify))
        add = accum is not None
        if accum is None:
            accum = np.zeros((h, w, 4), np.float32)
        rays = self.L.orc_render(self.s, C.byref(cam), w, h, spp, seed, sample_offset, sample_stride, int(add), max_bounces, _p(accum))
        return accum, rays

    def threads(self, n=0):
        """OpenMP threads render() uses; n > 0 sets the count first"""
        return int(self.L.orc_threads(int(n)))

    def tonemap(self, accum, sample_count):
        accum = np.ascontiguousarray(accum, np.float32)
        out = np.zeros(accum.shape[:-1] + (4,), np.uint8)
        self.L.orc_tonemap(_p(accum), accum.size // 4, sample_count, _p(out))
        return out

    def philox(self, c, k):
        out = np.zeros(4, np.uint32)
        self.L.orc_philox(*[int(x) for x in c], *[int(x) for x in k], _p(out))
        return out

    def texture_lookup(self, handle, u, v):
        out = np.zeros(4, np.float32)
        self.L.orc_texture_lookup(self.s, handle, u, v, _p(out))
        return out


def have_ref_host():
    return os.path.exists(REF_HOST_SO)


class RefHost:
    """the reference's own host/device math, g++ build (oracle/_ref/libref_host.so).  Process-global state."""

    def __init__(self):
        L = C.CDLL(REF_HOST_SO)
        self.L = L
        L.refh_load_scene_file.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32]
        L.refh_set_scene.argtypes = [C.c_size_t, C.c_void_p]
        L.refh_set_camera.argtypes = [C.c_void_p]
        L.refh_get_camera.argtypes = [C.c_void_p]
        L.refh_texture_path.restype = C.c_char_p
        L.refh_skybox_handle.restype = C.c_uint32
        L.refh_set_sky.argtypes = [C.c_int, C.c_int, C.c_void_p]
        L.refh_object_bytes.argtypes = [C.c_int, C.c_void_p]
        L.refh_bvh_info.argtypes = [C.c_void_p] * 3
        L.refh_hit_object.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p]
        L.refh_aabb_hit.argtypes = [C.c_void_p] * 4 + [C.c_float, C.c_float]
        L.refh_camera_ray.argtypes = [C.c_float, C.c_float, C.c_void_p]
        L.refh_material_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.refh_tonemap.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]
        L.refh_primary_pass.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.refh_trace_rays.argtypes = [C.c_size_t, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
        L.refh_render.restype = C.c_uint64
        L.refh_render.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]

    def threads(self, n=0):
        """OpenMP threads render() uses; n > 0 sets the count first"""
        return int(self.L.refh_threads(int(n)))

    def load_scene_file(self, path, w, h, cwd=None):
        old = os.getcwd()
        try:
            if cwd:
                os.chdir(cwd)
            return self.L.refh_load_scene_file(os.fsencode(path), w, h)
        finally:
            os.chdir(old)

    def set_scene(self, objects):
        arr = object_array(objects)
        return self.L.refh_set_scene(len(objects), C.byref(arr))

    def set_camera(self, cam):
        self.L.refh_set_camera(C.byref(cam))

    def get_camera(self):
        out = np.zeros(23, np.float32)
        self.L.refh_get_camera(_p(out))
        return out

    def camera_rotate(self, pitch, yaw, roll=0.0):
        self.L.refh_camera_rotate(C.c_float(pitch), C.c_float(yaw), C.c_float(roll))

    def camera_translate(self, x, y, z):
        self.L.refh_camera_translate(C.c_float(x), C.c_float(y), C.c_float(z))

    def textures(self):
        return [self.L.refh_texture_path(i).decode() for i in range(self.L.refh_texture_count())], self.L.refh_skybox_handle()

    def set_sky(self, img):
        if img is None:
            self.L.refh_set_sky(0, 0, None)
            return
        img = np.ascontiguousarray(img, np.float32)
        self.L.refh_set_sky(img.shape[1], img.shape[0], _p(img))

    def object_bytes(self, i):
        out = np.zeros(128, np.uint8)
        n = self.L.refh_object_bytes(i, _p(out))
        assert n == 128
        rows = out[:48].view(np.float32).copy()
        mat = out[48:88].copy()
        box = out[88:112].view(np.float32).copy()
        typ = int(out[112:116].view(np.uint32)[0])
        return rows, mat, box, typ

    def bvh_info(self):
        n, d, v = C.c_uint32(), C.c_uint32(), C.c_int32()
        self.L.refh_bvh_info(C.byref(n), C.byref(d), C.byref(v))
        return n.value, d.value, bool(v.value)

    def hit_object(self, i, o, d, tmin=0.001, tmax=3.4028234663852886e38):
        o = np.asarray(o, np.float32)
        d = np.asarray(d, np.float32)
        out = np.zeros(10, np.float32)
        ok = self.L.refh_hit_object(i, _p(o), _p(d), tmin, tmax, _p(out))
        return out if ok else None

    def camera_ray(self, s, t):
        out = np.zeros(6, np.float32)
        self.L.refh_camera_ray(s, t, _p(out))
        return out

    def material_sample(self, mat, N, in_dir, seed):
        N = np.asarray(N, np.float32)
        in_dir = np.asarray(in_dir, np.float32)
        out = np.zeros(13, np.float32)
        self.L.refh_material_sample(C.byref(mat), _p(N), _p(in_dir), seed, _p(out))
        return out

    def tonemap(self, accum, sample_count):
        accum = np.ascontiguousarray(accum, np.float32)
        out = np.zeros(accum.shape[:-1] + (4,), np.uint8)
        self.L.refh_tonemap(_p(accum), accum.size // 4, sample_count, _p(out))
        return out

    def primary_pass(self, w, h):
        idx = np.zeros(w * h, np.int32)
        t = np.zeros(w * h, np.float32)
        st = np.zeros(2, np.uint64)
        self.L.refh_primary_pass(w, h, _p(idx), _p(t), _p(st))
        return idx, t, st

    def trace_rays(self, o, d, tmin=0.001):
        o = np.ascontiguousarray(o, np.float32)
        d = np.ascontiguousarray(d, np.float32)
        n = o.shape[0]
        idx = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        nrm = np.zeros((n, 3), np.float32)
        self.L.refh_trace_rays(n, _p(o), _p(d), tmin, _p(idx), _p(t), _p(nrm))
        return idx, t, nrm

    def render(self, w, h, spp, seed_base=1984):
        accum = np.zeros((h, w, 4), np.float32)
        rays = self.L.refh_render(w, h, spp, seed_base, _p(accum))
        return accum, rays


def write_blob(path, objects, cam, width, height):
    """scene blob for oracle/_ref/ref_gpu (see oracle/ref_harness/ref_gpu.cu)"""
    import struct
    arr = object_array(objects)
    with open(path, "wb") as f:
        f.write(struct.pack("<4I", 0x32425450, width, height, len(objects)))
        f.write(bytes(cam))
        f.write(bytes(arr)[: len(objects) * C.sizeof(ObjectDesc)])


def ref_gpu_primary(objects, cam, width, height, workdir):
    """run the reference's own hitBVH on the GPU for pixel-centre rays -> (scene-order index, t)"""
    blob = os.path.join(workdir, "scene.blob")
    out = os.path.join(workdir, "primary.bin")
    write_blob(blob, objects, cam, width, height)
    subprocess.check_call([REF_GPU, "primary", blob, out], stdout=subprocess.DEVNULL)
    n = width * height
    raw = np.fromfile(out, np.uint8)
    return raw[: n * 4].view(np.int32).copy(), raw[n * 4: n * 8].view(np.float32).copy()


def ref_gpu_count(objects, cam, width, height, spp, workdir):
    """rays the reference traceKernel traces for this scene/size/spp (its own seeds and 8-spp slicing)"""
    import json
    blob = os.path.join(workdir, "scene.blob")
    write_blob(blob, objects, cam, width, height)
    return json.loads(subprocess.check_output([REF_GPU, "count", blob, str(spp)]).decode().strip().splitlines()[-1])
