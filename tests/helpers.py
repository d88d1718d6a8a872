"""shared helpers of the test-suite"""
import os

import numpy as np

import pathtracercuda_b200 as pt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
SHAPES7 = ["SPHERE", "CYLINDER", "DISK", "CONE", "PARABOLOID", "QUAD", "CUBE"]


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def golden_objects(d):
    import ctypes as C
    from pathtracercuda_b200.abi import CameraDesc, ObjectDesc
    raw = d["objects"].tobytes()
    n = len(raw) // C.sizeof(ObjectDesc)
    arr = (ObjectDesc * n).from_buffer_copy(raw)
    objs = [arr[i] for i in range(n)]
    cam = CameraDesc.from_buffer_copy(d["camera"].tobytes()) if "camera" in d.files else None
    return objs, cam


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def tie_aware_index_check(idx_a, t_a, idx_b, t_b, hit_t_fn, rel=1e-5):
    """Indices must match exactly, except at genuine geometric ties: a mismatching pixel is accepted only if the other
    side's object, intersected on its own with the same ray, hits at the same t (within `rel`) - SURVEY.md Q7/Q8.
    hit_t_fn(pixel, object_index) -> t or None.  Returns (n_mismatch, n_ties)."""
    mism = np.nonzero(idx_a != idx_b)[0]
    ties = 0
    for p in mism:
        ok = False
        if idx_a[p] >= 0 and idx_b[p] >= 0:
            ta = hit_t_fn(int(p), int(idx_a[p]))
            tb = hit_t_fn(int(p), int(idx_b[p]))
            if ta is not None and tb is not None and abs(ta - tb) <= rel * max(abs(ta), abs(tb)):
                ok = True
        assert ok, f"pixel {p}: index {idx_a[p]} (t={t_a[p]}) vs {idx_b[p]} (t={t_b[p]}) is not a geometric tie"
        ties += 1
    return len(mism), ties


def seven_shape_scene(W=48, H=36, seed=5):
    """a floor and a back wall that are not emitters, one emitter of every shape with a random rotation and non-uniform scale, and a
    large emissive panel (hoisted out of the BVH: its box spans the scene)"""
    rng = np.random.default_rng(seed)
    objs = [pt.make_object("QUAD", (0, 0, 0), (0, 0, 0), (4, 1, 4), base_color=(0.8, 0.8, 0.8)),
            pt.make_object("QUAD", (0, 2, -3), (90, 0, 0), (4, 1, 2), base_color=(0.6, 0.7, 0.8), material="LAMBERT_GGX", roughness=0.3),
            pt.make_object("QUAD", (0, 3.5, 0), (180, 0, 0), (3.5, 1, 3.5), emissive=(0.15, 0.15, 0.2))]
    for k, shape in enumerate(SHAPES7):
        pos = (-2.4 + 0.8 * k, 0.6 + 0.3 * (k % 2), -0.5 + 0.4 * (k % 3))
        rot = tuple(float(x) for x in rng.uniform(-180, 180, 3))
        sc = tuple(float(x) for x in rng.uniform(0.15, 0.35, 3))
        em = tuple(float(x) for x in rng.uniform(0.5, 4.0, 3))
        objs.append(pt.make_object(shape, pos, rot, sc, emissive=em, base_color=(0.5, 0.5, 0.5)))
    objs.append(pt.make_object("SPHERE", (0.3, 0.35, 0.8), (0, 0, 0), (0.35, 0.35, 0.35), material="GGX", roughness=0.2, base_color=(0.9, 0.8, 0.6)))
    cam = pt.make_camera((0, 1.6, 5.0), (0, 1.0, 0), 45.0, W / H)
    return objs, cam


def _local_ok(shape, lp, tol):
    x, y, z = lp[:, 0], lp[:, 1], lp[:, 2]
    r2 = x * x + z * z
    if shape == "SPHERE":
        return np.abs(np.sqrt(r2 + y * y) - 1) < tol
    if shape == "CYLINDER":
        return (np.abs(np.sqrt(r2) - 1) < tol) & (np.abs(y) <= 1 + tol)
    if shape == "DISK":
        return (np.abs(y) < tol) & (r2 <= 1 + tol)
    if shape == "QUAD":
        return (np.abs(y) < tol) & (np.abs(x) <= 1 + tol) & (np.abs(z) <= 1 + tol)
    if shape == "CUBE":
        return np.abs(np.abs(lp).max(1) - 1) < tol
    if shape == "CONE":
        return (np.abs(np.sqrt(r2) - np.abs(y)) < tol) & (np.abs(y) <= 1 + tol)
    return (np.abs(y - r2) < tol) & (y <= 1 + tol)  # PARABOLOID


def _mapped_area(shape, M, n=256):
    """world area of the mapped local surface by a fine triangulation (numpy, independent of the sampler)"""
    def grid(f, u0, u1, v0, v1):
        u, v = np.meshgrid(np.linspace(u0, u1, n + 1), np.linspace(v0, v1, n + 1), indexing="ij")
        P = f(u, v) @ M[:, :3].T + M[:, 3]
        a, b, c, d = P[:-1, :-1], P[1:, :-1], P[1:, 1:], P[:-1, 1:]
        return 0.5 * (np.linalg.norm(np.cross(b - a, c - a), axis=-1).sum() + np.linalg.norm(np.cross(c - a, d - a), axis=-1).sum())
    st = lambda *c: np.stack(np.broadcast_arrays(*c), -1)
    if shape == "SPHERE":
        return grid(lambda t, p: st(np.sin(t) * np.cos(p), np.cos(t), np.sin(t) * np.sin(p)), 0, np.pi, 0, 2 * np.pi)
    if shape == "CYLINDER":
        return grid(lambda y, p: st(np.cos(p), y, np.sin(p)), -1, 1, 0, 2 * np.pi)
    if shape == "DISK":
        return grid(lambda r, p: st(r * np.cos(p), 0 * r, r * np.sin(p)), 0, 1, 0, 2 * np.pi)
    if shape == "QUAD":
        return grid(lambda a, b: st(a, 0 * a, b), -1, 1, -1, 1)
    if shape == "CONE":
        return sum(grid(lambda h, p, s=s: st(h * np.cos(p), s * h, h * np.sin(p)), 0, 1, 0, 2 * np.pi) for s in (-1, 1))
    if shape == "PARABOLOID":
        return grid(lambda r, p: st(r * np.cos(p), r * r, r * np.sin(p)), 0, 1, 0, 2 * np.pi)
    tot = 0.0
    for ax in range(3):
        for s in (-1.0, 1.0):
            def f(a, b, ax=ax, s=s):
                c = [a, b]
                c.insert(ax, s + 0 * a)
                return st(*c)
            tot += grid(f, -1, 1, -1, 1)
    return tot
