"""State replaced on a reused context - the scene with its counts and emitter table, the sky's importance tables, the buffers of the
parity aids - renders the very bits a fresh context renders with the same scene, sky and options."""
import numpy as np
import pytest

import pathtracercuda_b200 as pt
from tests.helpers import bits, seven_shape_scene

W, H, SPP = 48, 36, 16


def _cornell_box():
    objs, _, _, cam = pt.parse_scene_py(f"{pt.ASSETS}/scenes/cornell_box.json", W, H)
    return objs, cam


SCENES = {"cornell_box": _cornell_box, "seven_shapes": lambda: seven_shape_scene(W, H)}


def _context():
    """a context with the two textures of every render here: earth.png (handle 1, cornell_box's sphere; also a sky) and skybox.hdr"""
    P = pt.Pathtracer(W, H)
    assert P.loadTexture(f"{pt.ASSETS}/earth.png") == 1
    assert P.loadTexture(f"{pt.ASSETS}/skybox.hdr") == 2
    return P


def _frame(P, cam, first_hit=False):
    P.render(cam, SPP, True)
    out = [bits(P.getHDRSum()), P.stats().rays]
    return out + list(P.firstHit()) if first_hit else out


def _fresh(scene, sky=0, **opts):
    objs, cam = SCENES[scene]()
    with _context() as P:
        P.setScene(objs)
        P.setSkyboxTextureHandle(sky)
        for k, v in opts.items():
            P.setOption(k, v)
        return _frame(P, cam, opts.get("first_hit", 0))


def _assert_same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_scene_replaced_on_a_reused_context():
    """light_is: cornell_box (one emitter), the seven-shape scene (eight), cornell_box again on one context"""
    with _context() as P:
        P.setOption("light_is", 1)
        for scene in ("cornell_box", "seven_shapes", "cornell_box"):
            objs, cam = SCENES[scene]()
            P.setScene(objs)
            _assert_same(_frame(P, cam), _fresh(scene, light_is=1))


@pytest.mark.gpu
def test_sky_switched_on_a_reused_context():
    """env_is: the importance tables follow the sky handle 1 -> 2 -> 1"""
    objs, cam = SCENES["seven_shapes"]()
    want = {sky: _fresh("seven_shapes", sky, env_is=1) for sky in (1, 2)}
    assert not np.array_equal(want[1][0], want[2][0])
    with _context() as P:
        P.setScene(objs)
        P.setOption("env_is", 1)
        for sky in (1, 2, 1):
            P.setSkyboxTextureHandle(sky)
            _assert_same(_frame(P, cam), want[sky])


@pytest.mark.gpu
def test_parity_aids_toggled_on_a_reused_context():
    """first_hit on, off, on; then jitter 0, 1, 0 (with first_hit still on)"""
    objs, cam = SCENES["cornell_box"]()
    opts = {}
    with _context() as P:
        P.setScene(objs)
        for key, v in (("first_hit", 1), ("first_hit", 0), ("first_hit", 1), ("jitter", 0), ("jitter", 1), ("jitter", 0)):
            P.setOption(key, v)
            opts[key] = v
            _assert_same(_frame(P, cam, opts["first_hit"]), _fresh("cornell_box", **opts))
