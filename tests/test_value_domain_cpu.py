"""Known answers that pin the oracle on the value-domain cases (non-finite and extreme scene values), derived by hand
from the reference's expressions, and a check that every scene of the case table builds through rh_flatten.  The GPU
tests of tests/test_value_domain_gpu.py are only as good as this oracle.  No GPU needed."""
import math

import numpy as np
import pytest

from oracle.orc import OracleScene
from tests import value_cases as vc


def frame(rs, depth=0):
    return OracleScene(rs.raw).render(rs.camera, rs.width, rs.height, depth)


def test_zero_times_inf_in_diffuse_prints_255():
    """A Diffuse plane lit from behind, cd = (-1e200, .5, .5), light colour (1e200, 1, 1): l.n < 0, so diffuse is
    0 * (cd (*) lc) = 0 * -inf = NaN in red (Material.hs:31-33), and the ambient 0.2 * 0.5 = 0.1 in green and blue:
    [nan, .1, .1], which prints as [255, 25, 25] (min NaN 1 = 1; truncate 25.5 = 25)."""
    m = {"kind": "diffuse", "color1": (-vc.BIG, 0.5, 0.5)}
    rs = vc.scene([vc.with_mat(vc.PLANE, 0)], [m], [vc.point(vec=(0.2, 0.1, 3.0), color=(vc.BIG, 1, 1))])
    r = frame(rs)
    assert np.isnan(r["rgb_f64"][..., 0]).all() and (r["rgb_f64"][..., 1:] == 0.1).all()
    assert (r["rgb_u8"].reshape(-1, 3) == (255, 25, 25)).all() and (r["rgb_int"].reshape(-1, 3) == (255, 25, 25)).all()


@pytest.mark.parametrize("depth", [0, 1, 3])
def test_mirror_with_ior_minus_one_is_nan_at_any_depth(depth):
    """r0 1 (-1) = (2 / 0)^2 = inf, so fresnel = inf + (1 - inf) * x^5 is NaN (or inf - inf * 0 = NaN at normal
    incidence); the Mirror's colour is fresnel * specular, NaN whether specular is black (maxDepth) or not."""
    r = frame(vc.specular("mirror", -1.0), depth)
    c = r["rgb_f64"][vc.H // 2, vc.W // 2]
    assert np.isnan(c).all(), c
    assert (r["rgb_u8"][vc.H // 2, vc.W // 2] == 255).all()


def test_light_radius_minus_distance_has_an_infinite_falloff():
    """s = 1 + dd / (-dd) = 0, falloff = 1 / (0 * 0) = inf: the middle pixel's lit colour is +inf in every channel."""
    r = frame(vc.light_at_minus_distance())
    assert np.isposinf(r["rgb_f64"][vc.H // 2, vc.W // 2]).all()
    assert np.isfinite(r["rgb_f64"][0, 0]).all()


@pytest.mark.parametrize("size", [0.0, math.inf, math.nan])
def test_checker_size_without_a_remainder_selects_color2(size):
    """mod' u 0 (and mod' of a non-finite size) is NaN here, NaN * NaN < 0 is False: colorAt gives color2."""
    rs = vc.checker(size)
    orc = OracleScene(rs.raw)
    for u, v in ((0.3, 0.7), (-1.2, 0.1), (5.0, -3.0)):
        assert list(orc.color_at(0, u, v)) == [0.1, 0.3, 0.9]


def test_to_int_c_at_the_boundaries():
    """toIntC = truncate (255 * min c 1) (Image.hs:54-55), clamped to int32 in rgb_int: k/255 -> k, 1 and
    nextafter(1, 2) -> 255, 0.5 -> 127, -1/255 -> -1 (a negative channel), -0.999/255 and -0.0 -> 0, -inf -> INT32_MIN."""
    r = frame(vc.emitters())
    got = {tuple(x) for x in r["rgb_int"].reshape(-1, 3).tolist()}
    want = {(1, 2, 128), (255, 254, 255), (255, 127, 63), (-1, 0, 0), (-2 ** 31, 0, 255), (100, 37, 200), (0, 0, 0)}
    assert got == want, got
    neg = (r["rgb_int"] < 0).any(axis=-1)
    assert neg.sum() > 0 and np.array_equal(neg, (r["rgb_f64"] <= -1 / 255).any(axis=-1))


def test_nan_colour_prints_255_and_counts_as_no_negative():
    r = frame(vc.MATERIALS["nan"][0](*vc.MATERIALS["nan"][1]))
    assert (r["rgb_u8"][..., 0] == 255).all() and not (r["rgb_int"] < 0).any()


@pytest.mark.parametrize("name,factory", [(c[0], c[1]) for c in vc.cases()], ids=[c[0] for c in vc.cases()])
def test_case_scenes_flatten(name, factory):
    """rh_scene_create takes any double here: the flatten (host side, no device) accepts every case's scene."""
    rs = factory()
    assert rs.flat is not None
