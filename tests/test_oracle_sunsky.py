"""The host-side bake of Mitsuba's sunsky emitter (ppg_b200/sunsky.py) against the reference's own sky model compiled verbatim
(oracle/_ref/libskymodel_ref.so, built by `make -C oracle skyref` where the original project is present; its outputs stored under tests/golden
otherwise) and against known answers.  The Hosek-Wilkie coefficient tables come from tests/golden/sky_model_rgb.npz (tests/conftest.py)."""
import ctypes as C
import math
import os

import numpy as np

from common import ROOT, load_fixture_scene
from reference_outputs import reference

SKY_REF = os.path.join(ROOT, "oracle", "_ref", "libskymodel_ref.so")
KITCHEN_PROPS = dict(hour="9", turbidity="5", sunRadiusScale="4", scale="50")      # scenes/kitchen/kitchen-improved.xml:2930-2938


def test_sky_model_matches_the_reference_code():
    """arhosek_rgb_skymodelstate_alloc_init + arhosek_tristim_skymodel_radiance (src/emitters/sunsky/skymodel.cpp:329-381) vs the restatement."""
    from ppg_b200 import sunsky
    T = sunsky._sky_tables()
    rng = np.random.default_rng(1)
    args = []
    for k in range(300):
        turb = 10.0 if k == 0 else (float(int(rng.uniform(1, 10))) if k < 20 else rng.uniform(1, 10))
        alb, el = rng.uniform(0, 1), rng.uniform(0, math.pi / 2); th, ga, ch = rng.uniform(0, math.pi / 2 - 1e-3), rng.uniform(0, math.pi), int(rng.integers(3))
        args.append((turb, alb, el, th, ga, ch))
    def live():
        lib = C.CDLL(SKY_REF); lib.skyref_rgb.restype = C.c_double; lib.skyref_rgb.argtypes = [C.c_double] * 5 + [C.c_int]
        return [np.array([lib.skyref_rgb(*a) for a in args])]
    rows, (refs,) = reference("sky_model_rgb", live if os.path.exists(SKY_REF) else None, len(args))
    for k, ref in zip(rows, refs):
        turb, alb, el, th, ga, ch = args[k]
        cfg, rad = sunsky.cook_configuration(T[f"datasetRGB{ch + 1}"], T[f"datasetRGBRad{ch + 1}"], turb, alb, el)
        mine = float(sunsky.sky_radiance_internal(cfg, np.float64(th), np.float64(ga)) * rad)
        assert abs(mine - ref) <= 1e-12 * max(abs(ref), 1e-9), (turb, alb, el, th, ga, ch)


def test_sun_position_known_answers():
    """computeSunCoordinates (sunmodel.h:119-231).  Tokyo, 2010-07-10 (the plugin defaults): at 09:00 JST the sun stands ESE about 51 degrees
    above the horizon, at 15:00 it is in the west; solar noon (about 11:46 JST) is nearly overhead (declination 22.2, latitude 35.7)."""
    from ppg_b200 import sunsky
    el, az = sunsky.sun_coordinates(dict(hour="9"))
    assert abs(math.degrees(el) - 38.48) < 0.05 and abs(math.degrees(az) - 98.85) < 0.05        # zenith angle, azimuth clockwise from north
    el15, az15 = sunsky.sun_coordinates(dict(hour="15"))
    assert 180 < math.degrees(az15) < 300 and 30 < math.degrees(el15) < 50
    eln, azn = sunsky.sun_coordinates(dict(hour="11", minute="46"))
    assert abs(math.degrees(eln) - (35.6894 - 22.2)) < 0.3 and abs(math.degrees(azn) - 180) < 3


def test_kitchen_environment_map_is_the_baked_sunsky():
    """The fixture's environment map is what sunsky.bake produces for kitchen.xml's emitter; physical sanity of the bake: nothing below the
    horizon, the sun texels hold the splatted disc (sunsky.cpp:160-207) and fit half precision (envmap.cpp:102-103), and the integrated sun
    irradiance equals radiance x solid angle of the true disc."""
    from ppg_b200 import sunsky
    img, info = sunsky.bake(KITCHEN_PROPS)
    sc = load_fixture_scene("kitchen-improved")
    assert np.array_equal(img.astype(np.float16).view(np.uint16), sc.envmap["texels"])
    H, W = img.shape[:2]
    assert img[H // 2:].max() == 0 and img[:H // 2].min() > 0 and img.max() < 65504
    # sky alone vs sun + sky: the difference integrates (d omega = sin(theta) d theta d phi) to the sun's irradiance
    sky, _ = sunsky.bake(dict(KITCHEN_PROPS, sunScale="0"))
    theta = (np.arange(H) + 0.5) * math.pi / H
    domega = (np.sin(theta) * (math.pi / H) * (2 * math.pi / W))[:, None, None]
    e_sun = ((img.astype(np.float64) - sky) * domega).sum(axis=(0, 1))
    th = math.radians(sunsky.SUN_APP_RADIUS * 0.5)
    expect = info["sun_radiance"] * 2 * math.pi * (1 - math.cos(th))
    assert np.allclose(e_sun, expect, rtol=0.02), (e_sun, expect)
    assert np.all(np.diff(info["sun_radiance"]) < 0)                                              # a low morning sun is reddish
    assert 11000 < info["n_samples"] < 12000


def test_low_discrepancy_points_of_the_sun_splat():
    """sample02 = (van der Corput, Sobol' 2) (include/mitsuba/core/qmc.h:43-59, 82-87, 115-120)."""
    from ppg_b200 import sunsky
    i = np.arange(8, dtype=np.uint32)
    assert np.allclose(sunsky._radical_inverse2(i), [0, 0.5, 0.25, 0.75, 0.125, 0.625, 0.375, 0.875])
    assert np.allclose(sunsky._sobol2(i), [0, 0.5, 0.75, 0.25, 0.625, 0.125, 0.375, 0.875])      # direction numbers v ^= v >> 1


def test_sky_and_sun_emitters_are_the_two_halves_of_sunsky(tmp_path):
    """The loader bakes <emitter type="sky"> (src/emitters/sky.cpp) and <emitter type="sun"> (src/emitters/sun.cpp:142-225) with the same code as sunsky, which
    nests exactly these two (sunsky.cpp:122-207): their maps add up to the sunsky map, `scale` acts like skyScale / sunScale."""
    from ppg_b200 import scene as S
    body = '<float name="turbidity" value="4"/><float name="hour" value="9"/><float name="latitude" value="48"/><float name="longitude" value="11"/><float name="timezone" value="1"/>'
    def env(typ, extra=""):
        xml = f"""<scene version="0.5.0"><integrator type="guided_path"/>
          <sensor type="perspective"><transform name="toWorld"><lookat origin="0,1,4" target="0,0,0" up="0,1,0"/></transform><film type="hdrfilm"><integer name="width" value="8"/><integer name="height" value="8"/></film></sensor>
          <emitter type="{typ}">{body}{extra}</emitter>
          <shape type="rectangle"><bsdf type="diffuse"/></shape></scene>"""
        p = tmp_path / f"{typ}.xml"; p.write_text(xml)
        return S.load_mitsuba_xml(str(p)).envmap["texels"].view(np.float16).astype(np.float64)
    both, sky, sun = env("sunsky"), env("sky"), env("sun")
    assert sky[sky.shape[0] // 2:].max() == 0 and sky.max() > 0 and (sun > 0).sum() < 0.01 * sun.size and sun.max() > 100 * sky.max()
    assert np.allclose(sky + sun, both, rtol=2e-3, atol=1e-3)                       # (each map is rounded to half precision on its own)
    assert np.allclose(env("sky", '<float name="scale" value="2"/>'), 2 * sky, rtol=2e-3, atol=1e-3)
    assert np.allclose(env("sun", '<float name="scale" value="0.5"/>'), 0.5 * sun, rtol=2e-3, atol=1e-3)
