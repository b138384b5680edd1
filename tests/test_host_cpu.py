"""CPU-side tests: the C-ABI library loads and exports every symbol of include/ppg.h, parameter handling mirrors the
reference constructor, the product path fails loudly without a GPU, and the scene loader reproduces Mitsuba's values."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

from common import ROOT, gpu_available, load_cbox, reference_file
from ppg_b200 import capi, integrator as I


def test_library_exports_every_declared_symbol():
    lib = capi.load_library()
    hdr = open(os.path.join(ROOT, "include", "ppg.h")).read()
    declared = set(re.findall(r"^(?:int|void|const char \*)\s*\*?(ppg_[a-z_0-9]+)\s*\(", hdr, re.M))
    assert declared == set(capi.EXPORTED_SYMBOLS), declared ^ set(capi.EXPORTED_SYMBOLS)
    for s in declared:
        assert hasattr(lib, s), s
    assert lib.ppg_description() == b"Guided path tracer"      # MTS_EXPORT_PLUGIN(GuidedPathTracer, "Guided path tracer"), GP:2422
    assert lib.ppg_abi_version() == 2


def test_struct_layouts_match_header():
    src = '#include "%s"\n#include <stdio.h>\nint main(){printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu", sizeof(ppg_params), sizeof(ppg_bsdf), sizeof(ppg_shape), sizeof(ppg_scene_desc), sizeof(ppg_iteration_stats), sizeof(ppg_stats), sizeof(ppg_sphere));}' % os.path.join(ROOT, "include", "ppg.h")
    import subprocess, tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.run(["/usr/bin/gcc", os.path.join(d, "s.c"), "-o", os.path.join(d, "s")], check=True)
        sizes = [int(x) for x in subprocess.run([os.path.join(d, "s")], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [C.sizeof(capi.PpgParams), C.sizeof(capi.PpgBsdf), C.sizeof(capi.PpgShape), C.sizeof(capi.PpgSceneDesc), C.sizeof(capi.PpgIterationStats), C.sizeof(capi.PpgStats), C.sizeof(capi.PpgSphere)]
    assert C.sizeof(capi.PpgBsdf) == 112 and C.sizeof(capi.PpgSphere) == 24


def test_parameter_defaults_are_the_references():
    p = I.make_params()
    # GP:1015-1084 and integrator.cpp:190-225
    assert (p.nee, p.sample_combination, p.spatial_filter, p.directional_filter, p.bsdf_sampling_fraction_loss) == (0, 1, 0, 0, 0)
    assert (p.sd_tree_max_memory, p.s_tree_threshold, p.spp_per_pass, p.budget_type, p.dump_sd_tree) == (-1, 12000, 4, 1, 0)
    assert (p.d_tree_threshold, p.bsdf_sampling_fraction, p.budget) == (pytest.approx(0.01), 0.5, 300.0)
    assert (p.max_depth, p.rr_depth, p.strict_normals, p.hide_emitters) == (-1, 5, 0, 0)


@pytest.mark.parametrize("name,value", [("sampleCombination", "sometimes"), ("spatialFilter", "gauss"), ("directionalFilter", "stochastic"),
                                        ("bsdfSamplingFractionLoss", "l2"), ("budgetType", "minutes"), ("nee", "sometimes"), ("rrDepth", "0"),
                                        ("maxDepth", "0"), ("maxDepth", "-2"), ("strictNormals", "yes"), ("notAParameter", "1")])
def test_invalid_parameters_are_rejected_like_the_reference(name, value):
    """Unknown enum strings Assert(false) in the reference (GP:1023,1034,1045,1054,1065,1080); rrDepth <= 0 and
    maxDepth not in {-1, >0} Log(EError) (integrator.cpp:220-224)."""
    with pytest.raises(I.PpgError) as e:
        I.make_params({name: value})
    assert e.value.code == -1


def test_all_reference_parameter_strings_are_accepted():
    for name, vals in {"nee": ["never", "kickstart", "always"], "sampleCombination": ["discard", "automatic", "inversevar"], "spatialFilter": ["nearest", "stochastic", "box"],
                       "directionalFilter": ["nearest", "box"], "bsdfSamplingFractionLoss": ["none", "kl", "var"], "budgetType": ["spp", "seconds"]}.items():
        for i, v in enumerate(vals):
            I.make_params({name: v})
    p = I.make_params(load_cbox(improved=True).integrator)
    assert (p.sample_combination, p.bsdf_sampling_fraction_loss, p.spatial_filter, p.directional_filter, p.s_tree_threshold, p.spp_per_pass) == (2, 1, 1, 1, 4000, 1)
    assert (p.max_depth, p.rr_depth, p.strict_normals, p.budget_type, p.budget) == (10, 10, 1, 0, 127.0)


@pytest.mark.skipif(gpu_available(), reason="only meaningful on a box without a GPU")
def test_no_cpu_fallback():
    """The product path must fail loudly without a CUDA device -- it never routes through the oracle or any CPU code."""
    with pytest.raises(I.PpgError) as e:
        I.GuidedPathTracer({})
    assert e.value.code == -2
    with pytest.raises(I.PpgError) as e2:
        I.op_stree_lookup(np.zeros((1, 2), np.uint32), [0, 0, 0], [1, 1, 1], np.zeros((1, 3), np.float32))
    assert e2.value.code == -2


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "practical-path-guiding_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oracle" not in txt.lower() or f == "ppg_device.cuh" and "oracle/ppg_cpu_tracer.h" in txt, os.path.join(dirpath, f)


def test_cbox_rgb_values_match_mitsubas_spectrum_conversion():
    """The CBOX spectra converted by our loader give the RGB triples Mitsuba 0.5 computes (its well-known cbox-rgb values);
    this needs the reference's mirrored InterpolatedSpectrum::eval (spectrum.cpp:701-706), which the loader restates."""
    sc = load_cbox()
    refl = {n: sc.bsdfs[i, 2:5] for i, n in enumerate(sc.bsdf_names)}
    assert np.allclose(refl["white"], [0.885809, 0.698859, 0.666422], atol=2e-4)
    assert np.allclose(refl["red"], [0.570068, 0.0430135, 0.0443706], atol=2e-4)
    assert np.allclose(refl["green"], [0.105421, 0.37798, 0.076425], atol=2e-4)
    assert np.allclose(sc.area_radiance[0], [2 * 18.387, 2 * 10.9873, 2 * 2.75357], rtol=2e-4)
    assert np.allclose(sc.aabb_min, [0, 0, -800]) and np.allclose(sc.aabb_max, [556, 548.8, 559.2])   # geometry + sensor position (scene.cpp:387-413)
    assert len(sc.indices) == 36


def test_fixture_is_what_the_loader_produces_from_the_reference_xml():
    """scenes/cbox.npz is the loader's output for the original project's scenes/cbox/cbox.xml (stored with its meshes under tests/golden/cbox)."""
    from ppg_b200.scene import load_mitsuba_xml
    a = load_mitsuba_xml(os.path.join(ROOT, "tests", "golden", "cbox", "cbox.xml")); b = load_cbox()
    for k in ("positions", "normals", "indices", "triangle_shape", "shapes", "bsdfs", "area_radiance", "cam_to_world", "aabb_min", "aabb_max"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert a.integrator == b.integrator and a.x_fov_deg == b.x_fov_deg


@pytest.mark.skipif(reference_file("scenes", "spaceship", "spaceship-improved.xml") is None, reason="needs the original project's SPACESHIP assets (tests/common.py: reference_dir)")
def test_spaceship_fixture_is_what_the_loader_produces_from_the_reference_xml():
    """spaceship-improved.xml exercises the whole loader: matrix transforms, OBJ meshes with faceNormals, rectangles, a sphere with
    flipNormals, twosided wrappers, roughconductor / roughplastic (reduced transmittance tables) / roughdielectric, named and referenced BSDFs."""
    from ppg_b200.scene import load_mitsuba_xml, SceneDesc
    a = load_mitsuba_xml(reference_file("scenes", "spaceship", "spaceship-improved.xml"))
    b = SceneDesc.load(os.path.join(ROOT, "scenes", "spaceship-improved.npz"))
    for k in ("positions", "normals", "indices", "triangle_shape", "shapes", "bsdfs", "bsdf_tables", "spheres", "area_radiance", "cam_to_world", "aabb_min", "aabb_max"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert len(a.indices) == 457560 and len(a.spheres) == 1 and a.spheres[0, 3] == 100.0
    types = a.bsdfs[:, 0].view(np.uint32)
    assert sorted(set(types.tolist())) == [0, 4, 5, 6]                      # diffuse, roughconductor, roughplastic, roughdielectric
    assert a.integrator["bsdfSamplingFractionLoss"] == "kl" and a.integrator["sppPerPass"] == "1"


def test_rough_transmittance_reduction_has_the_physical_limits():
    """rtrans.py (= RoughTransmittance::setEta/setAlpha/evalDiffuse): at low roughness the table tends to 1 - Fresnel; the diffuse
    internal reflectance matches fresnelDiffuseReflectance(1/eta) (both integrate the same quantity for a smooth interface)."""
    from ppg_b200 import rtrans
    from ppg_b200.scene import fresnel_diffuse_reflectance
    lut, fdr = rtrans.reduce_for_material("beckmann", 1.5, 0.02)
    assert lut.shape == (100,) and lut.dtype == np.float32
    c = ((np.arange(100) / 99.0) ** 4)[70:]                                  # table abscissa is cos(theta)^(1/4); cos > 0.25 (roughness matters at grazing angles)
    ct = np.sqrt(1 - (1 - c * c) / 2.25)
    F = 0.5 * (((c - 1.5 * ct) / (c + 1.5 * ct)) ** 2 + ((1.5 * c - ct) / (1.5 * c + ct)) ** 2)
    assert np.allclose(lut[70:], 1 - F, atol=0.01)
    assert abs(fdr - fresnel_diffuse_reflectance(1 / 1.5)) < 0.01
    lut2, fdr2 = rtrans.reduce_for_material("ggx", 1.5, 0.4)
    assert np.all(np.diff(lut2[10:]) > -1e-3) and 0.5 < fdr2 < 0.65           # transmittance grows towards normal incidence


def test_fresnel_diffuse_reflectance_matches_the_published_fits():
    """src/libcore/util.cpp:822-853 quotes two fits of the same integral with <= 0.1 % error for eta in [1, 2]."""
    from ppg_b200.scene import fresnel_diffuse_reflectance as fdr
    for eta in (1.1, 1.33, 1.5, 1.9):
        ie = 1 / eta
        fit_gt1 = 0.919317 - 3.4793 * ie + 6.75335 * ie ** 2 - 7.80989 * ie ** 3 + 4.98554 * ie ** 4 - 1.36881 * ie ** 5
        fit_lt1 = -1.4399 * ie * ie + 0.7099 * ie + 0.6681 + 0.0636 / ie
        assert abs(fdr(eta) - fit_gt1) < 2e-3 * max(fit_gt1, 0.05) + 2e-4
        assert abs(fdr(ie) - fit_lt1) < 6e-3 * fit_lt1


def test_unsupported_scene_content_is_refused_not_substituted(tmp_path):
    """Content outside the hot-path scope raises instead of being silently replaced (e.g. a textured mask opacity, a constant environment emitter)."""
    from ppg_b200.scene import load_mitsuba_xml
    head = """<scene version="0.5.0"><integrator type="guided_path"/><sensor type="perspective"><film type="hdrfilm"><rfilter type="box"/></film></sensor>"""
    for body in ('<emitter type="constant"/>', '<shape type="cylinder"/>', '<bsdf type="phong" id="x"/>',
                 '<bsdf type="twosided" id="x"><bsdf type="mask"><bsdf type="diffuse"/></bsdf></bsdf>'):
        p = tmp_path / "bad.xml"; p.write_text(head + body + '<shape type="rectangle"/></scene>')
        with pytest.raises(NotImplementedError):
            load_mitsuba_xml(str(p))


@pytest.mark.skipif(reference_file("scenes", "kitchen", "kitchen-improved.xml") is None, reason="needs the original project's KITCHEN assets (tests/common.py: reference_dir)")
def test_kitchen_fixture_is_what_the_loader_produces_from_the_reference_xml():
    """kitchen-improved.xml (BASELINE config 3): 291 OBJ meshes, 13 bitmap textures, the sunsky emitter, bump maps whose nested BSDF carries the id."""
    from ppg_b200.scene import load_mitsuba_xml, SceneDesc, BSDF_FLAG_BUMPMAP
    a = load_mitsuba_xml(reference_file("scenes", "kitchen", "kitchen-improved.xml"))
    b = SceneDesc.load(os.path.join(ROOT, "scenes", "kitchen-improved.npz"))
    for k in ("positions", "normals", "uvs", "indices", "triangle_shape", "shapes", "bsdfs", "bsdf_tables", "area_radiance", "cam_to_world", "aabb_min", "aabb_max", "texels"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert a.textures.tobytes() == b.textures.tobytes() and np.array_equal(a.envmap["texels"], b.envmap["texels"])
    assert len(a.indices) == 1414391 and len(a.textures) == 13 and a.envmap["texels"].shape == (256, 512, 3)
    flags = a.bsdfs[:, 1].view(np.uint32); used = set(a.shapes[:, 2].tolist())
    bumped = [i for i in range(len(flags)) if flags[i] & BSDF_FLAG_BUMPMAP]
    assert len(bumped) == 2 and not (set(bumped) & used)      # <ref id="Cushion1"> resolves to the NESTED twosided BSDF: the bump maps are dead in the reference too
    assert sum(1 for i in used if a.bsdfs[i, 25:26].view(np.uint32)[0]) >= 10     # textured reflectances in use
    assert a.integrator["sampleCombination"] == "inversevar" and a.integrator["sTreeThreshold"] == "4000"


def test_loader_parses_every_supported_bsdf_and_shape(tmp_path):
    """One synthetic Mitsuba XML with every BSDF plugin / wrapper / shape the hot path implements: the loader must fill ppg_bsdf rows
    (type, flags, parameters) and ppg_sphere entries as the C ABI documents them."""
    from ppg_b200 import scene as S
    xml = """<scene version="0.5.0">
      <integrator type="guided_path"><string name="budgetType" value="spp"/><float name="budget" value="8"/><string name="nee" value="always"/></integrator>
      <sensor type="perspective"><float name="fov" value="40"/>
        <transform name="toWorld"><lookat origin="0, 1, -5" target="0, 1, 0" up="0, 1, 0"/></transform>
        <film type="hdrfilm"><integer name="width" value="64"/><integer name="height" value="48"/><rfilter type="box"/></film></sensor>
      <bsdf type="diffuse" id="d"><rgb name="reflectance" value="0.1, 0.2, 0.3"/></bsdf>
      <bsdf type="twosided" id="rc"><bsdf type="roughconductor"><float name="alpha" value="0.2"/><string name="distribution" value="ggx"/>
        <rgb name="eta" value="1.5, 1.0, 0.5"/><rgb name="k" value="3, 2, 1"/><float name="extEta" value="1"/></bsdf></bsdf>
      <bsdf type="dielectric" id="g"><float name="intIOR" value="1.5"/><float name="extIOR" value="1"/></bsdf>
      <bsdf type="thindielectric" id="tg"><float name="intIOR" value="1.33"/><float name="extIOR" value="1"/></bsdf>
      <bsdf type="roughdielectric" id="rg"><float name="alpha" value="0.05"/><string name="distribution" value="beckmann"/><float name="intIOR" value="1.5"/><float name="extIOR" value="1"/></bsdf>
      <bsdf type="plastic" id="p"><rgb name="diffuseReflectance" value="0.5, 0.1, 0.1"/><float name="intIOR" value="1.5"/><float name="extIOR" value="1"/><boolean name="nonlinear" value="true"/></bsdf>
      <bsdf type="mask" id="m"><rgb name="opacity" value="0.6, 0.6, 0.6"/><bsdf type="twosided"><bsdf type="diffuse"><rgb name="reflectance" value="0.6, 0.5, 0.4"/></bsdf></bsdf></bsdf>
      <bsdf type="conductor" id="c"><string name="material" value="none"/></bsdf>
      <bsdf type="bumpmap" id="bm"><texture type="bitmap" name="map"><string name="filename" value="bump.png"/><float name="gamma" value="1.0"/><float name="uscale" value="2"/></texture>
        <bsdf type="twosided" id="inner"><bsdf type="roughplastic"><texture type="bitmap" name="diffuseReflectance"><string name="filename" value="albedo.png"/>
          <string name="wrapModeU" value="clamp"/><string name="wrapModeV" value="mirror"/><float name="voffset" value="0.25"/></texture></bsdf></bsdf></bsdf>
      <emitter type="envmap"><string name="filename" value="env.png"/><float name="scale" value="2"/><transform name="toWorld"><rotate y="1" angle="90"/></transform></emitter>
      <shape type="rectangle"><ref id="bm"/></shape>
      <shape type="rectangle"><ref id="inner"/></shape>
      <shape type="rectangle"><transform name="toWorld"><scale x="2" y="2"/><translate x="0" y="3" z="0"/></transform><ref id="d"/>
        <emitter type="area"><rgb name="radiance" value="5, 5, 5"/></emitter></shape>
      <shape type="rectangle"><ref id="m"/></shape>
      <shape type="sphere"><point name="center" x="1" y="1" z="0"/><float name="radius" value="0.5"/><ref id="g"/></shape>
      <shape type="sphere"><boolean name="flipNormals" value="true"/><transform name="toWorld"><scale value="50"/></transform>
        <emitter type="area"><rgb name="radiance" value="0.1, 0.1, 0.1"/></emitter></shape>
    </scene>"""
    import cv2
    rng = np.random.default_rng(3)
    albedo = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8); cv2.imwrite(str(tmp_path / "albedo.png"), albedo[..., ::-1])
    cv2.imwrite(str(tmp_path / "bump.png"), rng.integers(0, 256, (4, 4), dtype=np.uint8)); cv2.imwrite(str(tmp_path / "env.png"), rng.integers(1, 256, (4, 8, 3), dtype=np.uint8))
    p = tmp_path / "scene.xml"; p.write_text(xml)      # nee = always: the lamp, the emitting shell and the environment map are all light-sampled
    sc = S.load_mitsuba_xml(str(p))
    # textures: sRGB-decoded (gamma 0) vs linear (gamma 1), half precision, wrap modes / uv transform in ppg_texture
    assert len(sc.textures) == 2 and sc.texels.dtype == np.uint16
    t_alb = sc.textures[[int(t["channels"]) for t in sc.textures].index(3)]; t_bmp = sc.textures[[int(t["channels"]) for t in sc.textures].index(1)]
    assert (int(t_alb["width"]), int(t_alb["height"]), int(t_alb["wrap_u"]), int(t_alb["wrap_v"])) == (7, 5, 1, 2) and np.allclose(t_alb["uv_offset"], [0, 0.25])
    v = albedo.astype(np.float64) / 255; lin = np.where(v <= 0.04045, v / 12.92, ((v + 0.055) / 1.055) ** 2.4)
    got = sc.texels[int(t_alb["first_texel"]):int(t_alb["first_texel"]) + 105].view(np.float16).astype(np.float64).reshape(5, 7, 3)
    assert np.allclose(got, lin, rtol=2e-3, atol=1e-4)
    assert np.allclose(t_bmp["uv_scale"], [2, 1]) and int(t_bmp["width"]) == 4
    bm, inner = sc.bsdf_names.index("bm"), sc.bsdf_names.index("inner")
    fb, fi = int(sc.bsdfs[bm, 1:2].view(np.uint32)[0]), int(sc.bsdfs[inner, 1:2].view(np.uint32)[0])
    assert fb == (S.BSDF_FLAG_BUMPMAP | S.BSDF_FLAG_TWOSIDED) and fi == S.BSDF_FLAG_TWOSIDED                 # the nested id is registered without the bump map
    assert sc.bsdfs[bm, 25:27].view(np.uint32).tolist() == [1 + list(sc.textures).index(t_alb), 1 + list(sc.textures).index(t_bmp)] and sc.bsdfs[inner, 26:27].view(np.uint32)[0] == 0
    assert np.allclose(sc.bsdfs[bm, 2:5], lin.reshape(-1, 3).mean(0), rtol=1e-3)                              # constant slot = texture average (feeds specularSamplingWeight)
    assert sc.envmap["texels"].shape == (4, 8, 3) and sc.envmap["scale"] == 2.0 and np.allclose(sc.envmap["world_to_env"] @ np.array([1.0, 0, 0]), [0, 0, 1], atol=1e-6)
    sc.save(str(tmp_path / "rt.npz")); rt = S.SceneDesc.load(str(tmp_path / "rt.npz"))                       # npz round trip keeps textures and the environment map
    assert rt.textures.tobytes() == sc.textures.tobytes() and np.array_equal(rt.texels, sc.texels) and np.array_equal(rt.envmap["texels"], sc.envmap["texels"])
    row = {n: sc.bsdfs[i] for i, n in enumerate(sc.bsdf_names)}
    ty = lambda n: int(row[n][:1].view(np.uint32)[0]); fl = lambda n: int(row[n][1:2].view(np.uint32)[0])
    assert sc.bsdfs.shape[1] == 28
    assert (ty("d"), ty("rc"), ty("g"), ty("tg"), ty("rg"), ty("p"), ty("m"), ty("c")) == (0, 4, 2, 8, 6, 7, 0, 3)
    assert fl("rc") == S.BSDF_FLAG_TWOSIDED and fl("m") == (S.BSDF_FLAG_MASK | S.BSDF_FLAG_TWOSIDED) and fl("p") == S.BSDF_FLAG_NONLINEAR
    assert np.allclose(row["m"][22:25], 0.6) and np.allclose(row["m"][2:5], [0.6, 0.5, 0.4])
    assert np.allclose(row["rc"][8:11], [1.5, 1.0, 0.5]) and np.allclose(row["rc"][11:14], [3, 2, 1]) and np.isclose(row["rc"][14], 0.2) and int(row["rc"][15:16].view(np.int32)[0]) == 1
    assert np.isclose(row["rg"][14], 0.05) and int(row["rg"][15:16].view(np.int32)[0]) == 0 and np.isclose(row["tg"][8], 1.33)
    assert np.isclose(row["p"][19], S.fresnel_diffuse_reflectance(1 / 1.5)) and 0 < row["p"][20] < 1
    assert len(sc.indices) == 8 and sc.spheres.shape == (2, 6)
    assert np.allclose(sc.spheres[0, :4], [1, 1, 0, 0.5]) and np.allclose(sc.spheres[1, :4], [0, 0, 0, 50])
    assert sc.spheres[:, 5].view(np.int32).tolist() == [0, 1]                    # flipNormals
    assert sc.spheres[:, 4].view(np.int32).tolist() == [4, 5] and sc.shapes[5, 3] == 1 and sc.shapes[2, 3] == 0     # shape / emitter indices
    assert np.allclose(sc.aabb_min, -50) and np.allclose(sc.aabb_max, 50)
    assert (sc.film_width, sc.film_height) == (64, 48)
    # and the oracle renders it (all models on one path: light sampling of the three emitters through the mask, the glass sphere, the shell)
    import oracle_lib as O
    o = O.Oracle(O.params_from_xml(sc.integrator), sc, kind="port"); img, st = o.render()
    assert img.shape == (48, 64, 3) and np.isfinite(img).all() and img.mean() > 0.01 and st["total_paths"] == 64 * 48 * 8


def test_flat_scene_file_round_trip(tmp_path):
    """python -m ppg_b200.convert -> ppg_scene_file_load (the route of the Mitsuba plugin shim, integration/guided_path_b200.cpp): every array of the
    scene description comes back bit for bit, textures and the environment map included; no CUDA device is involved."""
    from common import load_fixture_scene
    sc = load_fixture_scene("cbox-textured")
    path = str(tmp_path / "scene.ppgscene")
    sc.save_flat(path)
    lib = capi.load_library()
    d = capi.PpgSceneDesc(); fh = C.c_void_p(); props = C.c_char_p()
    assert lib.ppg_scene_file_load(path.encode(), C.byref(d), C.byref(fh), C.byref(props)) == 0, lib.ppg_last_error()
    ref = capi.SceneArrays(sc).desc
    assert (d.n_vertices, d.n_triangles, d.n_shapes, d.n_bsdfs, d.n_emitters, d.n_textures, d.n_texels) == (ref.n_vertices, ref.n_triangles, ref.n_shapes, ref.n_bsdfs, ref.n_emitters, ref.n_textures, ref.n_texels)
    as_np = lambda ptr, n, t: np.ctypeslib.as_array(C.cast(ptr, C.POINTER(t)), shape=(n,)).copy()
    assert np.array_equal(as_np(d.positions, 3 * d.n_vertices, C.c_float), sc.positions.reshape(-1)) and np.array_equal(as_np(d.indices, 3 * d.n_triangles, C.c_uint32), sc.indices.reshape(-1))
    assert np.array_equal(as_np(d.bsdfs, 28 * d.n_bsdfs, C.c_float).view(np.uint32), np.asarray(sc.bsdfs, np.float32).reshape(-1).view(np.uint32))
    assert np.array_equal(as_np(d.texels, d.n_texels, C.c_uint16), sc.texels) and bytes(as_np(d.textures, 48 * d.n_textures, C.c_uint8)) == sc.textures.tobytes()
    assert (d.envmap.width, d.envmap.height) == (32, 16) and np.array_equal(as_np(d.envmap.texels, 32 * 16 * 3, C.c_uint16), sc.envmap["texels"].reshape(-1))
    assert np.isclose(d.envmap.scale, 1.5) and np.allclose(list(d.envmap.world_to_env), np.asarray(sc.envmap["world_to_env"]).reshape(-1))
    assert (d.camera.film_width, d.camera.film_height) == (sc.film_width, sc.film_height) and np.isclose(d.camera.x_fov_deg, sc.x_fov_deg)
    assert dict(l.split("=", 1) for l in props.value.decode().splitlines()) == sc.integrator
    lib.ppg_scene_file_free(fh)
    assert lib.ppg_scene_file_load(str(tmp_path / "missing").encode(), C.byref(d), C.byref(fh), None) == -7      # PPG_ERR_IO


def test_bvh_build_is_valid_and_independent_of_the_thread_count():
    """ppg_op_bvh_build (host only): the binned-SAH BVH ppg_set_scene builds over SPACESHIP's 457 560 triangles.  Every triangle sits in exactly one
    leaf, leaves hold at most 4 triangles, children lie inside their parents, the boxes are tight -- and the arrays are byte-identical for 1, 3 and 8
    host threads and equal to the layout of the serial builder the GPU parity runs of round 2 were made with (pinned by hash), so parallelising the
    host set-up cannot move a single hit."""
    import hashlib
    from ppg_b200.integrator import op_bvh_build
    from ppg_b200.scene import SceneDesc
    sc = SceneDesc.load(os.path.join(ROOT, "scenes", "spaceship-improved.npz"))
    nodes, order, depth, ms = op_bvh_build(sc.positions, sc.indices, 1)
    for threads in (3, 8):
        n2, o2, d2, _ = op_bvh_build(sc.positions, sc.indices, threads)
        assert d2 == depth and n2.tobytes() == nodes.tobytes() and o2.tobytes() == order.tobytes()
    assert hashlib.sha256(nodes.tobytes() + order.tobytes()).hexdigest().startswith("e459259d0c4e618a")
    assert (len(nodes), depth) == (454573, 29) and depth < 64                       # PPG_BVH_STACK
    assert np.array_equal(np.sort(order), np.arange(len(sc.indices), dtype=np.uint32))
    left = nodes[:, 3].copy().view(np.uint32); count = nodes[:, 7].copy().view(np.uint32)
    inner = count == 0
    assert count[~inner].max() <= 4 and count[~inner].sum() == len(sc.indices)
    # children inside the parent; every node but the root is the child of exactly one inner node
    kids = np.concatenate([left[inner], left[inner] + 1]); par = np.concatenate([np.nonzero(inner)[0]] * 2)
    assert np.array_equal(np.sort(kids), np.arange(1, len(nodes)))
    assert (nodes[kids, 0:3] >= nodes[par, 0:3]).all() and (nodes[kids, 4:7] <= nodes[par, 4:7]).all()
    # leaf boxes are the bounds of their triangles
    tri = sc.positions[sc.indices]                                                   # (T, 3, 3)
    tmin, tmax = tri.min(axis=1), tri.max(axis=1)
    leaves = np.nonzero(~inner)[0][:20000]
    for i in leaves[::97]:
        t = order[left[i]:left[i] + count[i]]
        assert np.array_equal(nodes[i, 0:3], tmin[t].min(axis=0)) and np.array_equal(nodes[i, 4:7], tmax[t].max(axis=0))
    assert np.array_equal(nodes[0, 0:3], tmin.min(axis=0)) and np.array_equal(nodes[0, 4:7], tmax.max(axis=0))


def test_plain_c_host_builds_and_fails_loudly_without_a_device(tmp_path):
    """integration/ppg_render_cli.c: a C99 host over include/ppg.h alone (-Wall -Wextra -pedantic clean).  Without a CUDA device it loads a flat scene
    file, applies the XML's integrator block and -D overrides through ppg_params_set (the plugin constructor's validation and messages), and then fails
    with PPG_ERR_NO_DEVICE -- no CPU fallback behind the C ABI either."""
    import subprocess
    from ppg_b200.scene import SceneDesc
    mk = subprocess.run(["make", "-C", os.path.join(ROOT, "integration")], capture_output=True, text=True)
    assert mk.returncode == 0 and "warning" not in (mk.stdout + mk.stderr).lower(), mk.stdout + mk.stderr
    cli = os.path.join(ROOT, "integration", "ppg_render_cli")
    scene = str(tmp_path / "cbox.ppgscene")
    SceneDesc.load(os.path.join(ROOT, "scenes", "cbox-improved.npz")).with_film(48, 32).save_flat(scene)
    r = subprocess.run([cli, scene, "--check", "-D", "budget=28", "-D", "nee=kickstart"], capture_output=True, text=True)
    assert r.returncode == 0 and "36 triangles" in r.stderr and "film 48 x 32" in r.stderr and "check ok" in r.stderr, r.stderr
    r = subprocess.run([cli, scene, "--check", "-D", "spatialFilter=gaussian"], capture_output=True, text=True)
    assert r.returncode == 1 and "spatialFilter" in r.stderr                           # PPG_ERR_INVALID_ARGUMENT, the reference Assert(false)s (GP:1045)
    r = subprocess.run([cli, str(tmp_path / "missing.ppgscene"), "--check"], capture_output=True, text=True)
    assert r.returncode == 7                                                            # PPG_ERR_IO
    import ctypes
    try:
        ctypes.CDLL("libcuda.so.1"); have_driver = True
    except OSError:
        have_driver = False
    if not have_driver or not __import__("common").gpu_available():
        r = subprocess.run([cli, scene, str(tmp_path / "out.pfm")], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU fallback" in r.stderr and not os.path.exists(tmp_path / "out.pfm"), r.stderr


def test_corrupt_scene_files_are_rejected_not_trusted(tmp_path):
    """ppg_scene_file_load on damaged input: truncated anywhere, dimension fields overwritten with huge or inconsistent values, arrays whose sizes do not
    match each other -- always PPG_ERR_IO with a message, never a crash, an unbounded allocation or a description that would make ppg_set_scene read out of bounds."""
    from common import load_fixture_scene
    sc = load_fixture_scene("cbox-textured")
    good = str(tmp_path / "good.ppgscene"); sc.save_flat(good)
    raw = open(good, "rb").read()
    lib = capi.load_library()

    def load(data):
        p = str(tmp_path / "t.ppgscene"); open(p, "wb").write(data)
        d = capi.PpgSceneDesc(); fh = C.c_void_p()
        rc = lib.ppg_scene_file_load(p.encode(), C.byref(d), C.byref(fh), None)
        if rc == 0:
            lib.ppg_scene_file_free(fh)
        return rc

    assert load(raw) == 0
    rng = np.random.default_rng(5)
    for cut in [0, 4, 8, 9, 20] + list(rng.integers(21, len(raw) - 1, 40)):
        assert load(raw[:int(cut)]) == -7, cut                                      # (a cut exactly between two arrays drops required arrays: also an error)
    # the first array is "positions": [u32 6]["positi..."][u32 dtype][u32 ndim][u64 dim0][u64 dim1]: blow up its first dimension
    off = 8 + 4 + len("positions") + 8
    assert raw[12:21] == b"positions"
    for dim in (2 ** 62, 2 ** 40, len(raw), sc.positions.shape[0] - 1, sc.positions.shape[0] + 1):
        bad = bytearray(raw); bad[off:off + 8] = int(dim).to_bytes(8, "little")
        assert load(bytes(bad)) == -7, dim
    assert b"array" in lib.ppg_last_error() or b"corrupt" in lib.ppg_last_error() or b"truncated" in lib.ppg_last_error() or b"lacks" in lib.ppg_last_error()
    bad = bytearray(raw); bad[:8] = b"PPGSCN01"
    assert load(bytes(bad)) == -7
    # a file whose normals array is shorter than its positions (consistent in itself, inconsistent as a scene)
    import copy
    sc2 = copy.copy(sc); sc2.normals = sc.normals[:-1]
    p2 = str(tmp_path / "short_normals.ppgscene"); sc2.save_flat(p2)
    assert load(open(p2, "rb").read()) == -7 and b"do not match" in lib.ppg_last_error()


def _scene_xml(shapes):
    return f"""<scene version="0.5.0"><integrator type="guided_path"><string name="budgetType" value="spp"/><float name="budget" value="4"/></integrator>
      <sensor type="perspective"><float name="fov" value="45"/><transform name="toWorld"><lookat origin="0,1,6" target="0,0,0" up="0,1,0"/></transform>
        <film type="hdrfilm"><integer name="width" value="32"/><integer name="height" value="24"/></film></sensor>
      <shape type="rectangle"><transform name="toWorld"><rotate x="1" angle="90"/><scale value="0.5"/><translate y="3"/></transform>
        <emitter type="area"><rgb name="radiance" value="10,10,10"/></emitter></shape>
      {shapes}</scene>"""


def test_loader_reads_ply_meshes(tmp_path):
    """<shape type="ply"> as src/shapes/ply.cpp reads it: binary little / big endian and ascii, triangles and quads (a quad (a,b,c,d) -> (a,b,c), (d,a,c)),
    normals and texture coordinates when the file has them, angle-weighted normals when it does not; toWorld applied like every mesh."""
    import struct
    from ppg_b200 import scene as S
    rng = np.random.default_rng(4)
    V = rng.normal(size=(7, 3)).astype(np.float32); Nn = rng.normal(size=(7, 3)).astype(np.float32); UV = rng.random((7, 2)).astype(np.float32)
    faces = [[0, 1, 2], [2, 3, 4, 5], [4, 5, 6]]
    hdr = lambda fmt: (f"ply\nformat {fmt} 1.0\ncomment test\nelement vertex 7\nproperty float x\nproperty float y\nproperty float z\nproperty float nx\nproperty float ny\n"
                       "property float nz\nproperty float s\nproperty float t\nproperty uchar red\nelement face 3\nproperty list uchar int vertex_indices\nend_header\n").encode()
    def binary(end):
        b = hdr("binary_little_endian" if end == "<" else "binary_big_endian")
        for i in range(7):
            b += struct.pack(end + "8fB", *V[i], *Nn[i], *UV[i], 200)
        for f in faces:
            b += struct.pack(end + "B%di" % len(f), len(f), *f)
        return b
    ascii_ = hdr("ascii") + "".join(" ".join(repr(float(x)) for x in (*V[i], *Nn[i], *UV[i])) + " 200\n" for i in range(7)).encode() + \
        "".join(f"{len(f)} " + " ".join(map(str, f)) + "\n" for f in faces).encode()
    M = np.eye(4); M[:3, :3] = np.diag([2.0, 1.0, 0.5]); M[:3, 3] = [1, 2, 3]
    out = []
    for name, blob in (("le.ply", binary("<")), ("be.ply", binary(">")), ("a.ply", ascii_)):
        (tmp_path / name).write_bytes(blob)
        out.append(S._load_ply(str(tmp_path / name), M))
    for P, N, uv, I in out:
        assert np.allclose(P, V * [2, 1, 0.5] + [1, 2, 3], atol=1e-6) and np.allclose(uv, UV, atol=1e-6)
        nw = Nn / [2, 1, 0.5]; nw /= np.linalg.norm(nw, axis=1, keepdims=True)
        assert np.allclose(N, nw, atol=1e-6)                                       # normals: inverse transpose, normalised
        assert I.tolist() == [[0, 1, 2], [2, 3, 4], [5, 2, 4], [4, 5, 6]]
    # through the XML: face normals + flipNormals swap the winding, no vertex normals are kept
    (tmp_path / "m.xml").write_text(_scene_xml('<shape type="ply"><string name="filename" value="le.ply"/><boolean name="faceNormals" value="true"/><boolean name="flipNormals" value="true"/><bsdf type="diffuse"/></shape>'))
    sc = S.load_mitsuba_xml(str(tmp_path / "m.xml"))
    assert sc.shapes[1, 1] == 4 and sc.shapes[1, 4] == 0 and sc.indices[2:].tolist() == (np.array([[1, 0, 2], [3, 2, 4], [2, 5, 4], [5, 4, 6]]) + 4).tolist()
    bunny = reference_file("mitsuba", "data", "tests", "bunny.ply")                # the mesh of the reference's test_kd.cpp
    if bunny is not None:
        P, N, uv, I = S._load_ply(bunny, np.eye(4))
        assert P.shape == (35947, 3) and I.shape == (69451, 3) and uv is None and np.allclose(np.linalg.norm(N, axis=1), 1, atol=1e-4)
        ctr = P.mean(0); tri = P[I]; fn = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
        assert ((fn * (tri.mean(1) - ctr)).sum(1) > 0).mean() > 0.8                  # outward winding, and the smooth normals follow it
        assert ((N[I[:, 0]] * fn).sum(1) > 0).mean() > 0.99


def test_loader_reads_serialized_meshes_and_cubes(tmp_path):
    """<shape type="serialized"> (TriMesh::loadCompressed, trimesh.cpp:176-250): header, zlib stream, flags (normals / texcoords / colours / face normals /
    double precision), versions 3 and 4, several meshes behind the offset table at the end of the file; and <shape type="cube"> (shapes/cube.cpp)."""
    import struct
    import zlib
    from ppg_b200 import scene as S
    rng = np.random.default_rng(6)
    def mesh(nv, nt, flags, ver):
        P = rng.normal(size=(nv, 3)); N = rng.normal(size=(nv, 3)); UV = rng.random((nv, 2)); C = rng.random((nv, 3)); I = rng.integers(0, nv, (nt, 3)).astype("<u4")
        ft = "<f8" if flags & 0x2000 else "<f4"
        body = struct.pack("<I", flags) + (b"name\0" if ver == 4 else b"") + struct.pack("<QQ", nv, nt) + P.astype(ft).tobytes()
        if flags & 1: body += N.astype(ft).tobytes()
        if flags & 2: body += UV.astype(ft).tobytes()
        if flags & 8: body += C.astype(ft).tobytes()
        body += I.tobytes()
        return struct.pack("<HH", 0x041C, ver) + zlib.compress(body), (P.astype(ft), N.astype(ft), UV.astype(ft), I)
    for ver in (3, 4):
        blobs = [mesh(5, 3, 0x0001 | 0x0002 | 0x0008, ver), mesh(9, 6, 0x2000 | 0x0001, ver), mesh(4, 2, 0x0010 | 0x0002, ver)]
        offs = np.cumsum([0] + [len(b[0]) for b in blobs[:-1]])
        table = b"".join(struct.pack("<Q" if ver == 4 else "<I", int(o)) for o in offs) + struct.pack("<I", len(blobs))
        path = tmp_path / f"v{ver}.serialized"; path.write_bytes(b"".join(b[0] for b in blobs) + table)
        M = np.eye(4); M[:3, 3] = [0.5, -1, 2]
        for k, (_, (P, N, UV, I)) in enumerate(blobs):
            p, n, uv, i = S._load_serialized(str(path), k, M)
            assert np.allclose(p, P + [0.5, -1, 2], atol=1e-6) and np.array_equal(i, I)
            if k == 2:
                assert n is None and np.allclose(uv, UV, atol=1e-6)                # EFaceNormals
            else:
                assert np.allclose(n, N / np.linalg.norm(N, axis=1, keepdims=True), atol=1e-6) and ((uv is None) == (k == 1))
        with pytest.raises(ValueError):
            S._load_serialized(str(path), 3, M)
    (tmp_path / "bad.serialized").write_bytes(b"\x04\x1c\x04\x00garbage")
    with pytest.raises(ValueError):
        S._load_serialized(str(tmp_path / "bad.serialized"), 0, np.eye(4))
    # cube: [-1,1]^3 under toWorld, outward normals, per-face texture coordinates; rendered by the oracle like any mesh
    (tmp_path / "c.xml").write_text(_scene_xml('<shape type="cube"><transform name="toWorld"><scale x="1" y="0.5" z="2"/><translate y="-1"/></transform><bsdf type="diffuse"/></shape>'
                                               '<shape type="serialized"><string name="filename" value="v4.serialized"/><integer name="shapeIndex" value="1"/><bsdf type="diffuse"/></shape>'))
    sc = S.load_mitsuba_xml(str(tmp_path / "c.xml"))
    f, n = int(sc.shapes[1, 0]), int(sc.shapes[1, 1])
    assert n == 12 and sc.shapes[1, 4] == 1 and sc.shapes[1, 5] == 1 and sc.shapes[2, 1] == 6
    tri = sc.positions[sc.indices[f:f + n]]
    assert np.allclose(tri.reshape(-1, 3).min(0), [-1, -1.5, -2]) and np.allclose(tri.reshape(-1, 3).max(0), [1, -0.5, 2])
    fn = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]); ctr = np.array([0, -1.0, 0])
    assert ((fn * (tri.mean(1) - ctr)).sum(1) > 0).all()                               # counter-clockwise seen from outside
    assert ((sc.normals[sc.indices[f:f + n, 0]] * fn).sum(1) > 0).all()
    assert set(map(tuple, sc.uvs[np.unique(sc.indices[f:f + n])].tolist())) == {(0.0, 0.0), (0.0, 1.0), (1.0, 0.0), (1.0, 1.0)}
    import oracle_lib as O
    (tmp_path / "only_cube.xml").write_text(_scene_xml('<shape type="cube"><transform name="toWorld"><scale x="1" y="0.5" z="2"/><translate y="-1"/></transform><bsdf type="diffuse"/></shape>'))
    sc = S.load_mitsuba_xml(str(tmp_path / "only_cube.xml"))
    img, st = O.Oracle(O.params_from_xml(sc.integrator), sc, kind="port").render()
    assert np.isfinite(img).all() and img.mean() > 1e-3


def test_python_command_line_host(tmp_path):
    """python -m ppg_b200 scene -o out [-D name=value]: the reference's `mitsuba -D ... -o ... scene.xml` for this integrator.  On the CPU: scene + parameter
    handling (--check), the plugin constructor's error for a bad enum value, the loud failure without a device, and the three film writers."""
    import subprocess
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "practical-path-guiding_b200"))
    run = lambda *a: subprocess.run([sys.executable, "-m", "ppg_b200", *a], capture_output=True, text=True, env=env)
    scene = os.path.join(ROOT, "scenes", "cbox-improved.npz")
    r = run(scene, "--check", "-D", "budget=28", "--size", "40", "30")
    assert r.returncode == 0 and "film 40 x 30" in r.stderr and "check ok" in r.stderr, r.stderr
    r = run(scene, "--check", "-D", "sampleCombination=median")
    assert r.returncode == 1 and "sampleCombination" in r.stderr
    if not __import__("common").gpu_available():
        r = run(scene, "-o", str(tmp_path / "o.pfm"))
        assert r.returncode == 2 and "no CPU fallback" in r.stderr and not os.path.exists(tmp_path / "o.pfm")
    from ppg_b200.__main__ import write_image
    img = np.random.default_rng(0).random((5, 7, 3)).astype(np.float32)
    for ext in ("exr", "pfm", "npy"):
        write_image(str(tmp_path / f"w.{ext}"), img)
    os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")
    import cv2
    assert np.array_equal(cv2.imread(str(tmp_path / "w.exr"), cv2.IMREAD_UNCHANGED)[..., ::-1], img) and np.array_equal(np.load(tmp_path / "w.npy"), img)
    raw = open(tmp_path / "w.pfm", "rb").read()
    assert raw.startswith(b"PF\n7 5\n-1.0\n") and np.array_equal(np.frombuffer(raw[12:], "<f4").reshape(5, 7, 3)[::-1], img)
