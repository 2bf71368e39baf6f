"""Parity of the device path tracer (SURVEY 8(f) N3: etxb_set_integrator(ETXB_INTEGRATOR_PT), kernels_pt.cuh / dpt.cuh) against the
oracle = the reference's run_path_iteration (rt/shared/path_tracing_shared.hxx:485-510) compiled in place + the restated CPUPathTracing
driver and Film members (oracle/oracle_vcm.cxx: run_pt_iteration).  Run with -m gpu.

parity flavor: camera image, normal / albedo / adaptive layers, per-path radiance, end-of-path sampler states and the per-pixel history
(sample count, converged, tmp) are BIT-EXACT.  Product flavor: converged statistical test (relMSE against the oracle's run-to-run floor) —
its transcendentals / division are approximate and, in opaque scenes with stochastic BSDFs, its shadow segments go through k_shadow_resolve.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, Digest, bit_equal, golden, rel_l2, same_bits
from etx_tracer_b200 import scenes, structs as S

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from etx_tracer_b200 import api as m
    return m


LAYERS = (S.FILM_CAMERA, S.FILM_NORMALS, S.FILM_ALBEDO, S.FILM_CAMERA_ADAPTIVE, S.FILM_RESULT)


def _oracle(oracle_mod, sd, iterations, options=None, settings=None, flavor="parity", threads=1, first=0):
    o = oracle_mod.Oracle(sd, flavor)
    o.set_integrator(S.INTEGRATOR_PT)
    opts = S.default_pt_options()
    for k, v in (options or {}).items():
        opts[k] = v
    o.pt_set_options(opts)
    if settings is not None:
        o.set_scene_settings(*settings)
    o.begin(first)
    o.run(iterations, threads=threads)
    return o


def _device(api, sd, iterations, options=None, settings=None, flavor="parity", first=0):
    g = api.GPUPathTracing(sd, flavor=flavor)
    for k, v in (options or {}).items():
        g.pt_options[k] = v
    if settings is not None:
        g.set_scene_settings(*settings)
    st = g.render(iterations, first_iteration=first)
    assert st["completed_iterations"] == iterations and st["overflow"] == 0
    return g


PT_BUFFERS = ((S.BUF_CAMERA_SAMPLER, np.uint32), (S.BUF_CAMERA_GATHERED, np.float32), (S.BUF_PIXEL_INFO, np.uint32))


def _outputs(x, sd):
    """What the parity tests compare, of a device context or an oracle: the counters come as a dict from the one, a record from the other."""
    out = {f"buffer {bid}": x.buffer(bid, dt) for bid, dt in PT_BUFFERS}
    out.update({f"film layer {layer}": x.film(layer)[..., :3] for layer in LAYERS})
    out["pixels_processed"] = x.pt_status()["pixels_processed"]
    c = x.counters()
    # one shaded event per run_path_iteration call that got past the length test; closest-hit queries likewise unless a subsurface walk adds its own
    out["bounces_camera"] = int(np.asarray(c["bounces_camera"]).reshape(-1)[0])
    if int(sd.scene["subsurface_scatter_material"][0]) == S.INVALID:
        out["rays_closest"] = int(np.asarray(c["rays_closest"]).reshape(-1)[0])
    return out


def _assert_bit_exact(got, ref, what=""):
    assert sorted(got) == sorted(ref), what
    for k in ref:
        a, b = got[k], ref[k]
        if isinstance(b, Digest):
            assert same_bits(a, b), f"{what} {k} differs from the oracle's"
            continue
        a, b = np.asarray(a), np.asarray(b)
        assert a.shape == b.shape, f"{what} {k}: {a.shape} vs {b.shape}"
        same = a.view(np.uint32) == b.view(np.uint32) if a.dtype.itemsize == 4 else a == b
        assert same.all(), f"{what} {k}: {100.0 * same.mean():.3f}% identical, first mismatch at {int(np.argmin(same))}"


def _compare(api, oracle_record, sd, iterations, options=None, settings=None, what=""):
    ref = oracle_record(what, lambda m: _outputs(_oracle(m, sd, iterations, options, settings), sd))
    g = _device(api, sd, iterations, options, settings)
    _assert_bit_exact(_outputs(g, sd), ref, what)
    g.close()


C1 = dict(samples=16, spectral=False)
C2 = dict(samples=256, spectral=True, sphere=True)


def test_path_tracer_matches_committed_golden_render(api):
    """tests/golden/oracle_pt_c2_32.npz (tools/make_golden.py): the fixture travels to the GPU box, the reference does not."""
    ref = golden("oracle_pt_c2_32.npz")
    g = _device(api, scenes.cornell_box(32, 32, **C2), int(ref["iterations"][0]))
    assert bit_equal(g.buffer(S.BUF_CAMERA_SAMPLER, np.uint32), ref["camera_sampler"])
    assert bit_equal(g.film(S.FILM_CAMERA)[..., :3], ref["film_camera"][..., :3])
    assert bit_equal(g.film(S.FILM_NORMALS)[..., :3], ref["film_normals"][..., :3])
    assert bit_equal(g.film(S.FILM_ALBEDO)[..., :3], ref["film_albedo"][..., :3])
    assert g.lib.etxb_build_flavor().decode() == "parity" and g.counters()["kernel_launches"] > 0
    g.close()


@pytest.mark.parametrize("kwargs,options,settings", [
    (C1, None, None), (C2, None, None),
    (C1, dict(nee=0), None),                   # BSDF sampling + direct hits only
    (C2, dict(mis=0, blue_noise=0), None),     # no MIS, Sampler-only randoms at the first vertex
    (C1, dict(direct=0), None),                # light sampling only
    (C2, None, (0.0, 0.5)),                    # radiance clamp (path_tracing.cxx:73-78)
])
def test_iterations_are_bit_exact_against_live_oracle(api, oracle_record, kwargs, options, settings):
    sd = scenes.cornell_box(48, 40, **kwargs)  # non-square film exercises the y-flip and aspect handling
    _compare(api, oracle_record, sd, 3, options, settings, what=f"{kwargs} {options} {settings}")


def test_running_mean_and_first_iteration_offset(api):
    """Film::accumulate_camera_image (film.cxx:173-230): two iterations = lerp(second, first, 1/2) exactly; the colour of an iteration depends on
    (pixel, iteration index) only; the first iteration of a run (index 0) uses the empty pixel filter (path_tracing_shared.hxx:245)."""
    sd = scenes.cornell_box(40, 40, **C1)
    g = _device(api, sd, 1)
    a0 = g.film(S.FILM_CAMERA)[..., :3].copy()
    g.render(1, first_iteration=1)
    a1 = g.film(S.FILM_CAMERA)[..., :3].copy()
    g.render(2)
    both = g.film(S.FILM_CAMERA)[..., :3]
    assert bit_equal(both, (a1 * np.float32(0.5) + a0 * np.float32(0.5)).astype(np.float32))
    info = g.buffer(S.BUF_PIXEL_INFO, np.uint32)
    assert (info == 2).all()
    nrm = g.film(S.FILM_NORMALS)[..., :3]
    assert (nrm >= 0.0).all() and (nrm <= 1.0).all()
    g.close()


@pytest.mark.parametrize("spectral", [False, True])
@pytest.mark.parametrize("kind", sorted(scenes.MATERIAL_KINDS))
def test_every_material_class_is_bit_exact(api, oracle_record, kind, spectral):
    """bsdf::sample / evaluate / albedo of every Material::Class through handle_hit_ray and evaluate_light (path_tracing_shared.hxx:300-460);
    the subsurface kinds go through subsurface::gather and the per-exit emitter samples (:408-414)."""
    _compare(api, oracle_record, scenes.material_box(kind, 32, 32, spectral=spectral), 2, what=kind)


@pytest.mark.parametrize("spectral", [False, True])
@pytest.mark.parametrize("variant", [dict(), dict(sun=False, area_light=False), dict(env=False, area_light=False, textures=False)])
def test_distant_emitters_and_textures_are_bit_exact(api, oracle_record, variant, spectral):
    """handle_missed_ray (:462-481) over environment / directional emitters, alpha-tested and textured surfaces."""
    _compare(api, oracle_record, scenes.sky_room(40, 32, spectral=spectral, **variant), 2, what=str(variant))


@pytest.mark.parametrize("spectral", [False, True])
@pytest.mark.parametrize("kind", ["fog", "cloud", "tinted", "camera"])
def test_participating_media_are_bit_exact(api, oracle_record, kind, spectral):
    """try_sampling_medium / handle_sampled_medium (:259-298), Boundary crossings (:363-369), transmittance through sorted crossings."""
    _compare(api, oracle_record, scenes.media_box(kind, 32, 32, spectral=spectral), 2, what=kind)


@pytest.mark.parametrize("kind", scenes.CAMERA_KINDS)
def test_camera_variants_are_bit_exact(api, oracle_record, kind):
    _compare(api, oracle_record, scenes.camera_box(kind, 32, 32, spectral=True), 2, what=kind)


def test_million_triangle_room_is_bit_exact(api, oracle_record):
    sd = scenes.procedural_room(64, 36, env_size=(256, 128))
    _compare(api, oracle_record, sd, 1, what="C3 room")


def test_config4_and_config5_scenes_are_bit_exact(api, oracle_record):
    _compare(api, oracle_record, scenes.sss_dragon(32, 32), 1, what="C4 subsurface mesh")
    _compare(api, oracle_record, scenes.cloud_box(32, 32, grid=64), 2, what="C5 cloud")


def test_reference_loaded_cornell_asset_is_bit_exact(api, oracle_record):
    """The reference loader's own PODs (committed dump): the Blackman-Harris pixel-filter image is sampled from iteration 1 on (Film::sample,
    film.cxx:137-145), fog behind a Boundary mesh, sun + sky."""
    from etx_tracer_b200 import pod_io
    sd = pod_io.load(os.path.join(GOLDEN, "ref_cornell_40.npz"))
    assert int(sd.scene["pixel_sampler_image"][0]) != S.INVALID
    _compare(api, oracle_record, sd, 3, what="reference Cornell asset")


def test_adaptive_sampling_is_bit_exact(api, oracle_mod):
    """Film::estimate_noise_levels (film.cxx:233-330) after the even iterations from 32 on: error level, convergence, the two dilation passes;
    converged pixels are skipped by the next iterations (Film::active_pixel), so their sample counts stop."""
    sd = scenes.cornell_box(40, 36, **C1)
    n, thr = 41, 0.25
    o = _oracle(oracle_mod, sd, n, settings=(thr, 0.0))
    g = _device(api, sd, n, settings=(thr, 0.0))
    info_o = o.buffer(S.BUF_PIXEL_INFO, np.uint32)
    conv = (info_o & S.PIXEL_CONVERGED) != 0
    counts = info_o & S.PIXEL_COUNT_MASK
    assert 0 < conv.sum() < conv.size, "the case must have converged and active pixels"
    assert counts.min() < n and counts.max() == n
    _assert_bit_exact(_outputs(g, sd), _outputs(o, sd), "adaptive")
    assert bit_equal(g.buffer(S.BUF_PIXEL_ERROR, np.float32), o.buffer(S.BUF_PIXEL_ERROR, np.float32))
    gs, os_ = g.pt_status(), o.pt_status()
    assert gs["active_pixels"] == os_["active_pixels"]
    assert abs(gs["noise_level"] - os_["noise_level"]) <= 1e-4 * abs(os_["noise_level"])  # a float sum in another order
    g.close()
    o.close()


def test_update_loop_stops_when_every_pixel_converged(api):
    """CPUPathTracingImpl::update (path_tracing.cxx:85-110): non-blocking pump; the run ends at scene.samples or when an iteration
    processed no pixel."""
    import time
    sd = scenes.cornell_box(24, 24, samples=48, spectral=False)
    g = api.GPUPathTracing(sd, flavor="fast")
    g.set_scene_settings(1e9, 0.0)  # everything converges at the first estimate (iteration 32)
    g.run()
    t0 = time.time()
    while g.update():
        assert time.time() - t0 < 120.0
    st = g.status()
    assert st["completed_iterations"] == 34  # 0..32 rendered, the estimate after 32 converges all, iteration 33 processes nothing
    assert g.pt_status()["pixels_processed"] == 0
    info = g.buffer(S.BUF_PIXEL_INFO, np.uint32)
    assert ((info & S.PIXEL_COUNT_MASK) == 33).all() and ((info & S.PIXEL_CONVERGED) != 0).all()
    g.close()


# ---- product build: converged statistical parity ----------------------------------------------------------------------------------------
def _lum(img):
    return img[..., 0].astype(np.float64) * 0.212671 + img[..., 1].astype(np.float64) * 0.715160 + img[..., 2].astype(np.float64) * 0.072169


def _rel_mse(a, b, ref):
    eps = (0.01 * ref.mean()) ** 2
    return float((((a - b) ** 2) / (ref ** 2 + eps)).mean())


PRODUCT = {
    "C1": lambda: scenes.cornell_box(48, 48, samples=16, spectral=False),
    "C2": lambda: scenes.cornell_box(48, 48, samples=256, spectral=True, sphere=True),
    "C3": lambda: scenes.procedural_room(64, 36, env_size=(256, 128)),
    "C4": lambda: scenes.sss_dragon(40, 40),
    "C5": lambda: scenes.cloud_box(40, 40, grid=64),
}


@pytest.mark.parametrize("name", sorted(PRODUCT))
def test_product_build_statistical_parity(api, oracle_mod, name):
    """SURVEY 8(c) Tier C for the path tracer's product build: two oracle renders over different iteration windows give the run-to-run relMSE;
    the product render must be within 2x of it against either, and its mean within 1 % or 1.5x the oracle's own window-to-window difference."""
    sd = PRODUCT[name]()
    spp = 512
    threads = os.cpu_count() or 1
    flavor = "native" if oracle_mod.available("native") else "parity"
    oa = _oracle(oracle_mod, sd, spp, flavor=flavor, threads=threads, first=0)
    ob = _oracle(oracle_mod, sd, spp, flavor=flavor, threads=threads, first=4096)
    a, b = _lum(oa.film(S.FILM_CAMERA)[..., :3]), _lum(ob.film(S.FILM_CAMERA)[..., :3])
    g = _device(api, sd, spp, flavor="fast")
    img = g.film(S.FILM_CAMERA)[..., :3]
    assert np.isfinite(img).all()
    p = _lum(img)
    ref = 0.5 * (a + b)
    floor = _rel_mse(a, b, ref)
    vs_a, vs_b = _rel_mse(p, a, ref), _rel_mse(p, b, ref)
    bias = abs(p.mean() - ref.mean()) / ref.mean()
    own = abs(a.mean() - b.mean()) / ref.mean()
    print(f"\n[pt product parity {name}] relMSE floor {floor:.3e}  product vs A {vs_a / floor:.2f}x  vs B {vs_b / floor:.2f}x  mean bias {100 * bias:.3f} % (oracle {100 * own:.3f} %)")
    assert vs_b <= 2.0 * floor and vs_a <= 2.0 * floor
    assert bias <= max(0.01, 1.5 * own)
    nrm_g, nrm_o = g.film(S.FILM_NORMALS)[..., :3], oa.film(S.FILM_NORMALS)[..., :3]
    assert rel_l2(nrm_g, nrm_o) < 2e-2  # the first-hit layers share the stream: same geometry up to a few flipped hits per thousand
    g.close()


def test_iterations_in_flight_render_the_same_frame(api):
    """etxb_group lanes with the path tracer (adaptive sampling off): the lanes render the iteration indices 0..n-1 between them, the combined film is the
    mean over those iterations = the single-context frame up to float summation order."""
    sd = scenes.cornell_box(64, 48, **C2)
    n = 9
    ref = api.GPUPathTracing(sd, flavor="fast")
    ref.set_scene_settings(0.0, 0.0)
    ref.render(n)
    grp = api.GPUVCMGroup(sd, lanes=3, flavor="fast")
    grp.set_integrator(S.INTEGRATOR_PT)
    st = grp.render(n)
    assert st["completed_iterations"] == n and st["iteration_in_flight"] == 0
    a, b = grp.film(S.FILM_CAMERA)[..., :3], ref.film(S.FILM_CAMERA)[..., :3]
    assert np.isfinite(a).all() and rel_l2(a, b) < 1e-5, rel_l2(a, b)
    grp.close()
    ref.close()
