"""Scene FILES on the device (SURVEY 8(f) N2, end to end): the module's C++ loader -> etxb_scene_file_commit -> the integrators -> film export, as a
native program (host/render_main.cpp) next to the Python front end, and the procedural atmosphere of a file without distant emitters rendered bit-exactly
against the oracle.  Collected last on purpose: these are the newest device tests."""
import subprocess

import numpy as np
import pytest

from test_host_cpp import _build_native_renderer, _tiny_scene

pytestmark = pytest.mark.gpu


def test_native_renderer_renders_what_the_python_front_end_renders(tmp_path):
    """The C++ program and `python -m etx_tracer_b200.render` on the same scene file: same film (the light image is a float-atomic sum, so equal to
    rounding), both integrators, EXR and tone-mapped PNG."""
    from etx_tracer_b200 import loader, render
    exe = _build_native_renderer(tmp_path)
    scene = _tiny_scene(tmp_path)
    a, b = str(tmp_path / "native.exr"), str(tmp_path / "python.exr")
    out = subprocess.run([exe, scene, "-o", a, "--spp", "5", "--option", "vcm-merging=0"], capture_output=True, text=True)
    assert out.returncode == 0, (out.returncode, out.stdout[-500:], out.stderr[-500:])
    assert "5 of 5 iterations" in out.stdout
    assert render.main([scene, "-o", b, "--spp", "5", "--option", "vcm-merging=0"]) == 0
    fa, fb = loader.read_image(a)[0].astype(np.float64), loader.read_image(b)[0].astype(np.float64)
    assert fa.shape == fb.shape == (30, 40, 4) and fb[..., :3].mean() > 1e-3
    err = float(np.sqrt(((fa - fb)[..., :3] ** 2).sum()) / np.sqrt((fb[..., :3] ** 2).sum()))
    assert err < 1e-5, f"relative L2 {err:.3e}"
    a, b = str(tmp_path / "native.png"), str(tmp_path / "python.png")
    out = subprocess.run([exe, scene, "-o", a, "--integrator", "pt", "--spp", "6", "--png-exposure", "2.0", "--option", "bn=0"], capture_output=True, text=True)
    assert out.returncode == 0, (out.returncode, out.stdout[-500:], out.stderr[-500:])
    assert render.main([scene, "-o", b, "--integrator", "pt", "--spp", "6", "--exposure", "2.0", "--option", "bn=0"]) == 0
    pa, pb = loader.read_image(a)[0].astype(np.int32), loader.read_image(b)[0].astype(np.int32)
    assert pa.shape == pb.shape == (30, 40, 4) and pb[..., :3].max() > 30
    assert np.abs(pa - pb).max() <= 1


def test_default_atmosphere_scene_renders_bit_exact_on_the_device(oracle_record, tmp_path):
    """A scene file without distant emitters: the loader adds the default sun (Directional emitter with its 128 x 128 extinction image) and sky
    (Environment emitter, 256 x 128 image with an importance table, clamped in u).  The parity build against the oracle on those PODs, both integrators."""
    from conftest import same_bits
    from etx_tracer_b200 import api, structs as S
    sd = api.SceneFile(_tiny_scene(tmp_path), flavor="parity")
    assert int(sd.scene["environment_emitter_count"][0]) == 2
    buffers = ((S.BUF_LIGHT_SAMPLER, np.uint32), (S.BUF_LV_POS, np.float32), (S.BUF_CAMERA_SAMPLER, np.uint32), (S.BUF_CAMERA_GATHERED, np.float32))
    layers = (S.FILM_CAMERA, S.FILM_NORMALS, S.FILM_ALBEDO)

    def run(m):
        o = m.Oracle(sd)
        o.begin(0)
        o.run(2, threads=1)
        out = {f"vcm buffer {bid}": o.buffer(bid, dt) for bid, dt in buffers}
        out["vcm film camera"] = o.film(S.FILM_CAMERA)[..., :3]
        o.set_integrator(S.INTEGRATOR_PT)
        o.pt_set_options(S.default_pt_options())
        o.begin(0)
        o.run(3, threads=1)
        out["pt camera sampler"] = o.buffer(S.BUF_CAMERA_SAMPLER, np.uint32)
        out.update({f"pt film {layer}": o.film(layer)[..., :3] for layer in layers})
        o.close()
        return out

    ref = oracle_record("", run)
    g = api.GPUVCM(sd, flavor="parity")
    g.render(2)
    for bid, dt in buffers:
        assert same_bits(g.buffer(bid, dt), ref[f"vcm buffer {bid}"]), f"buffer {bid}"
    assert same_bits(g.film(S.FILM_CAMERA)[..., :3], ref["vcm film camera"])
    g.close()
    p = api.GPUPathTracing(sd, flavor="parity")
    p.render(3)
    assert same_bits(p.buffer(S.BUF_CAMERA_SAMPLER, np.uint32), ref["pt camera sampler"])
    for layer in layers:
        assert same_bits(p.film(layer)[..., :3], ref[f"pt film {layer}"]), layer
    p.close()


def test_nanovdb_medium_scene_renders_bit_exact_on_the_device(oracle_mod, tmp_path):
    """`et::medium … volume cloud.nvdb` read by the module's NanoVDB reader into the dense grid of a heterogeneous medium: the parity build against the
    oracle on the loader's PODs (delta tracking through the grid), both integrators."""
    import os
    from conftest import bit_equal
    from etx_tracer_b200 import api, structs as S
    from test_loader import MTL, NVDB_MAKE, _write_scene
    if not os.path.exists(NVDB_MAKE):
        pytest.skip("oracle/_ref/nvdb_make not built")
    subprocess.check_call([NVDB_MAKE, "blobs", str(tmp_path / "cloud.nvdb")])
    sd = api.SceneFile(_write_scene(tmp_path, mtl=MTL.replace("scattering 0.4", "scattering 0.4\nvolume cloud.nvdb")), flavor="parity")
    assert 1 in [int(m["cls"]) for m in np.frombuffer((__import__("ctypes").c_char * (int(sd.scene["mediums"]["count"][0]) * S.MEDIUM.itemsize)).from_address(
        int(sd.scene["mediums"]["a"][0])), dtype=S.MEDIUM)]
    o = oracle_mod.Oracle(sd)
    o.begin(0)
    o.run(2, threads=1)
    g = api.GPUVCM(sd, flavor="parity")
    g.render(2)
    for bid, dt in ((S.BUF_LIGHT_SAMPLER, np.uint32), (S.BUF_LV_POS, np.float32), (S.BUF_CAMERA_SAMPLER, np.uint32), (S.BUF_CAMERA_GATHERED, np.float32)):
        assert bit_equal(g.buffer(bid, dt), o.buffer(bid, dt)), f"buffer {bid}"
    assert bit_equal(g.film(S.FILM_CAMERA)[..., :3], o.film(S.FILM_CAMERA)[..., :3])
    g.close()
    o.set_integrator(S.INTEGRATOR_PT)
    o.pt_set_options(S.default_pt_options())
    o.begin(0)
    o.run(2, threads=1)
    p = api.GPUPathTracing(sd, flavor="parity")
    p.render(2)
    assert bit_equal(p.buffer(S.BUF_CAMERA_SAMPLER, np.uint32), o.buffer(S.BUF_CAMERA_SAMPLER, np.uint32))
    assert bit_equal(p.film(S.FILM_CAMERA)[..., :3], o.film(S.FILM_CAMERA)[..., :3])
    p.close()
    o.close()
