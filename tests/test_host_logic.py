"""Host-side logic that runs without a GPU: scene generators, struct layout, C-ABI surface, error behaviour."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, bit_equal
from etx_tracer_b200 import build as etx_build
from etx_tracer_b200 import scenes, structs as S


def test_rgb_reflectance_restatement_matches_reference(oracle_mod):
    # scenes.spd_rgb_reflectance restates SpectralDistribution::rgb_reflectance (render/host/spectrum.cxx:135-148)
    lib = oracle_mod.load("parity")
    for rgb in ([1, 1, 1], [0.906, 0.906, 0.906], [1, 0, 0], [0, 1, 0], [0.2, 0.5, 0.7]):
        want = np.zeros(1, S.SPECTRUM)
        lib.oracle_spectrum_rgb_reflectance(oracle_mod._p(np.array(rgb, np.float32)), oracle_mod._p(want))
        got = scenes.spd_rgb_reflectance(rgb)
        assert bit_equal(got["entries"]["power"], want["entries"]["power"])
        assert bit_equal(got["integrated"], want["integrated"]) and got["entry_count"] == want["entry_count"]
    want = np.zeros(1, S.SPECTRUM)
    lib.oracle_spectrum_rgb_luminance(oracle_mod._p(np.array([10.018, 3.918, 0.932], np.float32)), oracle_mod._p(want))
    got = scenes.spd_rgb_luminance([10.018, 3.918, 0.932])
    assert bit_equal(got["entries"]["power"], want["entries"]["power"]) and bit_equal(got["integrated"], want["integrated"])


def test_camera_restatement_matches_reference_build_camera(oracle_mod):
    lib = oracle_mod.load("parity")
    sd = scenes.cornell_box(40, 30, samples=4)
    ref = sd.camera.copy()
    o = np.array([0.0, 1.0, 3.82], np.float32)
    t = np.array([0.0, 1.0, -6.18], np.float32)
    u = np.array([0.0, 1.0, 0.0], np.float32)
    lib.oracle_build_camera(oracle_mod._p(ref), oracle_mod._p(o), oracle_mod._p(t), oracle_mod._p(u), 40, 30, np.float32(39.597755335771296))
    for f in ("position", "side", "up", "direction", "tan_half_fov", "aspect", "area", "image_plane", "view_proj"):
        np.testing.assert_allclose(sd.camera[f], ref[f], rtol=2e-6, atol=1e-7, err_msg=f)


def test_scene_generator_invariants():
    sd = scenes.cornell_box(64, 64, samples=256, spectral=True, sphere=True)
    assert sd.triangle_count == 20480 + 26  # BASELINE config 2: 20 480-triangle sphere
    assert sd.scene["flags"][0] & S.SCENE_SPECTRAL
    d = sd.a_dist
    assert d["cdf"][0] == 0 and d["cdf"][-1] == 1 and np.all(np.diff(d["cdf"]) >= 0)
    np.testing.assert_allclose(d["pdf"][:-1].sum(), 1.0, rtol=1e-6)
    gn = sd.a_triangles["geo_n"]
    np.testing.assert_allclose(np.linalg.norm(gn, axis=1), 1.0, rtol=1e-5)
    em = sd.a_tri_to_emitter[sd.a_tri_to_emitter != S.INVALID]
    assert sorted(em) == list(range(sd.a_emitters.shape[0]))
    # every material got the defaults validate_materials would add (scene_representation.cxx:262-300)
    for m in sd.a_materials:
        assert m["reflectance"]["spectrum_index"] != S.INVALID and m["int_ior"]["eta_index"] != S.INVALID


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "etx_b200.h")).read()
    return sorted(set(re.findall(r"\b(etxb_[a-z_0-9]+)\s*\(", text)))


@pytest.mark.parametrize("flavor", ["fast", "parity"])
def test_c_abi_library_loads_and_exports_every_declared_symbol(flavor):
    path = etx_build.lib_path(flavor)
    if not os.path.exists(path):
        etx_build.build((flavor,))
    lib = ctypes.CDLL(path)
    names = _declared_functions()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/etx_b200.h but not exported by {os.path.basename(path)}"
    lib.etxb_build_flavor.restype = ctypes.c_char_p
    assert lib.etxb_build_flavor().decode() == flavor


def test_options_keys_follow_the_reference():
    # VCMOptions::load keys (rt/integrators/vcm_shared.cxx:15-28)
    lib = ctypes.CDLL(etx_build.lib_path("fast"))
    lib.etxb_options_set_key.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_double]
    o = np.zeros(1, S.VCM_OPTIONS)
    lib.etxb_options_default(o.ctypes.data_as(ctypes.c_void_p))
    ref = S.default_vcm_options()
    assert o.tobytes() == ref.tobytes()
    p = o.ctypes.data_as(ctypes.c_void_p)
    assert lib.etxb_options_set_key(p, b"vcm-merging", 0.0) == 0 and not (o["options"][0] & S.VCM_ENABLE_MERGING)
    assert lib.etxb_options_set_key(p, b"vcm-radius_decay", 128.0) == 0 and o["radius_decay"][0] == 128
    assert lib.etxb_options_set_key(p, b"vcm-initial_radius", 0.25) == 0 and o["initial_radius"][0] == np.float32(0.25)
    assert lib.etxb_options_set_key(p, b"vcm-kernel", 0.0) == 0 and o["kernel"][0] == 0
    assert lib.etxb_options_set_key(p, b"vcm-no-such-key", 1.0) < 0


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from etx_tracer_b200.api import EtxbError, GPUVCM
    with pytest.raises(EtxbError):
        GPUVCM(scenes.cornell_box(16, 16, samples=1))


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the reference's CPU VCM through oracle/_ref) runs without a GPU: one JSON line with the keys the driver
    reads — same metric/unit as the GPU arm, impl = reference, zero host<->device bytes, a cpu_baseline describing the run."""
    import json
    import os
    import subprocess
    import sys
    from oracle import oracle_py
    if not (oracle_py.available("native") or oracle_py.available("parity")):
        import pytest
        pytest.skip("oracle/_ref not built")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "C1", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True and d["metric"].startswith("Msamples/s")
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "C1" in d["config"]["workload"]


def test_bench_algorithmic_bytes_follow_the_survey_formula():
    """SURVEY.md 8(d): per-kernel byte costs x event counters; the whole-step figure is their sum."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    c = dict(bounces_light=10, bounces_camera=20, light_vertices=7, connections=30, merge_queries=5, merge_candidates=400, merge_accepts=60, splats=3, rays_shadow=50,
             rays_closest=30)
    total, per = bench.algorithmic_bytes(c, n_pixels=16, steps=2)
    assert per["camera_merge"] == 128 * 5 + 12 * 400 + 48 * 60
    assert per["camera_connect"] == 516 * 30
    assert per["camera_shade"] == 756 * 20 and per["trace_closest(camera)"] == 48 * 20
    assert per["camera_continue"] == 352 * 20 + 104 * 16 * 2
    assert per["shadow_trace"] == 48 * (50 - 7)
    once = {k: v for k, v in per.items() if k != "camera_merge_generic"}  # the two gather kernels share one figure
    assert total == sum(once.values())


def test_replica_mode_deals_every_iteration_exactly_once():
    """etxb_group_enqueue in replica mode (module.cu replica_plan, through the device-free test hook): whole frames round-robin; with a split lane
    the n % world left-over iterations are split over world / (n % world) ranks each by camera tile.  Whatever (world, n): every ordinal is
    rendered exactly once — by one rank as a whole frame, or by `parts` ranks holding the parts 0 .. parts - 1 — and no rank carries more than
    ceil(n / world) units of work."""
    import ctypes as C
    from etx_tracer_b200 import api
    lib = api.load_library("fast")
    lib.etxb_debug_replica_plan.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_uint32]
    buf = np.zeros(3 * 256, dtype=np.uint32)
    for world in range(1, 9):
        for n in range(1, 41):
            for split in (0, 1):
                whole, parts_seen, load = {}, {}, [0.0] * world
                for rank in range(world):
                    k = lib.etxb_debug_replica_plan(world, rank, 100, n, split, buf.ctypes.data_as(C.c_void_p), 256)
                    assert k >= 0
                    for i in range(k):
                        j, part, parts = (int(v) for v in buf[i * 3:i * 3 + 3])
                        assert 100 <= j < 100 + n
                        if parts == 1:
                            whole[j] = whole.get(j, 0) + 1
                            load[rank] += 1.0
                        else:
                            assert split and n >= world and parts == world // (n % world) and parts >= 2
                            parts_seen.setdefault(j, []).append(part)
                            load[rank] += 1.0 / parts
                for j in range(100, 100 + n):
                    if j in whole:
                        assert whole[j] == 1 and j not in parts_seen, (world, n, split, j)
                    else:
                        p = sorted(parts_seen[j])
                        assert p == list(range(len(p))) and len(p) == world // (n % world), (world, n, split, j, p)
                assert max(load) <= -(-n // world) + 1e-9
                if split and n >= world and n % world and world // (n % world) >= 2:
                    assert max(load) < -(-n // world)  # the point of the split: nobody a whole iteration behind
