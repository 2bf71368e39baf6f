"""ctypes binding of the C ABI (include/etx_b200.h) + `GPUVCM`, the Python mirror of the reference's
Integrator interface for this path (sources/etx/rt/integrators/integrator.hxx:12-98, vcm_cpu.cxx:247-310).

There is no CPU fallback: loading fails loudly if the CUDA library is missing, and every call raises
EtxbError with the module's message when the device path cannot do what was asked.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build
from . import scenes as _scenes
from . import structs as S

_libs = {}


class EtxbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"etxb error {code}: {message}")
        self.code = code


def load_library(flavor="fast"):
    if flavor in _libs:
        return _libs[flavor]
    path = _build.lib_path(flavor)
    if not os.path.exists(path):
        raise EtxbError(-100, f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
    lib = C.CDLL(path)
    vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
    lib.etxb_build_flavor.restype = C.c_char_p
    lib.etxb_last_error.restype = C.c_char_p
    lib.etxb_last_error.argtypes = [vp]
    lib.etxb_create.argtypes = [C.POINTER(vp), vp]
    lib.etxb_destroy.argtypes = [vp]
    lib.etxb_destroy.restype = None
    lib.etxb_upload_scene.argtypes = [vp, vp, u64, vp, u64]
    lib.etxb_upload_blue_noise.argtypes = [vp, vp, vp, vp]
    lib.etxb_upload_color_tables.argtypes = [vp, vp, vp]
    lib.etxb_scene_file_load.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(vp), C.c_char_p, u64]
    lib.etxb_scene_file_free.argtypes = [vp]
    lib.etxb_scene_file_free.restype = None
    lib.etxb_scene_file_set_samples.argtypes = [vp, u32]
    lib.etxb_scene_file_set_samples.restype = None
    lib.etxb_scene_file_commit.argtypes = [vp, vp]
    lib.etxb_scene_file_table.argtypes = [vp, C.c_char_p, C.POINTER(u64)]
    lib.etxb_scene_file_table.restype = vp
    lib.etxb_atmosphere_images.argtypes = [C.c_char_p, vp, C.c_float, vp, u32, u32, vp, vp]
    lib.etxb_options_file_string.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, u64]
    lib.etxb_mesh_tangents.argtypes = [vp, u64, vp, u64]
    lib.etxb_image_file_read.argtypes = [C.c_char_p, vp, vp, vp, vp, u64, C.c_char_p, u64]
    lib.etxb_nvdb_density.argtypes = [C.c_char_p, vp, vp, u64, C.c_char_p, u64]
    for fn in (lib.etxb_scene_file_scene, lib.etxb_scene_file_camera):
        fn.argtypes = [vp]
        fn.restype = vp
    for fn in (lib.etxb_scene_file_warning_count, lib.etxb_scene_file_material_count):
        fn.argtypes = [vp]
        fn.restype = u32
    for fn in (lib.etxb_scene_file_warning, lib.etxb_scene_file_material_name):
        fn.argtypes = [vp, u32]
        fn.restype = C.c_char_p
    lib.etxb_options_default.argtypes = [vp]
    lib.etxb_options_default.restype = None
    lib.etxb_options_set_key.argtypes = [vp, C.c_char_p, C.c_double]
    lib.etxb_set_options.argtypes = [vp, vp]
    lib.etxb_set_next_iteration.argtypes = [vp, u32]
    lib.etxb_group_create.argtypes = [C.POINTER(vp), vp, u32]
    lib.etxb_group_destroy.argtypes = [vp]
    lib.etxb_group_destroy.restype = None
    lib.etxb_group_lanes.argtypes = [vp]
    lib.etxb_group_lanes.restype = u32
    lib.etxb_group_lane.argtypes = [vp, u32]
    lib.etxb_group_lane.restype = vp
    lib.etxb_group_last_error.argtypes = [vp]
    lib.etxb_group_last_error.restype = C.c_char_p
    lib.etxb_group_begin.argtypes = [vp, u32]
    lib.etxb_group_enqueue.argtypes = [vp, u32]
    lib.etxb_group_wait.argtypes = [vp]
    lib.etxb_group_poll.argtypes = [vp, vp]
    lib.etxb_group_read_film.argtypes = [vp, u32, vp, u64]
    lib.etxb_group_set_stride.argtypes = [vp, u32]
    lib.etxb_group_combine.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u32)]
    lib.etxb_comm_unique_id.argtypes = [vp, u64]
    lib.etxb_comm_init.argtypes = [vp, u32, u32, vp, u64]
    lib.etxb_comm_world.argtypes = [vp, C.POINTER(u32), C.POINTER(u32)]
    lib.etxb_comm_reduce_film.argtypes = [vp, u32, vp, u64]
    lib.etxb_group_comm_init.argtypes = [vp, u32, u32, vp, u32]
    lib.etxb_group_comm_reduce_film.argtypes = [vp, u32, vp, u64]
    lib.etxb_group_comm_init_replicas.argtypes = [vp, u32, u32, vp, u64]
    lib.etxb_group_reserve_split_lane.argtypes = [vp]
    lib.etxb_set_integrator.argtypes = [vp, u32]
    lib.etxb_pt_options_default.argtypes = [vp]
    lib.etxb_pt_options_default.restype = None
    lib.etxb_pt_options_set_key.argtypes = [vp, C.c_char_p, C.c_double]
    lib.etxb_pt_set_options.argtypes = [vp, vp]
    lib.etxb_pt_get_status.argtypes = [vp, vp]
    lib.etxb_set_scene_settings.argtypes = [vp, C.c_float, C.c_float]
    lib.etxb_set_partition.argtypes = [vp, u32, u32]
    lib.etxb_set_iteration_stride.argtypes = [vp, u32]
    lib.etxb_begin.argtypes = [vp, u32]
    lib.etxb_enqueue_iteration.argtypes = [vp]
    lib.etxb_enqueue_light_pass.argtypes = [vp]
    lib.etxb_enqueue_grid_build.argtypes = [vp, vp, u64]
    lib.etxb_enqueue_camera_pass.argtypes = [vp]
    lib.etxb_poll.argtypes = [vp, vp]
    lib.etxb_wait.argtypes = [vp]
    lib.etxb_stop.argtypes = [vp, C.c_int]
    lib.etxb_read_film.argtypes = [vp, u32, vp, u64]
    lib.etxb_film_size.argtypes = [vp, C.POINTER(u32), C.POINTER(u32)]
    lib.etxb_read_film_ldr.argtypes = [vp, u32, C.c_float, vp, u64]
    lib.etxb_save_film.argtypes = [vp, u32, C.c_char_p, u32, C.c_float]
    lib.etxb_write_exr.argtypes = [C.c_char_p, vp, u32, u32]
    lib.etxb_write_png.argtypes = [C.c_char_p, vp, u32, u32]
    lib.etxb_tonemap_rgba8.argtypes = [vp, u64, C.c_float, vp]
    lib.etxb_get_counters.argtypes = [vp, vp]
    lib.etxb_get_kernel_times.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.POINTER(u32), u32]
    lib.etxb_read_buffer.argtypes = [vp, u32, vp, u64, C.POINTER(u64)]
    lib.etxb_device_pointer.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u64)]
    lib.etxb_stream.restype = vp
    lib.etxb_stream.argtypes = [vp]
    lib.etxb_debug_trace.argtypes = [vp, vp, vp, u32, vp, vp]
    lib.etxb_debug_select_tree.argtypes = [vp, C.c_int]
    lib.etxb_debug_sampler.argtypes = [vp, vp, vp, u32, u32, vp, vp]
    lib.etxb_debug_math.argtypes = [vp, u32, vp, vp, u32, vp]
    _libs[flavor] = lib
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def read_image(file_name, flavor="fast"):
    """The module's image readers (PNG in every form, OpenEXR, Radiance HDR, PFM): (H, W, 4) uint8 or float32, rows in file order."""
    lib = load_library(flavor)
    w, h, eight = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    err = C.create_string_buffer(512)
    if lib.etxb_image_file_read(os.fsencode(file_name), C.byref(w), C.byref(h), C.byref(eight), None, 0, err, len(err)) != 0:
        raise EtxbError(-4, err.value.decode(errors="replace"))
    out = np.zeros((h.value, w.value, 4), dtype=np.uint8 if eight.value else np.float32)
    if lib.etxb_image_file_read(os.fsencode(file_name), C.byref(w), C.byref(h), C.byref(eight), _p(out), out.nbytes, err, len(err)) != 0:
        raise EtxbError(-4, err.value.decode(errors="replace"))
    return out


def write_exr(file_name, rgba, flavor="fast"):
    """float4 image (H, W, 4) -> OpenEXR (32-bit float A, B, G, R channels, scan lines, no compression); host code of the module."""
    rgba = np.ascontiguousarray(rgba, dtype=np.float32)
    rc = load_library(flavor).etxb_write_exr(os.fsencode(file_name), _p(rgba), rgba.shape[1], rgba.shape[0])
    if rc != 0:
        raise EtxbError(rc, f"could not write {file_name}")


def write_png(file_name, rgba8, flavor="fast"):
    rgba8 = np.ascontiguousarray(rgba8, dtype=np.uint8)
    rc = load_library(flavor).etxb_write_png(os.fsencode(file_name), _p(rgba8), rgba8.shape[1], rgba8.shape[0])
    if rc != 0:
        raise EtxbError(rc, f"could not write {file_name}")


def tonemap(rgba, exposure=1.0, flavor="fast"):
    """The reference's LDR tone map on the host (app.cxx:268-282): 1 - exp(-exposure c), sRGB curve, 8 bits."""
    rgba = np.ascontiguousarray(rgba, dtype=np.float32)
    out = np.zeros(rgba.shape[:-1] + (4,), dtype=np.uint8)
    load_library(flavor).etxb_tonemap_rgba8(_p(rgba), rgba.size // 4, C.c_float(exposure), _p(out))
    return out


class SceneFile:
    """A scene file read by the module's C++ loader (csrc/scene_loader.cpp; replaces SceneRepresentation::load_from_file,
    render/host/scene_representation.cxx:679-838).  Duck-types scenes.SceneData for GPUVCM / GPUPathTracing / GPUVCMGroup: `.scene`, `.camera`
    (numpy views of the Scene / Camera PODs the loader object owns), width / height / triangle_count, `.warnings`, `.material_names`."""

    def __init__(self, file_name, flavor="fast", data_folder=None):
        self.lib = load_library(flavor)
        self.h = C.c_void_p()
        err = C.create_string_buffer(1024)
        rc = self.lib.etxb_scene_file_load(os.fsencode(file_name), os.fsencode(data_folder) if data_folder else None, C.byref(self.h), err, len(err))
        if rc != 0:
            self.h = C.c_void_p()
            raise EtxbError(rc, err.value.decode(errors="replace") or f"could not load {file_name}")
        self.scene = np.frombuffer((C.c_char * S.SCENE.itemsize).from_address(self.lib.etxb_scene_file_scene(self.h)), dtype=S.SCENE)
        self.camera = np.frombuffer((C.c_char * S.CAMERA.itemsize).from_address(self.lib.etxb_scene_file_camera(self.h)), dtype=S.CAMERA).copy()
        self.warnings = [self.lib.etxb_scene_file_warning(self.h, i).decode(errors="replace") for i in range(self.lib.etxb_scene_file_warning_count(self.h))]
        self.material_names = {self.lib.etxb_scene_file_material_name(self.h, i).decode(errors="replace"): i for i in range(self.lib.etxb_scene_file_material_count(self.h))}
        self.name = os.path.basename(os.fsdecode(file_name))

    @property
    def width(self):
        return int(self.camera["film_size"][0][0])

    @property
    def height(self):
        return int(self.camera["film_size"][0][1])

    @property
    def triangle_count(self):
        return int(self.scene["triangles"]["count"][0])

    def table(self, name, dtype=np.uint8):
        """a table of tables.bin by name ("bluenoise/sobol", "color_tables/xyz_441x3", ...), None when absent"""
        n = C.c_uint64(0)
        p = self.lib.etxb_scene_file_table(self.h, name.encode(), C.byref(n))
        return np.frombuffer((C.c_char * n.value).from_address(p), dtype=dtype).copy() if p else None

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.scene = None
            self.lib.etxb_scene_file_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def load_scene_file(file_name, flavor="fast"):
    return SceneFile(file_name, flavor=flavor)


COMM_ID_BYTES = 128


def comm_unique_ids(count, flavor="fast"):
    """`count` NCCL unique ids (ETXB_COMM_ID_BYTES each) from the module, for rank 0 to hand to the other ranks by any transport."""
    lib = load_library(flavor)
    ids = np.zeros(count * COMM_ID_BYTES, dtype=np.uint8)
    for k in range(count):
        rc = lib.etxb_comm_unique_id(ids[k * COMM_ID_BYTES:].ctypes.data_as(C.c_void_p), COMM_ID_BYTES)
        if rc != 0:
            raise EtxbError(rc, "etxb_comm_unique_id failed (libnccl.so.2 missing?)")
    return ids


class GPUVCM:
    """`name()/run()/update()/stop()/status()/options` like the reference's CPUVCM, driving the CUDA module."""

    def __init__(self, scene_data=None, flavor="fast", device=0, max_light_vertices=0, profile=False, _adopt=None):
        self.lib = load_library(flavor)
        self.flavor = flavor
        self.h = C.c_void_p()
        self._owned = _adopt is None
        if _adopt is not None:
            self.h = C.c_void_p(_adopt)  # a lane of an etxb_group: the group owns the context
        else:
            cfg = np.zeros(1, dtype=S.DEVICE_CONFIG)
            cfg["device_index"] = device
            cfg["max_light_vertices"] = max_light_vertices
            cfg["flags"] = 1 if profile else 0
            rc = self.lib.etxb_create(C.byref(self.h), _p(cfg))
            if rc != 0:
                raise EtxbError(rc, "etxb_create failed (no CUDA device? the module has no CPU fallback)")
        self.options = S.default_vcm_options()
        self.scene_data = None
        self._running = False
        self._target_iterations = 0
        ct = _scenes.tables("color_tables")
        self._xyz = np.ascontiguousarray(ct["xyz_441x3"], dtype=np.float32)
        self._rgbr = np.ascontiguousarray(ct["rgb_response_391x3"], dtype=np.float32)
        self._check(self.lib.etxb_upload_color_tables(self.h, _p(self._xyz), _p(self._rgbr)))
        if scene_data is not None:
            self.set_scene(scene_data)

    # -- plumbing ---------------------------------------------------------------------------------
    def _check(self, rc):
        if rc < 0:
            raise EtxbError(rc, self.lib.etxb_last_error(self.h).decode())
        return rc

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            if self._owned:
                self.lib.etxb_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- Integrator surface -------------------------------------------------------------------------
    @staticmethod
    def name():
        return "VCM (B200)"

    def set_scene(self, scene_data):
        """Raytracing::link_scene/link_camera + commit_changes."""
        self.scene_data = scene_data
        samples = int(scene_data.scene["samples"][0])
        # BNSampler variant = next_power(min(samples, 256)) (thirdparty/bluenoise/bluenoise.cxx:73-95)
        spp = 1
        while spp < min(max(samples, 1), 256):
            spp *= 2
        bn = _scenes.tables("bluenoise")
        self._bn = [np.ascontiguousarray(bn[k], dtype=np.uint8) for k in ("sobol", f"scrambling_{spp}", f"ranking_{spp}")]
        self._check(self.lib.etxb_upload_blue_noise(self.h, _p(self._bn[0]), _p(self._bn[1]), _p(self._bn[2])))
        self._check(self.lib.etxb_upload_scene(self.h, _p(scene_data.scene), scene_data.scene.nbytes, _p(scene_data.camera), scene_data.camera.nbytes))
        w, h = C.c_uint32(0), C.c_uint32(0)
        self._check(self.lib.etxb_film_size(self.h, C.byref(w), C.byref(h)))
        self.width, self.height = w.value, h.value

    def set_option(self, key, value):
        """Integrator::options() keys: vcm-initial_radius, vcm-radius_decay, vcm-blue_noise, vcm-kernel, vcm-direct_hit, ..."""
        rc = self.lib.etxb_options_set_key(_p(self.options), key.encode(), float(value))
        if rc != 0:
            raise EtxbError(rc, f"unknown option key {key}")

    def set_partition(self, rank, world):
        self._check(self.lib.etxb_set_partition(self.h, rank, world))

    def comm_init(self, world, rank, comm_id):
        """Pixel tiles over `world` processes (one GPU each): collective; comm_id = the 128 bytes rank 0 got from comm_unique_ids(1)."""
        comm_id = np.ascontiguousarray(comm_id, dtype=np.uint8)
        self._check(self.lib.etxb_comm_init(self.h, world, rank, _p(comm_id), comm_id.nbytes))

    def comm_reduce_film(self, layer=S.FILM_RESULT, out=None):
        """Collective: the whole frame on rank 0 (returned there; None elsewhere)."""
        w, r = C.c_uint32(1), C.c_uint32(0)
        self._check(self.lib.etxb_comm_world(self.h, C.byref(w), C.byref(r)))
        if (out is None) and (r.value == 0):
            out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._check(self.lib.etxb_comm_reduce_film(self.h, layer, _p(out) if r.value == 0 else None, out.nbytes if r.value == 0 else 0))
        return out if r.value == 0 else None

    def set_iteration_stride(self, stride):
        """This context renders iterations first, first + stride, ... (iteration-interleaved multi-GPU runs)."""
        self._check(self.lib.etxb_set_iteration_stride(self.h, stride))

    def run(self, first_iteration=0):
        """CPUVCM::run -> CPUVCMImpl::start: clears the film and arms iteration 0."""
        self._check(self.lib.etxb_set_options(self.h, _p(self.options)))
        self._check(self.lib.etxb_begin(self.h, first_iteration))
        self._running = True
        self._target_iterations = int(self.scene_data.scene["samples"][0])

    def update(self):
        """One pump of the integrator, non-blocking like CPUVCM::update (vcm_cpu.cxx:264-276): queues the next iteration once the previous one has
        finished; stops at scene.samples like the reference."""
        if not self._running:
            return False
        st = self.status()
        if st["iteration_in_flight"]:
            return True
        if st["completed_iterations"] >= self._target_iterations:
            self._running = False
            return False
        self._check(self.lib.etxb_enqueue_iteration(self.h))
        return True

    def render(self, iterations, first_iteration=0):
        self.run(first_iteration)
        for _ in range(iterations):
            self._check(self.lib.etxb_enqueue_iteration(self.h))
        self._check(self.lib.etxb_wait(self.h))
        return self.status()

    def iterate(self):
        self._check(self.lib.etxb_enqueue_iteration(self.h))

    def light_pass(self):
        self._check(self.lib.etxb_enqueue_light_pass(self.h))

    def grid_build(self, records_ptr=None, count=0):
        """complete_light_vertices: commits the light image, builds the photon grid (from gathered records in multi-GPU runs)."""
        self._check(self.lib.etxb_enqueue_grid_build(self.h, records_ptr, count))

    def camera_pass(self):
        self._check(self.lib.etxb_enqueue_camera_pass(self.h))

    def stop(self, wait_for_iteration=True):
        self._running = False
        self._check(self.lib.etxb_stop(self.h, 1 if wait_for_iteration else 0))

    def wait(self):
        self._check(self.lib.etxb_wait(self.h))

    def status(self):
        st = np.zeros(1, dtype=S.STATUS)
        self._check(self.lib.etxb_poll(self.h, _p(st)))
        return {k: st[k][0].item() for k in st.dtype.names}

    # -- results --------------------------------------------------------------------------------------
    def film(self, layer=S.FILM_RESULT, out=None):
        if out is None:
            out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._check(self.lib.etxb_read_film(self.h, layer, _p(out), out.nbytes))
        return out

    def film_ldr(self, layer=S.FILM_RESULT, exposure=1.0):
        """The tone-mapped 8-bit frame of the reference's viewer / LDR export (app.cxx:268-282), tone-mapped on the device."""
        out = np.zeros((self.height, self.width, 4), dtype=np.uint8)
        self._check(self.lib.etxb_read_film_ldr(self.h, layer, C.c_float(exposure), _p(out), out.nbytes))
        return out

    def save_image(self, file_name, layer=S.FILM_RESULT, tonemapped=False, exposure=1.0):
        """RTApplication::on_save_image_selected (app.cxx:261-295): the float layer as OpenEXR, or tone-mapped as PNG."""
        self._check(self.lib.etxb_save_film(self.h, layer, os.fsencode(file_name), 1 if tonemapped else 0, C.c_float(exposure)))

    def counters(self):
        c = np.zeros(1, dtype=S.COUNTERS)
        self._check(self.lib.etxb_get_counters(self.h, _p(c)))
        return {k: int(c[k][0]) for k in c.dtype.names}

    def kernel_times(self):
        cap = 32
        names = (C.c_char_p * cap)()
        ms = (C.c_float * cap)()
        launches = (C.c_uint32 * cap)()
        n = self._check(self.lib.etxb_get_kernel_times(self.h, names, ms, launches, cap))
        return {names[i].decode(): (float(ms[i]), int(launches[i])) for i in range(n)}

    def buffer(self, buf_id, dtype):
        n = C.c_uint64(0)
        self._check(self.lib.etxb_read_buffer(self.h, buf_id, None, 0, C.byref(n)))
        out = np.zeros(n.value // np.dtype(dtype).itemsize, dtype=dtype)
        if n.value:
            self._check(self.lib.etxb_read_buffer(self.h, buf_id, _p(out), out.nbytes, C.byref(n)))
        return out

    def device_pointer(self, buf_id):
        ptr, n = C.c_void_p(), C.c_uint64(0)
        self._check(self.lib.etxb_device_pointer(self.h, buf_id, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def stream(self):
        return self.lib.etxb_stream(self.h)

    # -- unit entry points (parity tests) -----------------------------------------------------------------
    def debug_select_tree(self, wide):
        """etxb_debug_trace walks the BVH2 (False) or the product build's 4-wide quantised tree (True); returns whether that tree exists."""
        return self.lib.etxb_debug_select_tree(self.h, 1 if wide else 0) == 1

    def debug_trace(self, rays, seeds):
        rays = np.ascontiguousarray(rays, dtype=np.float32)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32).copy()
        n = rays.shape[0]
        uvt = np.zeros((n, 3), dtype=np.float32)
        tri = np.zeros(n, dtype=np.uint32)
        self._check(self.lib.etxb_debug_trace(self.h, _p(rays), _p(seeds), n, _p(uvt), _p(tri)))
        return uvt, tri, seeds

    def debug_sampler(self, a, b, draws):
        a = np.ascontiguousarray(a, dtype=np.uint32)
        b = np.ascontiguousarray(b, dtype=np.uint32)
        n = a.shape[0]
        seeds = np.zeros((n, draws + 1), dtype=np.uint32)
        vals = np.zeros((n, max(draws, 1)), dtype=np.float32)
        self._check(self.lib.etxb_debug_sampler(self.h, _p(a), _p(b), n, draws, _p(seeds), _p(vals)))
        return seeds, vals[:, :draws]

    def debug_math(self, fn, x, y=None):
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.zeros_like(x)
        yy = np.ascontiguousarray(y, dtype=np.float32) if y is not None else None
        self._check(self.lib.etxb_debug_math(self.h, fn, _p(x), _p(yy) if yy is not None else None, x.shape[0], _p(out)))
        return out


class GPUPathTracing(GPUVCM):
    """`name()/run()/update()/stop()/status()/options` like the reference's CPUPathTracing (rt/integrators/path_tracing.cxx:122-170) on the same CUDA
    context type: one path per active pixel and iteration, normal / albedo layers, adaptive sampling (Film::estimate_noise_levels)."""

    def __init__(self, scene_data=None, flavor="fast", device=0, profile=False):
        super().__init__(scene_data, flavor=flavor, device=device, profile=profile)
        self.pt_options = S.default_pt_options()
        self._check(self.lib.etxb_set_integrator(self.h, S.INTEGRATOR_PT))

    @staticmethod
    def name():
        return "Path Tracing (B200)"

    def set_option(self, key, value):
        """The reference's option ids: "direct", "nee", "mis", "bn" (path_tracing.cxx:36-39)."""
        rc = self.lib.etxb_pt_options_set_key(_p(self.pt_options), key.encode(), float(value))
        if rc != 0:
            raise EtxbError(rc, f"unknown option key {key}")

    def set_scene_settings(self, noise_threshold, radiance_clamp=0.0):
        """Scene::noise_threshold / radiance_clamp without a new upload."""
        self._check(self.lib.etxb_set_scene_settings(self.h, C.c_float(noise_threshold), C.c_float(radiance_clamp)))

    def run(self, first_iteration=0):
        """CPUPathTracing::run -> CPUPathTracingImpl::start (path_tracing.cxx:35-48): options, film.clear(ClearCameraData), first task."""
        self._check(self.lib.etxb_pt_set_options(self.h, _p(self.pt_options)))
        self._check(self.lib.etxb_begin(self.h, first_iteration))
        self._running = True
        self._target_iterations = int(self.scene_data.scene["samples"][0])

    def update(self):
        """CPUPathTracingImpl::update (path_tracing.cxx:85-110), non-blocking: an iteration that processed no pixel (all converged) ends the run."""
        if not self._running:
            return False
        st = self.status()
        if st["iteration_in_flight"]:
            return True
        if st["completed_iterations"] and (self.pt_status()["pixels_processed"] == 0):
            self._running = False
            return False
        if st["completed_iterations"] >= self._target_iterations:
            self._running = False
            return False
        self._check(self.lib.etxb_enqueue_iteration(self.h))
        return True

    def pt_status(self):
        st = np.zeros(1, dtype=S.PT_STATUS)
        self._check(self.lib.etxb_pt_get_status(self.h, _p(st)))
        return {k: st[k][0].item() for k in st.dtype.names}


class GPUVCMGroup:
    """Several iterations in flight on one device (etxb_group): `lanes` contexts, one host thread each inside the module, pulling
    iteration indices from a shared counter.  Same Integrator-style surface as GPUVCM: run / enqueue / wait / status / film."""

    def __init__(self, scene_data, lanes=4, flavor="fast", device=0, max_light_vertices=0, profile=False):
        self.lib = load_library(flavor)
        self.h = C.c_void_p()
        cfg = np.zeros(1, dtype=S.DEVICE_CONFIG)
        cfg["device_index"] = device
        cfg["max_light_vertices"] = max_light_vertices
        cfg["flags"] = 1 if profile else 0
        rc = self.lib.etxb_group_create(C.byref(self.h), _p(cfg), lanes)
        if rc != 0:
            raise EtxbError(rc, "etxb_group_create failed (no CUDA device? the module has no CPU fallback)")
        self.lanes = [GPUVCM(scene_data, flavor=flavor, _adopt=self.lib.etxb_group_lane(self.h, k)) for k in range(lanes)]
        self.options = self.lanes[0].options
        self.scene_data = scene_data
        self.width, self.height = self.lanes[0].width, self.lanes[0].height

    def _check(self, rc):
        if rc < 0:
            raise EtxbError(rc, self.lib.etxb_group_last_error(self.h).decode() or self.lib.etxb_last_error(self.lanes[0].h).decode())
        return rc

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            for g in self.lanes:
                g.close()
            self.lib.etxb_group_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_integrator(self, integrator, pt_options=None):
        """Every lane renders with the VCM (default) or the path-tracing algorithm.  With iterations in flight each lane keeps its own film and per-pixel
        history, so the path tracer's adaptive sampling is switched off here (noise threshold 0: every pixel gets one sample per iteration, like the
        reference with `noise_threshold 0`); the combined film is the mean over the iterations of all lanes."""
        for g in self.lanes:
            g._check(self.lib.etxb_set_integrator(g.h, integrator))
            if integrator == S.INTEGRATOR_PT:
                g._check(self.lib.etxb_pt_set_options(g.h, _p(pt_options if pt_options is not None else S.default_pt_options())))
                g._check(self.lib.etxb_set_scene_settings(g.h, C.c_float(0.0), C.c_float(float(self.scene_data.scene["radiance_clamp"][0]))))

    def set_options(self):
        """Pushes self.options (the Integrator options) to every lane."""
        for g in self.lanes:
            g._check(self.lib.etxb_set_options(g.h, _p(self.options)))

    def run(self, first_iteration=0):
        self.set_options()
        self._check(self.lib.etxb_group_begin(self.h, first_iteration))

    def comm_init(self, world, rank, comm_ids):
        """Pixel tiles over `world` processes with len(self.lanes) iterations in flight on each: collective; comm_ids = the (lanes + 1) x 128
        bytes rank 0 got from comm_unique_ids(lanes + 1)."""
        comm_ids = np.ascontiguousarray(comm_ids, dtype=np.uint8)
        self._check(self.lib.etxb_group_comm_init(self.h, world, rank, _p(comm_ids), comm_ids.nbytes // COMM_ID_BYTES))
        self.comm_rank, self.comm_world = rank, world

    def comm_init_replicas(self, world, rank, comm_id, split_lane=False):
        """Whole-frame iterations dealt to `world` processes (the job's j-th iteration on rank j % world); enqueue(n) then counts iterations of
        the job.  Collective; comm_id = the 128 bytes rank 0 got from comm_unique_ids(1).  split_lane: reserve the last lane for camera-split
        iterations (the remainder of an enqueue that is not a multiple of `world`)."""
        if split_lane:
            self._check(self.lib.etxb_group_reserve_split_lane(self.h))
        comm_id = np.ascontiguousarray(comm_id, dtype=np.uint8)
        self._check(self.lib.etxb_group_comm_init_replicas(self.h, world, rank, _p(comm_id), comm_id.nbytes))
        self.comm_rank, self.comm_world = rank, world

    def comm_reduce_film(self, layer=S.FILM_RESULT, out=None):
        """Collective: the whole frame (mean over the iterations finished so far) on rank 0; None elsewhere."""
        rank = getattr(self, "comm_rank", 0)
        if (out is None) and (rank == 0):
            out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._check(self.lib.etxb_group_comm_reduce_film(self.h, layer, _p(out) if rank == 0 else None, out.nbytes if rank == 0 else 0))
        return out if rank == 0 else None

    def set_stride(self, stride):
        """Iteration-interleaved multi-GPU runs: this group renders indices first, first + stride, ..."""
        self._check(self.lib.etxb_group_set_stride(self.h, stride))

    def enqueue(self, iterations=1):
        self._check(self.lib.etxb_group_enqueue(self.h, iterations))

    def combined(self, layer=S.FILM_RESULT):
        """(device pointer, bytes, iterations) of the combined layer, left on the device."""
        ptr, n, done = C.c_void_p(), C.c_uint64(0), C.c_uint32(0)
        self._check(self.lib.etxb_group_combine(self.h, layer, C.byref(ptr), C.byref(n), C.byref(done)))
        return ptr.value, n.value, done.value

    def wait(self):
        self._check(self.lib.etxb_group_wait(self.h))

    def render(self, iterations, first_iteration=0):
        self.run(first_iteration)
        self.enqueue(iterations)
        self.wait()
        return self.status()

    def status(self):
        st = np.zeros(1, dtype=S.STATUS)
        self._check(self.lib.etxb_group_poll(self.h, _p(st)))
        return {k: st[k][0].item() for k in st.dtype.names}

    def film(self, layer=S.FILM_RESULT, out=None):
        if out is None:
            out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._check(self.lib.etxb_group_read_film(self.h, layer, _p(out), out.nbytes))
        return out

    def counters(self):
        total = {}
        for g in self.lanes:
            for k, v in g.counters().items():
                total[k] = total.get(k, 0) + v
        return total

    def kernel_times(self):
        total = {}
        for g in self.lanes:
            for k, (ms, n) in g.kernel_times().items():
                a = total.get(k, (0.0, 0))
                total[k] = (a[0] + ms, a[1] + n)
        return total
