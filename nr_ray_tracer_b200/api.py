"""Python host mirror of the reference's render API over the C ABI (include/nrrt.h).

Reference interface mirrored here (names and meaning kept):
  Scene { camera, objects }  / Scene::render(progress) -> Rgb32FImage   ray-tracer-lib/src/scene.rs:7-18
  Camera::render(hitable, progress)                                      ray-tracer-lib/src/camera.rs:302-343
  SceneConfig::try_load_scene / try_build                                ray-tracer/src/scene_config.rs:475-496

Everything that computes runs in libnrrt_b200.so (CUDA, sm_100a).  There is no CPU fallback: if the
library or a GPU is missing, calls raise NrrtError.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Callable, Optional

import numpy as np

from . import _abi as A
from .scene_config import CameraConfig, SceneGraph, load_scene

# NRRT_B200_LIB lets a developer point at an experimental build of the SAME library (never at another backend)
_LIB_PATH = os.environ.get("NRRT_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                            "libnrrt_b200.so")
_lib = None


class NrrtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"nrrt error {code}: {msg}")
        self.code = code


def lib() -> C.CDLL:
    """Loads the native library; never falls back to anything else."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise NrrtError(A.ERR_NO_DEVICE, f"{_LIB_PATH} is not built (run `python -m nr_ray_tracer_b200.build`); "
                                             "there is no CPU fallback")
        L = C.CDLL(_LIB_PATH)
        L.nrrt_host_build.restype = C.c_void_p
        L.nrrt_host_build.argtypes = [C.POINTER(A.GraphDesc)]
        L.nrrt_host_build_ex.restype = C.c_void_p
        L.nrrt_host_build_ex.argtypes = [C.POINTER(A.GraphDesc), C.c_uint32]
        L.nrrt_host_scene_desc.restype = C.POINTER(A.SceneDesc)
        L.nrrt_host_scene_desc.argtypes = [C.c_void_p]
        L.nrrt_host_free.argtypes = [C.c_void_p]
        L.nrrt_host_last_error.restype = C.c_char_p
        L.nrrt_host_camera_build.argtypes = [C.POINTER(A.CameraConfig), C.POINTER(A.Camera)]
        L.nrrt_load_scene.restype = C.c_void_p
        L.nrrt_load_scene.argtypes = [C.c_char_p, C.c_char_p]
        L.nrrt_loaded_graph.restype = C.POINTER(A.GraphDesc)
        L.nrrt_loaded_graph.argtypes = [C.c_void_p]
        L.nrrt_loaded_camera.argtypes = [C.c_void_p, C.POINTER(A.CameraFile)]
        L.nrrt_loaded_free.argtypes = [C.c_void_p]
        L.nrrt_load_last_error.restype = C.c_char_p
        L.nrrt_camera_file_merge.argtypes = [C.POINTER(A.CameraFile), C.POINTER(A.CameraFile)]
        L.nrrt_camera_file_to_config.argtypes = [C.POINTER(A.CameraFile), C.POINTER(A.CameraConfig)]
        L.nrrt_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.nrrt_destroy.argtypes = [C.c_void_p]
        L.nrrt_last_error.restype = C.c_char_p
        L.nrrt_last_error.argtypes = [C.c_void_p]
        L.nrrt_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.nrrt_set_trace_time.argtypes = [C.c_void_p, C.c_double]
        L.nrrt_scene_upload.argtypes = [C.c_void_p, C.POINTER(A.SceneDesc)]
        L.nrrt_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_uint32,
                                      C.c_void_p, C.POINTER(A.TraceStats)]
        L.nrrt_render.argtypes = [C.c_void_p, C.POINTER(A.Camera), C.POINTER(A.RenderOpts), C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.POINTER(A.RenderStats)]
        L.nrrt_encode_rgb8.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_uint32, C.c_void_p]
        L.nrrt_render_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(A.SceneDesc), C.POINTER(A.Camera),
                                        C.POINTER(A.RenderOpts), C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(A.RenderStats), C.c_char_p, C.c_size_t]
        L.nrrt_chunk_starts.restype = C.c_uint32
        L.nrrt_chunk_starts.argtypes = [C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32), C.c_uint32]
        L.nrrt_work_items.restype = C.c_uint32
        L.nrrt_work_items.argtypes = [C.c_uint32] * 8 + [C.POINTER(C.c_uint32)]
        L.nrrt_pass_items.restype = C.c_uint32
        L.nrrt_pass_items.argtypes = [C.c_uint32] * 10 + [C.POINTER(C.c_uint32)]
        L.nrrt_accum_create.argtypes = [C.c_void_p, C.POINTER(A.Camera), C.POINTER(A.RenderOpts), C.POINTER(C.c_void_p)]
        L.nrrt_accum_render.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(A.RenderStats)]
        L.nrrt_accum_samples.restype = C.c_uint32
        L.nrrt_accum_samples.argtypes = [C.c_void_p]
        L.nrrt_accum_image.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.nrrt_accum_save.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
        L.nrrt_accum_restore.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.nrrt_accum_free.argtypes = [C.c_void_p]
        L.nrrt_abi_sizeof.restype = C.c_size_t
        L.nrrt_abi_sizeof.argtypes = [C.c_int]
        _lib = L
    return _lib


ABI_STRUCTS = [A.Object, A.Material, A.Texture, A.Image, A.GraphDesc, A.CameraConfig, A.Camera, A.Node, A.Box,
               A.Xform, A.Instance, A.SceneDesc, A.Hit, A.TraceStats, A.RenderOpts, A.RenderStats, A.CameraFile, A.WNode,
               A.HitCompact]


def chunk_starts(samples_per_pixel: int, total_pixels: int):
    """First sample of every work-item chunk of a pixel, and spp as the last entry (nrrt_chunk_starts)."""
    buf = (C.c_uint32 * 64)()
    n = lib().nrrt_chunk_starts(samples_per_pixel, total_pixels, buf, 64)
    return [int(buf[i]) for i in range(n + 1)]


def work_items(width: int, height: int, samples_per_pixel: int, rank: int = 0, world: int = 1,
               rows_per_block: int = 8) -> np.ndarray:
    """All work items of one rank's render in hand-out order, (n_items, 4) uint32: x, y, first sample, end sample
    (nrrt_work_items: the kernels' own decode, run on the host)."""
    n = lib().nrrt_work_items(width, height, samples_per_pixel, rank, world, rows_per_block, 0, 0, None)
    out = np.zeros((n, 4), dtype=np.uint32)
    if n:
        lib().nrrt_work_items(width, height, samples_per_pixel, rank, world, rows_per_block, 0, n,
                              out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return out


def pass_items(width: int, height: int, samples_per_pixel: int, c0: int, c1: int, rank: int = 0, world: int = 1,
               rows_per_block: int = 8) -> np.ndarray:
    """The work items of one progressive pass over chunks [c0, c1) in hand-out order, (n_items, 4) uint32 as in
    work_items (nrrt_pass_items: the kernels' decode with the pass's chunk offset, run on the host)."""
    args = (width, height, samples_per_pixel, rank, world, rows_per_block, c0, c1)
    n = lib().nrrt_pass_items(*args, 0, 0, None)
    out = np.zeros((n, 4), dtype=np.uint32)
    if n:
        lib().nrrt_pass_items(*args, 0, n, out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return out


def owned_rows(height: int, rank: int = 0, world: int = 1, rows_per_block: int = 0) -> int:
    """Rows rank `rank` of `world` renders: row-blocks b with b % world == rank (rows_per_block 0 -> 8)."""
    R = rows_per_block or 8
    return sum(min(R, height - b * R) for b in range(rank, (height + R - 1) // R, world))


_STATS = ("paths", "segments", "launches", "device_ms", "extend_ms", "extend_launches", "pixels", "mode", "node_visits",
          "box_exact", "prim_tests", "inst_entries", "inst_misses")


def camera_build(cfg: A.CameraConfig) -> A.Camera:
    """CameraBuilder::build (camera.rs:94-159) on the host."""
    cam = A.Camera()
    rc = lib().nrrt_host_camera_build(C.byref(cfg), C.byref(cam))
    if rc != 0:
        raise NrrtError(rc, "nrrt_host_camera_build: bad configuration")
    return cam


class NativeScene:
    """Scene file loaded by the native C++ loader (csrc/scene_loader.cpp): graph description + [camera] section."""

    def __init__(self, path: str, base_dir: Optional[str] = None):
        self._h = lib().nrrt_load_scene(path.encode(), base_dir.encode() if base_dir else None)
        if not self._h:
            raise NrrtError(A.ERR_IO, lib().nrrt_load_last_error().decode())
        self.graph = lib().nrrt_loaded_graph(self._h).contents
        self.camera_file = A.CameraFile()
        lib().nrrt_loaded_camera(self._h, C.byref(self.camera_file))

    def camera_config(self, override: Optional[A.CameraFile] = None) -> A.CameraConfig:
        """merge_with(override) then try_update onto the CameraBuilder defaults."""
        merged = A.CameraFile.from_buffer_copy(bytes(self.camera_file))
        if override is not None:
            lib().nrrt_camera_file_merge(C.byref(merged), C.byref(override))
        cfg = A.CameraConfig()
        rc = lib().nrrt_camera_file_to_config(C.byref(merged), C.byref(cfg))
        if rc != 0:
            raise NrrtError(rc, "image size needs exactly two of width / height / aspect ratio")
        return cfg

    def close(self):
        if getattr(self, "_h", None):
            lib().nrrt_loaded_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostScene:
    """Object graph -> reference BVH (objects/object.rs:41-73) -> flat device layout.  Pure host code."""

    def __init__(self, graph, bvh: str = "reference"):
        """graph: a SceneGraph (Python loader) or a NativeScene (C++ loader).
        bvh: "reference" = the reference's tree node for node (parity contract); "sah" = opt-in binned-SAH inner
        nodes over the same leaves and leaf order (NRRT_BUILD_SAH, include/nrrt.h)."""
        if bvh not in ("reference", "sah"):
            raise ValueError("bvh must be 'reference' or 'sah'")
        flags = A.BUILD_SAH if bvh == "sah" else A.BUILD_REFERENCE
        if isinstance(graph, NativeScene):
            self._holder = graph
            self._h = lib().nrrt_host_build_ex(C.byref(graph.graph), flags)
        else:
            self._holder = graph.to_desc()
            self._h = lib().nrrt_host_build_ex(self._holder.ptr(), flags)
        if not self._h:
            raise NrrtError(A.ERR_INVALID, lib().nrrt_host_last_error().decode())
        self.desc = lib().nrrt_host_scene_desc(self._h).contents

    def close(self):
        if getattr(self, "_h", None):
            lib().nrrt_host_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # numpy views for tests / inspection
    def nodes(self) -> np.ndarray:
        n = self.desc.n_nodes
        dt = np.dtype([("lo", "<f4", (2, 3)), ("hi", "<f4", (2, 3)), ("child", "<u4", (2,)), ("_pad", "<u4", (2,))])
        if n == 0:
            return np.zeros(0, dtype=dt)
        return np.ctypeslib.as_array(C.cast(self.desc.nodes, C.POINTER(C.c_uint8)), shape=(n * 64,)).view(dt).copy()

    def child_boxes(self) -> np.ndarray:
        n = self.desc.n_nodes
        if n == 0:
            return np.zeros((0, 2, 2, 3))
        a = np.ctypeslib.as_array(C.cast(self.desc.child_boxes, C.POINTER(C.c_double)), shape=(n, 2, 2, 3))
        return a.copy()

    def wnodes(self) -> np.ndarray:
        """The four-slot traversal nodes the kernels walk (nrrt_wnode)."""
        n = self.desc.n_wnodes
        dt = np.dtype([("lo", "<f4", (3, 4)), ("hi", "<f4", (3, 4)), ("child", "<u4", (4,)), ("meta", "<u4", (4,))])
        if n == 0:
            return np.zeros(0, dtype=dt)
        return np.ctypeslib.as_array(C.cast(self.desc.wnodes, C.POINTER(C.c_uint8)), shape=(n * 128,)).view(dt).copy()

    def wide_boxes(self) -> np.ndarray:
        """(n_wnodes, 4 slots, own / gate, lo / hi, 3) exact f64 boxes."""
        n = self.desc.n_wnodes
        if n == 0:
            return np.zeros((0, 4, 2, 2, 3))
        a = np.ctypeslib.as_array(C.cast(self.desc.wide_boxes, C.POINTER(C.c_double)), shape=(n, 4, 2, 2, 3))
        return a.copy()

    def instance_wide_inner(self) -> np.ndarray:
        n = self.desc.n_instances
        if n == 0:
            return np.zeros(0, dtype=np.uint32)
        return np.ctypeslib.as_array(self.desc.instance_wide_inner, shape=(n,)).copy()


class Context:
    """One GPU context (one process per GPU).  Owns all device memory."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        rc = lib().nrrt_create(device, C.byref(h))
        if rc != 0:
            raise NrrtError(rc, lib().nrrt_last_error(None).decode())
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            lib().nrrt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise NrrtError(rc, lib().nrrt_last_error(self._h).decode())

    def set_stream(self, cuda_stream: int):
        self._check(lib().nrrt_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_trace_time(self, time: float):
        """Ray::time of the rays given to trace_rays (ray.rs:8); only moving spheres read it."""
        self._check(lib().nrrt_set_trace_time(self._h, float(time)))

    def upload(self, scene: HostScene):
        self._check(lib().nrrt_scene_upload(self._h, C.byref(scene.desc)))

    def trace_rays(self, rays: np.ndarray, tmin: float = 0.001, tmax: float = float("inf"), visit_all: bool = False,
                   want_stats: bool = True):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        out = np.zeros(rays.shape[0], dtype=A.HIT_DTYPE)
        st = A.TraceStats()
        flags = (A.TRACE_VISIT_ALL if visit_all else A.TRACE_ORDERED) | (A.TRACE_COUNT if want_stats else 0)
        self._check(lib().nrrt_trace_rays(self._h, rays.ctypes.data, rays.shape[0], tmin, tmax, flags, out.ctypes.data,
                                          C.byref(st) if want_stats else None))
        return out, {"node_visits": st.node_visits, "box_exact": st.box_exact, "prim_tests": st.prim_tests,
                     "kernel_ms": st.kernel_ms}

    def trace_rays_device(self, rays_ptr: int, n: int, out_ptr: int, tmin: float = 0.001, tmax: float = float("inf"),
                          visit_all: bool = False, count: bool = False, compact: bool = False):
        """rays_ptr / out_ptr are device pointers (n x 6 f64, n x nrrt_hit — or n x 16-byte nrrt_hit_compact with
        compact=True: the closest-hit query alone, no HitRecord)."""
        st = A.TraceStats()
        flags = (A.TRACE_VISIT_ALL if visit_all else A.TRACE_ORDERED) | A.TRACE_DEVICE_BUFFERS | \
            (A.TRACE_COUNT if count else 0) | (A.TRACE_COMPACT if compact else 0)
        self._check(lib().nrrt_trace_rays(self._h, C.c_void_p(rays_ptr), n, tmin, tmax, flags, C.c_void_p(out_ptr),
                                          C.byref(st)))
        return {"node_visits": st.node_visits, "box_exact": st.box_exact, "prim_tests": st.prim_tests,
                "kernel_ms": st.kernel_ms}

    def render(self, cam: A.Camera, out: Optional[np.ndarray] = None, seed: int = 0, mode: int = A.MODE_AUTO,
               rank: int = 0, world: int = 1, rows_per_block: int = 0, max_slots: int = 0,
               out_device_ptr: Optional[int] = None, progress: Optional[Callable[[int, int], None]] = None,
               count: bool = False, packed: bool = False):
        """Camera::render.  Returns (image (H, W, 3) float32 or None for device output, stats dict).
        packed=True: the output buffer holds only this rank's rows, packed (NRRT_RENDER_OUT_PACKED)."""
        opts = A.RenderOpts(seed=seed, mode=mode, rank=rank, world=world, rows_per_block=rows_per_block,
                            max_slots=max_slots, flags=(A.RENDER_OUT_DEVICE if out_device_ptr is not None else 0) |
                            (A.RENDER_COUNT if count else 0) | (A.RENDER_OUT_PACKED if packed else 0))
        st = A.RenderStats()
        cb = A.PROGRESS_FN(lambda done, total, user: progress(done, total)) if progress else None
        if out_device_ptr is not None:
            ptr = C.c_void_p(out_device_ptr)
        else:
            if out is None:
                out = np.zeros((cam.height, cam.width, 3), dtype=np.float32)
            assert out.dtype == np.float32 and out.flags.c_contiguous and (packed or out.size == cam.height * cam.width * 3)
            ptr = C.c_void_p(out.ctypes.data)
        self._check(lib().nrrt_render(self._h, C.byref(cam), C.byref(opts), ptr, C.cast(cb, C.c_void_p) if cb else None,
                                      None, C.byref(st)))
        stats = {k: getattr(st, k) for k in _STATS}
        return (None if out_device_ptr is not None else out), stats

    def progressive(self, cam: A.Camera, seed: int = 0, mode: int = A.MODE_AUTO, rank: int = 0, world: int = 1,
                    rows_per_block: int = 0, max_slots: int = 0) -> "Progressive":
        """One frame of `cam` rendered in passes (nrrt_accum_*): see Progressive."""
        return Progressive(self, cam, seed=seed, mode=mode, rank=rank, world=world, rows_per_block=rows_per_block,
                           max_slots=max_slots)


    def encode_rgb8(self, image: Optional[np.ndarray] = None, gamma: float = 0.5, device_ptr: Optional[int] = None,
                    width: int = 0, height: int = 0) -> np.ndarray:
        """gamma_correction + to_rgb8 (render.rs:83-87) on the GPU -> (H, W, 3) uint8.  Default gamma 0.5 is the
        CLI's DEFAULT_IMAGE_GAMMA_VALUE (constants.rs:1)."""
        if device_ptr is not None:
            h, w, ptr, flags = height, width, C.c_void_p(device_ptr), A.RENDER_OUT_DEVICE
        else:
            image = np.ascontiguousarray(image, dtype=np.float32)
            h, w = image.shape[0], image.shape[1]
            ptr, flags = C.c_void_p(image.ctypes.data), 0
        out = np.zeros((h, w, 3), dtype=np.uint8)
        self._check(lib().nrrt_encode_rgb8(self._h, ptr, w, h, gamma, flags, C.c_void_p(out.ctypes.data)))
        return out


class Progressive:
    """A frame rendered in passes of whole work chunks, summed on the GPU into per-pixel f64 sums (nrrt_accum_*).

    render(min_samples) renders the next chunks until at least that many samples per pixel are done (pass boundaries
    are chunk_starts() boundaries); image() is the frame so far, sums / samples.  The finished frame is
    Context.render's image bit for bit, whatever the passes.  state() / restore() save and resume the sums.
    Keeps its Context alive; the scene must stay the one uploaded when the frame was created."""

    def __init__(self, ctx: Context, cam: A.Camera, seed: int = 0, mode: int = A.MODE_AUTO, rank: int = 0,
                 world: int = 1, rows_per_block: int = 0, max_slots: int = 0):
        self.ctx = ctx
        self.camera = cam
        self.samples_per_pixel = max(1, cam.samples_per_pixel)
        self.rows = owned_rows(cam.height, rank, world, rows_per_block)
        opts = A.RenderOpts(seed=seed, mode=mode, rank=rank, world=world, rows_per_block=rows_per_block,
                            max_slots=max_slots, flags=0)
        h = C.c_void_p()
        ctx._check(lib().nrrt_accum_create(ctx._h, C.byref(cam), C.byref(opts), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().nrrt_accum_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def samples(self) -> int:
        """Samples per pixel done so far."""
        return int(lib().nrrt_accum_samples(self._h))

    def render(self, min_samples: int) -> dict:
        """One pass: the next whole chunks until at least min(min_samples, spp) samples are done.  Returns its stats."""
        st = A.RenderStats()
        self.ctx._check(lib().nrrt_accum_render(self._h, min(int(min_samples), self.samples_per_pixel), C.byref(st)))
        return {k: getattr(st, k) for k in _STATS}

    def image(self, out: Optional[np.ndarray] = None, packed: bool = False,
              out_device_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        """The frame so far as linear f32 RGB, laid out as Context.render lays it out (full image with this rank's rows
        written, or packed=True: this rank's rows only).  None for device output."""
        flags = (A.RENDER_OUT_DEVICE if out_device_ptr is not None else 0) | (A.RENDER_OUT_PACKED if packed else 0)
        if out_device_ptr is not None:
            ptr = C.c_void_p(out_device_ptr)
        else:
            if out is None:
                out = np.zeros((self.rows if packed else self.camera.height, self.camera.width, 3), dtype=np.float32)
            assert out.dtype == np.float32 and out.flags.c_contiguous
            assert out.size == (self.rows if packed else self.camera.height) * self.camera.width * 3
            ptr = C.c_void_p(out.ctypes.data)
        self.ctx._check(lib().nrrt_accum_image(self._h, ptr, flags))
        return None if out_device_ptr is not None else out

    def state(self):
        """(samples done, f64 sums (owned rows, W, 3) in owned-row order): what restore() takes."""
        sums = np.zeros((self.rows, self.camera.width, 3), dtype=np.float64)
        n = C.c_uint32()
        self.ctx._check(lib().nrrt_accum_save(self._h, C.c_void_p(sums.ctypes.data), C.byref(n)))
        return int(n.value), sums

    def restore(self, samples: int, sums: np.ndarray):
        """Resumes from state(): `samples` must be a chunk boundary of this frame."""
        sums = np.ascontiguousarray(sums, dtype=np.float64)
        if sums.size != self.rows * self.camera.width * 3:
            raise ValueError(f"sums must hold {self.rows} x {self.camera.width} x 3 values")
        self.ctx._check(lib().nrrt_accum_restore(self._h, C.c_void_p(sums.ctypes.data), int(samples)))


def render_multi(devices, host_scene: "HostScene", cam: A.Camera, out: Optional[np.ndarray] = None, seed: int = 0,
                 mode: int = A.MODE_AUTO, out_device_ptr: Optional[int] = None):
    """Camera::render over several GPUs of one box from this one process (nrrt_render_multi): rows interleaved over
    `devices`, brought together inside the library (host image: parallel D2H copies; device image on devices[0]:
    peer-to-peer copies + one placement kernel).  Returns (image or None, stats summed over the devices)."""
    devs = (C.c_int * len(devices))(*devices)
    opts = A.RenderOpts(seed=seed, mode=mode, flags=A.RENDER_OUT_DEVICE if out_device_ptr is not None else 0)
    st = A.RenderStats()
    if out_device_ptr is not None:
        ptr = C.c_void_p(out_device_ptr)
    else:
        if out is None:
            out = np.zeros((cam.height, cam.width, 3), dtype=np.float32)
        ptr = C.c_void_p(out.ctypes.data)
    err = C.create_string_buffer(512)
    rc = lib().nrrt_render_multi(devs, len(devices), C.byref(host_scene.desc), C.byref(cam), C.byref(opts), ptr, None, None,
                                 C.byref(st), err, 512)
    if rc != 0:
        raise NrrtError(rc, err.value.decode())
    stats = {k: getattr(st, k) for k in ("paths", "segments", "launches", "device_ms", "pixels", "mode")}
    return (None if out_device_ptr is not None else out), stats


class Scene:
    """Drop-in for the reference's Scene (scene.rs:7-18): `Scene.load(path).render()`."""

    def __init__(self, graph: SceneGraph, device: int = 0, ctx: Optional[Context] = None, bvh: str = "reference"):
        self.graph = graph
        self.camera = camera_build(graph.camera.to_builder_config())
        self.host = HostScene(graph, bvh=bvh)
        self.ctx = ctx or Context(device)
        self.ctx.upload(self.host)

    @classmethod
    def load(cls, path: str, camera_override: Optional[CameraConfig] = None, base_dir: Optional[str] = None,
             device: int = 0, ctx: Optional[Context] = None, bvh: str = "reference") -> "Scene":
        """SceneConfig::try_load_scene + camera merge + try_build (render.rs:104-111)."""
        return cls(load_scene(path, base_dir=base_dir, camera_override=camera_override), device=device, ctx=ctx,
                   bvh=bvh)

    def render(self, progress: Optional[Callable[[int, int], None]] = None, **kw) -> np.ndarray:
        """Scene::render -> linear f32 RGB image (H, W, 3), no gamma, no clamp."""
        img, self.last_stats = self.ctx.render(self.camera, progress=progress, **kw)
        return img

    def render_progressive(self, every: Optional[int] = None, **kw):
        """Scene::render in passes: yields (samples done, image so far) after each pass.  every=None: one pass per work
        chunk; every=N: passes up to the next multiple of N samples (rounded up to a chunk boundary).  The last image
        yielded is render()'s.  kw: Context.progressive's options (seed, mode, ...)."""
        if every is not None and every < 1:
            raise ValueError("every must be >= 1")
        with self.ctx.progressive(self.camera, **kw) as p:
            while p.samples < p.samples_per_pixel:
                done = p.samples
                self.last_stats = p.render(done + 1 if every is None else (done // every + 1) * every)
                yield p.samples, p.image()
