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
        L.nrrt_accum_create_adaptive.argtypes = [C.c_void_p, C.POINTER(A.Camera), C.POINTER(A.RenderOpts),
                                                 C.POINTER(A.AdaptiveOpts), C.POINTER(C.c_void_p)]
        L.nrrt_accum_active.restype = C.c_uint32
        L.nrrt_accum_active.argtypes = [C.c_void_p]
        L.nrrt_accum_sample_map.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.nrrt_accum_error_image.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.nrrt_accum_adaptive_save.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.nrrt_accum_adaptive_restore.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.nrrt_adaptive_converged.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                              C.POINTER(A.AdaptiveOpts)]
        L.nrrt_pass_items_active.restype = C.c_uint32
        L.nrrt_pass_items_active.argtypes = [C.c_uint32] * 8 + [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                                                 C.POINTER(C.c_uint32)]
        L.nrrt_accum_aov.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32]
        L.nrrt_accum_denoise.argtypes = [C.c_void_p, C.POINTER(A.DenoiseOpts), C.c_void_p, C.c_uint32]
        L.nrrt_abi_sizeof.restype = C.c_size_t
        L.nrrt_abi_sizeof.argtypes = [C.c_int]
        _lib = L
    return _lib


ABI_STRUCTS = [A.Object, A.Material, A.Texture, A.Image, A.GraphDesc, A.CameraConfig, A.Camera, A.Node, A.Box,
               A.Xform, A.Instance, A.SceneDesc, A.Hit, A.TraceStats, A.RenderOpts, A.RenderStats, A.CameraFile, A.WNode,
               A.HitCompact, A.AdaptiveOpts, A.DenoiseOpts]


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


def pass_items_active(width: int, height: int, samples_per_pixel: int, c0: int, c1: int, active, rank: int = 0,
                      world: int = 1, rows_per_block: int = 8) -> np.ndarray:
    """pass_items for an adaptive pass over the owned pixels listed in `active` (owned-pixel indices, i.e. positions in
    a chunk of pass_items, strictly ascending) in hand-out order (nrrt_pass_items_active)."""
    act = np.ascontiguousarray(active, dtype=np.uint32)
    args = (width, height, samples_per_pixel, rank, world, rows_per_block, c0, c1, C.c_void_p(act.ctypes.data), len(act))
    n = lib().nrrt_pass_items_active(*args, 0, 0, None)
    out = np.zeros((n, 4), dtype=np.uint32)
    if n:
        lib().nrrt_pass_items_active(*args, 0, n, out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return out


def adaptive_opts(rel_error: float, abs_error: float = 0.0, min_samples: int = 0) -> A.AdaptiveOpts:
    return A.AdaptiveOpts(rel_error=float(rel_error), abs_error=float(abs_error), min_samples=int(min_samples))


def adaptive_converged(S, Q, samples: int, chunks: int, rel_error: float, abs_error: float = 0.0,
                       min_samples: int = 0) -> bool:
    """The adaptive test on one pixel's state (nrrt_adaptive_converged): S and Q are its 3 f64 sums."""
    S = np.ascontiguousarray(S, dtype=np.float64)
    Q = np.ascontiguousarray(Q, dtype=np.float64)
    assert S.size == 3 and Q.size == 3
    t = adaptive_opts(rel_error, abs_error, min_samples)
    return bool(lib().nrrt_adaptive_converged(S.ctypes.data, Q.ctypes.data, int(samples), int(chunks), C.byref(t)))


def default_min_samples(samples_per_pixel: int, total_pixels: int) -> int:
    """The first chunk boundary at or above spp / 8: where an adaptive frame starts testing pixels by default."""
    starts = chunk_starts(samples_per_pixel, total_pixels)
    return min(s for s in starts if 8 * s >= max(1, samples_per_pixel))


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
                    rows_per_block: int = 0, max_slots: int = 0, adaptive: Optional[dict] = None) -> "Progressive":
        """One frame of `cam` rendered in passes (nrrt_accum_*): see Progressive.  adaptive = {rel_error, abs_error=0.0,
        min_samples=None} makes it an adaptive frame (min_samples None: the first chunk boundary at or above spp / 8)."""
        return Progressive(self, cam, seed=seed, mode=mode, rank=rank, world=world, rows_per_block=rows_per_block,
                           max_slots=max_slots, adaptive=adaptive)


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
    Keeps its Context alive; the scene must stay the one uploaded when the frame was created.

    An adaptive frame (adaptive={rel_error, abs_error, min_samples}) renders each pass for the pixels still active only
    and retires a pixel once its error estimate meets the tolerance (include/nrrt.h): `active` counts the pixels left,
    sample_map() and error_image() show each pixel's samples and estimated error, image() divides each pixel by its
    own sample count, and state() / restore() carry (sums, sums of squares, samples)."""

    def __init__(self, ctx: Context, cam: A.Camera, seed: int = 0, mode: int = A.MODE_AUTO, rank: int = 0,
                 world: int = 1, rows_per_block: int = 0, max_slots: int = 0, adaptive: Optional[dict] = None):
        self.ctx = ctx
        self.camera = cam
        self.samples_per_pixel = max(1, cam.samples_per_pixel)
        self.rows = owned_rows(cam.height, rank, world, rows_per_block)
        opts = A.RenderOpts(seed=seed, mode=mode, rank=rank, world=world, rows_per_block=rows_per_block,
                            max_slots=max_slots, flags=0)
        h = C.c_void_p()
        self.adaptive = None
        if adaptive is None:
            ctx._check(lib().nrrt_accum_create(ctx._h, C.byref(cam), C.byref(opts), C.byref(h)))
        else:
            unknown = set(adaptive) - {"rel_error", "abs_error", "min_samples"}
            if unknown or "rel_error" not in adaptive:
                raise ValueError("adaptive takes rel_error and optionally abs_error and min_samples")
            ms = adaptive.get("min_samples")
            if ms is None:
                ms = default_min_samples(self.samples_per_pixel, cam.width * cam.height)
            self.adaptive = adaptive_opts(adaptive["rel_error"], adaptive.get("abs_error", 0.0), ms)
            ctx._check(lib().nrrt_accum_create_adaptive(ctx._h, C.byref(cam), C.byref(opts), C.byref(self.adaptive),
                                                        C.byref(h)))
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

    @property
    def active(self) -> int:
        """Pixels of an adaptive frame still active (0: the frame is finished); 0 for a plain progressive frame."""
        return int(lib().nrrt_accum_active(self._h))

    def _map(self, fn, shape, dtype, packed, out_device_ptr):
        flags = (A.RENDER_OUT_DEVICE if out_device_ptr is not None else 0) | (A.RENDER_OUT_PACKED if packed else 0)
        if out_device_ptr is not None:
            self.ctx._check(fn(self._h, C.c_void_p(out_device_ptr), flags))
            return None
        out = np.zeros(((self.rows if packed else self.camera.height), self.camera.width) + shape, dtype=dtype)
        self.ctx._check(fn(self._h, C.c_void_p(out.ctypes.data), flags))
        return out

    def sample_map(self, packed: bool = False, out_device_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        """Samples each pixel of an adaptive frame holds, (H, W) uint32 laid out as image()."""
        return self._map(lib().nrrt_accum_sample_map, (), np.uint32, packed, out_device_ptr)

    def error_image(self, packed: bool = False, out_device_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        """Estimated standard error of each pixel's mean per channel, (H, W, 3) f32 laid out as image(); +inf where a
        pixel holds fewer than two chunks."""
        return self._map(lib().nrrt_accum_error_image, (3,), np.float32, packed, out_device_ptr)

    def aov(self, samples: Optional[int] = None, packed: bool = False, out_device_ptr: Optional[int] = None):
        """Denoising guides: the mean first-hit albedo and normal of each pixel's first `samples` samples (None:
        min(spp, 16)), (albedo, normal) as (H, W, 3) f32 laid out as image().  out_device_ptr: two device buffers
        (albedo, normal) of that size; returns None then.  Computed once per sample count and kept by the frame."""
        n = 0 if samples is None else int(samples)
        if samples is not None and n < 1:
            raise ValueError("samples must be >= 1")
        flags = (A.RENDER_OUT_DEVICE if out_device_ptr is not None else 0) | (A.RENDER_OUT_PACKED if packed else 0)
        if out_device_ptr is not None:
            pa, pn = out_device_ptr
            self.ctx._check(lib().nrrt_accum_aov(self._h, n, C.c_void_p(pa), C.c_void_p(pn), flags))
            return None
        shape = ((self.rows if packed else self.camera.height), self.camera.width, 3)
        albedo, normal = np.zeros(shape, np.float32), np.zeros(shape, np.float32)
        self.ctx._check(lib().nrrt_accum_aov(self._h, n, C.c_void_p(albedo.ctypes.data), C.c_void_p(normal.ctypes.data),
                                             flags))
        return albedo, normal

    def denoised(self, iterations: int = 5, sigma_color: float = 4.0, aov_samples: Optional[int] = None,
                 out: Optional[np.ndarray] = None, out_device_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        """The frame so far through the a-trous filter (nrrt_accum_denoise): (H, W, 3) f32, or None for device output.
        Needs an adaptive frame (its per-pixel error estimate guides the filter) on one GPU (world == 1)."""
        if not 1 <= int(iterations) <= 8:
            raise ValueError("iterations must be 1..8")
        if not (np.isfinite(sigma_color) and sigma_color > 0):
            raise ValueError("sigma_color must be finite and > 0")
        if aov_samples is not None and int(aov_samples) < 1:
            raise ValueError("aov_samples must be >= 1")
        opts = A.DenoiseOpts(iterations=int(iterations), aov_samples=0 if aov_samples is None else int(aov_samples),
                             sigma_color=float(sigma_color))
        if out_device_ptr is not None:
            self.ctx._check(lib().nrrt_accum_denoise(self._h, C.byref(opts), C.c_void_p(out_device_ptr),
                                                     A.RENDER_OUT_DEVICE))
            return None
        if out is None:
            out = np.zeros((self.camera.height, self.camera.width, 3), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == self.camera.height * self.camera.width * 3
        self.ctx._check(lib().nrrt_accum_denoise(self._h, C.byref(opts), C.c_void_p(out.ctypes.data), 0))
        return out

    def state(self):
        """What restore() takes: (samples done, f64 sums (owned rows, W, 3) in owned-row order), or for an adaptive
        frame (sums, sums of squares (owned rows, W, 3) f64, samples (owned rows, W) uint32)."""
        sums = np.zeros((self.rows, self.camera.width, 3), dtype=np.float64)
        if self.adaptive is not None:
            sumsq = np.zeros_like(sums)
            samples = np.zeros((self.rows, self.camera.width), dtype=np.uint32)
            self.ctx._check(lib().nrrt_accum_adaptive_save(self._h, C.c_void_p(sums.ctypes.data),
                                                           C.c_void_p(sumsq.ctypes.data),
                                                           C.c_void_p(samples.ctypes.data)))
            return sums, sumsq, samples
        n = C.c_uint32()
        self.ctx._check(lib().nrrt_accum_save(self._h, C.c_void_p(sums.ctypes.data), C.byref(n)))
        return int(n.value), sums

    def restore(self, *state):
        """Resumes from state(): restore(samples, sums), where `samples` must be a chunk boundary of this frame, or for
        an adaptive frame restore(sums, sumsq, samples)."""
        npx = self.rows * self.camera.width
        if self.adaptive is not None:
            sums, sumsq, samples = state
            sums = np.ascontiguousarray(sums, dtype=np.float64)
            sumsq = np.ascontiguousarray(sumsq, dtype=np.float64)
            samples = np.ascontiguousarray(samples, dtype=np.uint32)
            if sums.size != npx * 3 or sumsq.size != npx * 3 or samples.size != npx:
                raise ValueError(f"sums and sumsq must hold {self.rows} x {self.camera.width} x 3 values and samples "
                                 f"{self.rows} x {self.camera.width}")
            self.ctx._check(lib().nrrt_accum_adaptive_restore(self._h, C.c_void_p(sums.ctypes.data),
                                                              C.c_void_p(sumsq.ctypes.data),
                                                              C.c_void_p(samples.ctypes.data)))
            return
        samples, sums = state
        sums = np.ascontiguousarray(sums, dtype=np.float64)
        if sums.size != npx * 3:
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

    def render_adaptive(self, rel_error: float, abs_error: float = 0.0, min_samples: Optional[int] = None,
                        every: Optional[int] = None, **kw):
        """Scene::render with adaptive sampling: each pixel stops once its estimated standard error is at most
        abs_error + rel_error * |its mean| (see Progressive).  Yields (samples done, pixels still active, image so far)
        after each pass; the last image is the finished frame.  every=None: passes end at doubling chunk counts from
        the first chunk boundary at or above min_samples (each pass ends in a drain of the GPU, so few passes are
        cheaper); every=N: as in render_progressive.  kw: Context.progressive's options (seed, mode, ...)."""
        if every is not None and every < 1:
            raise ValueError("every must be >= 1")
        ad = {"rel_error": rel_error, "abs_error": abs_error, "min_samples": min_samples}
        with self.ctx.progressive(self.camera, adaptive=ad, **kw) as p:
            for _ in self._adaptive_passes(p, every):
                yield p.samples, p.active, p.image()

    def _adaptive_passes(self, p: Progressive, every: Optional[int]):
        """Runs render_adaptive's passes on the adaptive frame p, yielding after each one."""
        spp = p.samples_per_pixel
        starts = chunk_starts(spp, self.camera.width * self.camera.height)
        k = next((i for i, s in enumerate(starts) if i and s >= p.adaptive.min_samples), len(starts) - 1)
        while p.active:
            done = p.samples
            if every is None:
                target = starts[min(k, len(starts) - 1)]
                k *= 2
            else:
                target = (done // every + 1) * every
            self.last_stats = p.render(min(target, spp))
            yield

    def render_denoised(self, rel_error: float = 0.0, abs_error: float = 0.0, iterations: int = 5,
                        sigma_color: float = 4.0, aov_samples: Optional[int] = None, **kw):
        """Scene::render followed by the a-trous filter (Progressive.denoised): returns (image, denoised), both (H, W, 3)
        f32.  The frame is adaptive with the given tolerances and render_adaptive's passes; with both tolerances 0 it is
        one pass and `image` is render()'s image bit for bit.  kw: Context.progressive's options (seed, mode, ...) and
        min_samples."""
        ad = {"rel_error": rel_error, "abs_error": abs_error, "min_samples": kw.pop("min_samples", None)}
        with self.ctx.progressive(self.camera, adaptive=ad, **kw) as p:
            if rel_error == 0.0 and abs_error == 0.0:
                self.last_stats = p.render(p.samples_per_pixel)
            else:
                for _ in self._adaptive_passes(p, None):
                    pass
            return p.image(), p.denoised(iterations=iterations, sigma_color=sigma_color, aov_samples=aov_samples)
