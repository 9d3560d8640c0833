#!/usr/bin/env python3
"""Generates rust/nrrt-sys/src/lib.rs — the Rust `-sys` bindings of include/nrrt.h — from the ctypes mirror
(nr_ray_tracer_b200/_abi.py), whose struct sizes the test suite checks against the compiled library
(nrrt_abi_sizeof).  One source of truth for every binding: a field added to the header and to _abi.py shows up in
the Rust structs by re-running this script; tests/test_rust_bindings.py fails when the committed file is stale.

Usage: python tools/gen_nrrt_sys.py [--check]"""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nr_ray_tracer_b200 import _abi as A  # noqa: E402

OUT = os.path.join(ROOT, "rust", "nrrt-sys", "src", "lib.rs")
STRUCTS = [("nrrt_object", A.Object), ("nrrt_material", A.Material), ("nrrt_texture", A.Texture), ("nrrt_image", A.Image),
           ("nrrt_graph_desc", A.GraphDesc), ("nrrt_camera_config", A.CameraConfig), ("nrrt_camera", A.Camera),
           ("nrrt_node", A.Node), ("nrrt_box", A.Box), ("nrrt_wnode", A.WNode), ("nrrt_xform", A.Xform),
           ("nrrt_instance", A.Instance), ("nrrt_scene_desc", A.SceneDesc), ("nrrt_hit", A.Hit),
           ("nrrt_hit_compact", A.HitCompact), ("nrrt_trace_stats", A.TraceStats), ("nrrt_render_opts", A.RenderOpts),
           ("nrrt_render_stats", A.RenderStats), ("nrrt_camera_file", A.CameraFile), ("nrrt_adaptive_opts", A.AdaptiveOpts),
           ("nrrt_denoise_opts", A.DenoiseOpts)]
NAMES = {cls: name for name, cls in STRUCTS}
SCALARS = {C.c_uint32: "u32", C.c_uint64: "u64", C.c_double: "f64", C.c_float: "f32", C.c_uint8: "u8", C.c_int: "c_int"}
# which = index accepted by nrrt_abi_sizeof (header order, see include/nrrt.h)
SIZEOF_ORDER = ["nrrt_object", "nrrt_material", "nrrt_texture", "nrrt_image", "nrrt_graph_desc", "nrrt_camera_config",
                "nrrt_camera", "nrrt_node", "nrrt_box", "nrrt_xform", "nrrt_instance", "nrrt_scene_desc", "nrrt_hit",
                "nrrt_trace_stats", "nrrt_render_opts", "nrrt_render_stats", "nrrt_camera_file", "nrrt_wnode",
                "nrrt_hit_compact", "nrrt_adaptive_opts", "nrrt_denoise_opts"]


def rust_type(t, field=""):
    if t in SCALARS:
        return SCALARS[t]
    if t in NAMES:
        return NAMES[t]
    if t is C.c_void_p:
        return "*const u8" if field == "rgb" else "*const c_void"
    if isinstance(t, type) and issubclass(t, C.Array):
        return f"[{rust_type(t._type_)}; {t._length_}]"
    if isinstance(t, type) and issubclass(t, C._Pointer):
        return f"*const {rust_type(t._type_)}"
    raise TypeError(f"no Rust mapping for {t!r}")


FUNCTIONS = '''
pub enum nrrt_ctx {}
pub enum nrrt_host_scene {}
pub enum nrrt_loaded_scene {}
pub enum nrrt_accum {}
pub type nrrt_progress_fn = Option<unsafe extern "C" fn(pixels_done: u64, pixels_total: u64, user: *mut c_void)>;

pub const NRRT_OK: c_int = 0;
pub const NRRT_ERR_INVALID: c_int = -1;
pub const NRRT_ERR_CUDA: c_int = -2;
pub const NRRT_ERR_NO_DEVICE: c_int = -3; // there is no CPU fallback
pub const NRRT_ERR_NO_SCENE: c_int = -4;
pub const NRRT_ERR_LIMIT: c_int = -5;
pub const NRRT_ERR_IO: c_int = -6;

pub const NRRT_OBJ_SPHERE: u32 = 0;
pub const NRRT_OBJ_QUAD: u32 = 1;
pub const NRRT_OBJ_TRIANGLE: u32 = 2;
pub const NRRT_OBJ_GROUP: u32 = 3;
pub const NRRT_OBJ_TRANSLATE: u32 = 4;
pub const NRRT_OBJ_ROTATE_X: u32 = 5;
pub const NRRT_OBJ_ROTATE_Y: u32 = 6;
pub const NRRT_OBJ_ROTATE_Z: u32 = 7;
pub const NRRT_OBJ_SCALE: u32 = 8;
pub const NRRT_MAT_LAMBERTIAN: u32 = 0;
pub const NRRT_MAT_METAL: u32 = 1;
pub const NRRT_MAT_DIELECTRIC: u32 = 2;
pub const NRRT_MAT_DIFFUSE_LIGHT: u32 = 3;
pub const NRRT_TEX_SOLID: u32 = 0;
pub const NRRT_TEX_CHECKER: u32 = 1;
pub const NRRT_TEX_IMAGE: u32 = 2;
pub const NRRT_TEX_NOISE: u32 = 3;
pub const NRRT_TEX_MARBLE: u32 = 4;
pub const NRRT_BUILD_REFERENCE: u32 = 0;
pub const NRRT_BUILD_SAH: u32 = 1;
pub const NRRT_MODE_WAVEFRONT: u32 = 0;
pub const NRRT_MODE_MEGAKERNEL: u32 = 1;
pub const NRRT_MODE_FUSED: u32 = 2;
pub const NRRT_MODE_POOL: u32 = 3;
pub const NRRT_MODE_AUTO: u32 = 4;
pub const NRRT_RENDER_OUT_DEVICE: u32 = 1;
pub const NRRT_RENDER_COUNT: u32 = 2;
pub const NRRT_RENDER_OUT_PACKED: u32 = 4;
pub const NRRT_TRACE_VISIT_ALL: u32 = 1;
pub const NRRT_TRACE_DEVICE_BUFFERS: u32 = 2;
pub const NRRT_TRACE_COUNT: u32 = 4;
pub const NRRT_TRACE_COMPACT: u32 = 8;

extern "C" {
    // host side: reference BVH build + flatten, camera, native scene loader (no GPU needed)
    pub fn nrrt_host_build(graph: *const nrrt_graph_desc) -> *mut nrrt_host_scene;
    pub fn nrrt_host_build_ex(graph: *const nrrt_graph_desc, flags: u32) -> *mut nrrt_host_scene;
    pub fn nrrt_host_scene_desc(scene: *const nrrt_host_scene) -> *const nrrt_scene_desc;
    pub fn nrrt_host_free(scene: *mut nrrt_host_scene);
    pub fn nrrt_host_last_error() -> *const c_char;
    pub fn nrrt_host_camera_build(config: *const nrrt_camera_config, out: *mut nrrt_camera) -> c_int;
    pub fn nrrt_load_scene(path: *const c_char, base_dir: *const c_char) -> *mut nrrt_loaded_scene;
    pub fn nrrt_loaded_graph(scene: *const nrrt_loaded_scene) -> *const nrrt_graph_desc;
    pub fn nrrt_loaded_camera(scene: *const nrrt_loaded_scene, out: *mut nrrt_camera_file) -> c_int;
    pub fn nrrt_loaded_free(scene: *mut nrrt_loaded_scene);
    pub fn nrrt_load_last_error() -> *const c_char;
    pub fn nrrt_camera_file_merge(base: *mut nrrt_camera_file, over: *const nrrt_camera_file);
    pub fn nrrt_camera_file_to_config(file: *const nrrt_camera_file, out: *mut nrrt_camera_config) -> c_int;
    // device side
    pub fn nrrt_create(device: c_int, out: *mut *mut nrrt_ctx) -> c_int;
    pub fn nrrt_destroy(ctx: *mut nrrt_ctx);
    pub fn nrrt_last_error(ctx: *const nrrt_ctx) -> *const c_char;
    pub fn nrrt_set_stream(ctx: *mut nrrt_ctx, cuda_stream: *mut c_void) -> c_int;
    pub fn nrrt_set_trace_time(ctx: *mut nrrt_ctx, time: f64) -> c_int;
    pub fn nrrt_scene_upload(ctx: *mut nrrt_ctx, scene: *const nrrt_scene_desc) -> c_int;
    pub fn nrrt_trace_rays(ctx: *mut nrrt_ctx, rays: *const f64, n: u64, tmin: f64, tmax: f64, flags: u32,
                           out: *mut nrrt_hit, stats: *mut nrrt_trace_stats) -> c_int;
    pub fn nrrt_render(ctx: *mut nrrt_ctx, camera: *const nrrt_camera, opts: *const nrrt_render_opts, out_rgb: *mut f32,
                       progress: nrrt_progress_fn, user: *mut c_void, stats: *mut nrrt_render_stats) -> c_int;
    pub fn nrrt_render_multi(devices: *const c_int, n_devices: c_int, scene: *const nrrt_scene_desc,
                             camera: *const nrrt_camera, opts: *const nrrt_render_opts, out_rgb: *mut f32,
                             progress: nrrt_progress_fn, user: *mut c_void, stats: *mut nrrt_render_stats,
                             err: *mut c_char, err_len: usize) -> c_int;
    pub fn nrrt_encode_rgb8(ctx: *mut nrrt_ctx, rgb: *const f32, width: u32, height: u32, gamma: f32, flags: u32,
                            out_rgb8: *mut u8) -> c_int;
    pub fn nrrt_chunk_starts(samples_per_pixel: u32, total_pixels: u64, starts: *mut u32, max: u32) -> u32;
    pub fn nrrt_work_items(width: u32, height: u32, samples_per_pixel: u32, rank: u32, world: u32, rows_per_block: u32,
                           first: u32, n: u32, out: *mut u32) -> u32;
    pub fn nrrt_pass_items(width: u32, height: u32, samples_per_pixel: u32, rank: u32, world: u32, rows_per_block: u32,
                           c0: u32, c1: u32, first: u32, n: u32, out: *mut u32) -> u32;
    // progressive rendering: one frame in passes of whole chunks, summed into per-pixel f64 sums on the device
    pub fn nrrt_accum_create(ctx: *mut nrrt_ctx, camera: *const nrrt_camera, opts: *const nrrt_render_opts,
                             out: *mut *mut nrrt_accum) -> c_int;
    pub fn nrrt_accum_render(accum: *mut nrrt_accum, min_samples: u32, stats: *mut nrrt_render_stats) -> c_int;
    pub fn nrrt_accum_samples(accum: *const nrrt_accum) -> u32;
    pub fn nrrt_accum_image(accum: *mut nrrt_accum, out_rgb: *mut f32, flags: u32) -> c_int;
    pub fn nrrt_accum_save(accum: *const nrrt_accum, sums: *mut f64, samples_done: *mut u32) -> c_int;
    pub fn nrrt_accum_restore(accum: *mut nrrt_accum, sums: *const f64, samples_done: u32) -> c_int;
    pub fn nrrt_accum_free(accum: *mut nrrt_accum);
    // adaptive sampling: passes render the pixels still active; a pixel retires once its error estimate meets the tolerance
    pub fn nrrt_accum_create_adaptive(ctx: *mut nrrt_ctx, camera: *const nrrt_camera, opts: *const nrrt_render_opts,
                                      adaptive: *const nrrt_adaptive_opts, out: *mut *mut nrrt_accum) -> c_int;
    pub fn nrrt_accum_active(accum: *const nrrt_accum) -> u32;
    pub fn nrrt_accum_sample_map(accum: *mut nrrt_accum, out: *mut u32, flags: u32) -> c_int;
    pub fn nrrt_accum_error_image(accum: *mut nrrt_accum, out_rgb: *mut f32, flags: u32) -> c_int;
    pub fn nrrt_accum_adaptive_save(accum: *const nrrt_accum, sums: *mut f64, sumsq: *mut f64, samples: *mut u32) -> c_int;
    pub fn nrrt_accum_adaptive_restore(accum: *mut nrrt_accum, sums: *const f64, sumsq: *const f64,
                                       samples: *const u32) -> c_int;
    pub fn nrrt_adaptive_converged(s: *const f64, q: *const f64, samples: u32, chunks: u32,
                                   adaptive: *const nrrt_adaptive_opts) -> c_int;
    pub fn nrrt_pass_items_active(width: u32, height: u32, samples_per_pixel: u32, rank: u32, world: u32,
                                  rows_per_block: u32, c0: u32, c1: u32, active: *const u32, n_active: u32, first: u32,
                                  n: u32, out: *mut u32) -> u32;
    // denoising: first-hit guides of a frame and the a-trous filter on an adaptive frame (an extra output)
    pub fn nrrt_accum_aov(accum: *mut nrrt_accum, aov_samples: u32, albedo: *mut f32, normal: *mut f32, flags: u32) -> c_int;
    pub fn nrrt_accum_denoise(accum: *mut nrrt_accum, opts: *const nrrt_denoise_opts, out_rgb: *mut f32, flags: u32) -> c_int;
    pub fn nrrt_abi_sizeof(which: c_int) -> usize;
}
'''


def generate() -> str:
    out = ["// GENERATED by tools/gen_nrrt_sys.py from nr_ray_tracer_b200/_abi.py (the ctypes mirror of include/nrrt.h that the",
           "// test suite checks against the compiled library) — do not edit by hand; re-run the script.",
           "//",
           "// Raw bindings of libnrrt_b200.so, the B200-native replacement of nr-ray-tracer's render hot path:",
           "//   Scene::render (ray-tracer-lib/src/scene.rs:13-18) -> Camera::render (camera.rs:302-343).",
           "// See INTEGRATION.md for the safe shim that keeps Scene::render's signature.",
           "#![allow(non_camel_case_types)]",
           "use std::os::raw::{c_char, c_int, c_void};", "",
           f"pub const NRRT_ABI_VERSION: u32 = {A.ABI_VERSION};",
           f"pub const NRRT_MAX_INSTANCE_DEPTH: usize = {A.MAX_INSTANCE_DEPTH};", ""]
    for name, cls in STRUCTS:
        out.append("#[repr(C)]")
        out.append("#[derive(Clone, Copy)]")
        out.append(f"pub struct {name} {{")
        for fname, ftype in cls._fields_:
            out.append(f"    pub {fname}: {rust_type(ftype, fname)},")
        out.append("}")
        out.append("")
    out.append(FUNCTIONS.strip("\n"))
    out.append("")
    out.append("/// `(which, size_of)` pairs for `nrrt_abi_sizeof`: call `check_abi()` once after loading the library.")
    out.append("pub fn abi_table() -> Vec<(c_int, usize)> {")
    out.append("    vec![")
    for i, name in enumerate(SIZEOF_ORDER):
        out.append(f"        ({i}, std::mem::size_of::<{name}>()),")
    out.append("    ]")
    out.append("}")
    out.append("")
    out.append("/// Panics if a struct of this binding does not have the size the loaded library was compiled with.")
    out.append("pub fn check_abi() {")
    out.append("    for (which, size) in abi_table() {")
    out.append("        let lib = unsafe { nrrt_abi_sizeof(which) };")
    out.append("        assert_eq!(lib, size, \"nrrt-sys struct #{which} is {size} bytes, libnrrt_b200.so says {lib}\");")
    out.append("    }")
    out.append("}")
    return "\n".join(out) + "\n"


def main():
    text = generate()
    if "--check" in sys.argv:
        cur = open(OUT).read() if os.path.exists(OUT) else ""
        if cur != text:
            sys.exit("rust/nrrt-sys/src/lib.rs is stale: run python tools/gen_nrrt_sys.py")
        print("rust/nrrt-sys/src/lib.rs is up to date")
        return
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    open(OUT, "w").write(text)
    print(OUT)


if __name__ == "__main__":
    main()
