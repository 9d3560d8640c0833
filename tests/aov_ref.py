"""Reference statement of the denoising guides (include/nrrt.h, nrrt_accum_aov) for the tests: oracle_aov, restated with
the CPU oracle's own camera ray, hit and texture code (oracle/oracle.cpp, compiled with one more entry point into a
temporary directory), in the library's operation order."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from nr_ray_tracer_b200 import _abi as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Guides for pixels [pixel_begin, pixel_end): the mean over samples 0 .. n-1 of each sample's first hit — albedo
# (Lambertian / Metal: the texture colour; Dielectric: 1; DiffuseLight: the texture colour clamped to [0, 1]) and the
# hit record's normal; a miss gives the background clamped to [0, 1] and a zero normal.  Summed in sample order,
# divided by n, cast to f32.  albedo / normal: W*H*3 f32 indexed by full-image pixel.
AOV_SRC = r'''
extern "C" int oracle_aov(const oracle_scene* s, const nrrt_camera* cam, uint64_t seed, uint32_t pixel_begin,
                          uint32_t pixel_end, uint32_t n, float* albedo, float* normal, int n_threads) {
    if (!s || !cam || !albedo || !normal || n == 0) return -1;
    const uint32_t W = cam->width;
    auto clamp01 = [](V3 c) {
        return v3(std::fmin(std::fmax(c.x, 0.0), 1.0), std::fmin(std::fmax(c.y, 0.0), 1.0),
                  std::fmin(std::fmax(c.z, 0.0), 1.0));
    };
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t p = pixel_begin; p < (int64_t)pixel_end; ++p) {
        Counters c;
        const uint32_t x = (uint32_t)(p % W), y = (uint32_t)(p / W);
        V3 sa = v3(0, 0, 0), sn = v3(0, 0, 0);
        for (uint32_t k = 0; k < n; ++k) {
            Sampler smp{seed, (uint32_t)p, k};
            Ray ray = get_ray(*cam, x, y, smp);
            OptHit h = s->sc->root->hit(ray, Interval{0.001, INF}, c);
            if (!h.some) {
                sa = sa + clamp01(ld3(cam->background));
                sn = sn + v3(0, 0, 0);
                continue;
            }
            const Material* m = h.h.material;
            V3 a;
            if (m->kind == NRRT_MAT_DIELECTRIC) a = v3(1, 1, 1);
            else if (m->kind == NRRT_MAT_DIFFUSE_LIGHT) a = clamp01(m->texture->get_color(h.h.u, h.h.v, h.h.point));
            else a = m->texture->get_color(h.h.u, h.h.v, h.h.point);
            sa = sa + a;
            sn = sn + h.h.normal;
        }
        const V3 ma = sa / (double)n, mn = sn / (double)n;
        albedo[3 * p] = (float)ma.x, albedo[3 * p + 1] = (float)ma.y, albedo[3 * p + 2] = (float)ma.z;
        normal[3 * p] = (float)mn.x, normal[3 * p + 1] = (float)mn.y, normal[3 * p + 2] = (float)mn.z;
    }
    return 0;
}
'''

_lib = None


def _aov_lib():
    global _lib
    if _lib is None:
        with tempfile.TemporaryDirectory(prefix="nrrt_aov_") as d:  # (a loaded library outlives its file)
            src = os.path.join(d, "aov.cpp")
            with open(src, "w") as f:
                f.write('#include "%s"\n' % os.path.join(ROOT, "oracle", "oracle.cpp") + AOV_SRC)
            so = os.path.join(d, "libaov.so")
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.run([cxx, "-O3", "-mtune=generic", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                            "-std=c++17", "-w", "-shared", "-o", so, src], check=True, capture_output=True)
            L = C.CDLL(so)
        L.oracle_build.restype = C.c_void_p
        L.oracle_build.argtypes = [C.POINTER(A.GraphDesc)]
        L.oracle_free.argtypes = [C.c_void_p]
        L.oracle_aov.argtypes = [C.c_void_p, C.POINTER(A.Camera), C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32,
                                 C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


def oracle_aov(graph, cam, n, seed=0, pixel_range=None, n_threads=0):
    """Guides of samples [0, n) of each pixel: (albedo, normal), each (H, W, 3) float32."""
    L = _aov_lib()
    holder = graph.to_desc()
    h = L.oracle_build(holder.ptr())
    assert h, "oracle_build failed"
    try:
        W, H = cam.width, cam.height
        p0, p1 = pixel_range if pixel_range is not None else (0, W * H)
        albedo = np.zeros((H, W, 3), dtype=np.float32)
        normal = np.zeros((H, W, 3), dtype=np.float32)
        assert L.oracle_aov(h, C.byref(cam), seed, p0, p1, n, albedo.ctypes.data, normal.ctypes.data, n_threads) == 0
        return albedo, normal
    finally:
        L.oracle_free(h)
