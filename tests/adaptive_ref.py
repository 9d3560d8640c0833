"""Reference statements of adaptive sampling (include/nrrt.h) for the tests: the convergence test and the error
estimate in numpy, in the order the library evaluates them, and the per-chunk f64 partial sums of the CPU oracle."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from nr_ray_tracer_b200 import _abi as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def e2(S, Q, N, K):
    """Squared standard error of the mean per channel: d / ((K - 1) N), d = max(Q - S*S/N, 0) (NaN propagates).
    S, Q: (..., 3) f64; N, K: (...) integers with K >= 2."""
    S, Q = np.asarray(S, np.float64), np.asarray(Q, np.float64)
    n = np.asarray(N, np.float64)[..., None]
    x = Q - (S * S) / n
    d = np.where(x < 0, 0.0, x)
    return d / ((np.asarray(K, np.float64)[..., None] - 1.0) * n)


def converged(S, Q, N, K, rel_error, abs_error=0.0, min_samples=0):
    """The adaptive test, vectorised over pixels: (...) bool."""
    S = np.asarray(S, np.float64)
    N, K = np.asarray(N), np.asarray(K)
    with np.errstate(divide="ignore", invalid="ignore"):
        m = S / np.asarray(N, np.float64)[..., None]
        tol = abs_error + rel_error * np.abs(m)
        ok = (e2(S, Q, N, np.maximum(K, 2)) <= tol * tol).all(axis=-1)
    return ok & (K >= 2) & (N >= min_samples) & (rel_error > 0 or abs_error > 0)


_lib = None


def _partials_lib():
    """oracle.cpp with one more entry point, oracle_render_partials, compiled into a temporary directory."""
    global _lib
    if _lib is None:
        with tempfile.TemporaryDirectory(prefix="nrrt_partials_") as d:  # (a loaded library outlives its file)
            src = os.path.join(d, "partials.cpp")
            with open(src, "w") as f:
                f.write('#include "%s"\n' % os.path.join(ROOT, "oracle", "oracle.cpp") + PARTIALS_SRC)
            so = os.path.join(d, "libpartials.so")
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.run([cxx, "-O3", "-mtune=generic", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                            "-std=c++17", "-w", "-shared", "-o", so, src], check=True, capture_output=True)
            L = C.CDLL(so)
        L.oracle_build.restype = C.c_void_p
        L.oracle_build.argtypes = [C.POINTER(A.GraphDesc)]
        L.oracle_free.argtypes = [C.c_void_p]
        L.oracle_render_partials.argtypes = [C.c_void_p, C.POINTER(A.Camera), C.c_uint64, C.c_uint32, C.c_uint32,
                                             C.c_void_p, C.c_uint32, C.c_void_p]
        _lib = L
    return _lib


# Chunk c's partial sum of each pixel: samples [starts[c], starts[c + 1]) summed in order from zero, as
# oracle_render_chunked sums them before adding the partials.  out: (pixel_end - pixel_begin) x n_chunks x 3 f64.
PARTIALS_SRC = r'''
extern "C" int oracle_render_partials(const oracle_scene* s, const nrrt_camera* cam, uint64_t seed, uint32_t pixel_begin,
                                      uint32_t pixel_end, const uint32_t* starts, uint32_t n_chunks, double* out) {
    if (!s || !cam || !out || !starts || n_chunks == 0) return -1;
    const uint32_t W = cam->width;
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t n = pixel_begin; n < (int64_t)pixel_end; ++n) {
        Counters c;
        const uint32_t x = (uint32_t)(n % W), y = (uint32_t)(n / W);
        for (uint32_t ch = 0; ch < n_chunks; ++ch) {
            V3 part = v3(0, 0, 0);
            for (uint32_t k = starts[ch]; k < starts[ch + 1]; ++k) {
                Sampler smp{seed, (uint32_t)n, k};
                Ray ray = get_ray(*cam, x, y, smp);
                part = part + get_ray_color(*cam, *s->sc, ray, 0, smp, c);
            }
            double* o = out + ((size_t)(n - pixel_begin) * n_chunks + ch) * 3;
            o[0] = part.x, o[1] = part.y, o[2] = part.z;
        }
    }
    return 0;
}
'''


def render_partials(graph, cam, starts, seed=0):
    """(H, W, n_chunks, 3) f64: every pixel's chunk partials over the chunks `starts` bounds."""
    L = _partials_lib()
    holder = graph.to_desc()
    h = L.oracle_build(holder.ptr())
    assert h, "oracle_build failed"
    try:
        st = np.ascontiguousarray(starts, dtype=np.uint32)
        out = np.zeros((cam.height, cam.width, len(st) - 1, 3), dtype=np.float64)
        assert L.oracle_render_partials(h, C.byref(cam), seed, 0, cam.width * cam.height, st.ctypes.data, len(st) - 1,
                                        out.ctypes.data) == 0
        return out
    finally:
        L.oracle_free(h)


def reduce_partials(P, starts, K):
    """S and Q of each pixel over its first K chunks, added in chunk order as the library adds them:
    S += p;  Q += (p * p) / n_c.  P: (..., n_chunks, 3); K: (...) chunk counts."""
    n_c = np.diff(np.asarray(starts, np.float64))
    S = np.zeros(P.shape[:-2] + (3,))
    Q = np.zeros_like(S)
    K = np.asarray(K)
    for c in range(P.shape[-2]):
        take = (K > c)[..., None]
        p = P[..., c, :]
        S = np.where(take, S + p, S)
        Q = np.where(take, Q + (p * p) / n_c[c], Q)
    return S, Q
