"""Reference statement of the denoising filter (include/nrrt.h, nrrt_accum_denoise) in float32 numpy, operation for
operation in the library's order: each numpy float32 operation rounds once, as the kernel's _rn intrinsics do, so the
result is the device's bit for bit."""
import numpy as np

from tests import adaptive_ref as R

F = np.float32
MIN_ALBEDO = F(2.0 ** -8)
EPS = F(1e-10)
B = (F(3 / 8), F(1 / 4), F(1 / 16))
INF = F(np.inf)


def inputs(S, Q, N, K):
    """C = (float)(S / N) and e2 = (float)e2 (+inf where K < 2) per channel, (H, W, 3) float32 each, from an adaptive
    frame's state (S, Q: (H, W, 3) f64; N, K: (H, W))."""
    N, K = np.asarray(N), np.asarray(K)
    with np.errstate(divide="ignore", invalid="ignore"):
        C = (np.asarray(S, np.float64) / N.astype(np.float64)[..., None]).astype(F)
        e2 = R.e2(S, Q, N, np.maximum(K, 2)).astype(F)
    e2[K < 2] = INF
    return C, e2


def _luma(E):
    return ((E[..., 0] + E[..., 1]) + E[..., 2]) / F(3)


def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def denoise(C, e2, albedo, normal, iterations=5, sigma_color=4.0):
    """The filter on one image: C, e2, albedo, normal (H, W, 3) float32 -> (H, W, 3) float32."""
    C, e2 = np.asarray(C, F), np.asarray(e2, F)
    A, Nrm = np.asarray(albedo, F), np.asarray(normal, F)
    H, W = C.shape[:2]
    sigma2 = F(sigma_color) * F(sigma_color)
    with np.errstate(all="ignore"):
        a = np.fmax(A, MIN_ALBEDO)
        E = C / a
        t = e2 / (a * a)
        v = ((t[..., 0] + t[..., 1]) + t[..., 2]) * (F(1) / F(9))
        ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
        for it in range(iterations):
            h = 1 << it
            lp = _luma(E)
            no_estimate = v == INF
            den = sigma2 * v + EPS
            sw = np.zeros((H, W), F)
            sE = np.zeros((H, W, 3), F)
            sv = np.zeros((H, W), F)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    qy, qx = ys + dy * h, xs + dx * h
                    inside = (qy >= 0) & (qy < H) & (qx >= 0) & (qx < W)
                    qy, qx = np.clip(qy, 0, H - 1), np.clip(qx, 0, W - 1)
                    Eq, vq = E[qy, qx], v[qy, qx]
                    k = B[abs(dx)] * B[abs(dy)]
                    if dx == 0 and dy == 0:
                        w = np.full((H, W), k, F)
                    else:
                        wn = np.fmax(_dot(Nrm, Nrm[qy, qx]), F(0))
                        for _ in range(7):
                            wn = wn * wn
                        d = A - A[qy, qx]
                        wa = F(1) / (F(1) + _dot(d, d) * F(64))
                        dl = lp - _luma(Eq)
                        wc = np.where(no_estimate, F(1), F(1) / (F(1) + (dl * dl) / den))
                        w = ((k * wn) * wa) * wc
                    ww = w * w
                    take = inside & (ww != 0)  # w == 0, or w * w underflows: 0 * inf must not reach the sums
                    sw = np.where(take, sw + w, sw)
                    sE = np.where(take[..., None], sE + w[..., None] * Eq, sE)
                    sv = np.where(take, sv + ww * vq, sv)
            E = sE / sw[..., None]
            v = sv / (sw * sw)
        return E * a
