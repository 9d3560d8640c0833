"""Adaptive sampling on the host side: the pass decode over an active list (nrrt_pass_items_active runs the kernels'
decode_item with the list), the convergence test against its numpy statement, and the CLI's checks that come before
any device is touched."""
import math
import os
import subprocess

import numpy as np
import pytest

from nr_ray_tracer_b200 import api
from tests import adaptive_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "nr_ray_tracer_b200", "bin", "nr-ray-tracer")
QUADS = os.path.join(ROOT, "scenes", "quads.toml")


@pytest.mark.parametrize("W,H,spp,world,R_", [(16, 9, 5, 1, 8), (37, 23, 64, 1, 8), (37, 23, 64, 3, 1),
                                               (64, 36, 1000, 2, 8), (40, 30, 7, 8, 1), (9, 5, 3, 8, 8)])
def test_active_passes_hand_out_each_active_pixel_s_samples_once(W, H, spp, world, R_):
    rng = np.random.default_rng(W * H + spp + world)
    starts = api.chunk_starts(spp, W * H)
    n_chunks = len(starts) - 1
    for rank in range(world):
        owned = api.owned_rows(H, rank, world, R_) * W
        if world == 8 and R_ == 8:
            assert owned == 0 or rank == 0  # 5 rows, one block: ranks 1..7 own nothing
        # pixel of each owned-pixel index: the order a chunk of a plain pass visits them
        pix = api.pass_items(W, H, spp, 0, 1, rank, world, R_)[:, :2].astype(np.int64)
        assert len(pix) == owned
        everything = np.arange(owned, dtype=np.uint32)
        for c0, c1 in [(0, n_chunks), (0, 1), (min(1, n_chunks - 1), n_chunks), (n_chunks // 2, n_chunks // 2 + 1)]:
            plain = api.pass_items(W, H, spp, c0, c1, rank, world, R_)
            assert np.array_equal(api.pass_items_active(W, H, spp, c0, c1, everything, rank, world, R_), plain)
            subsets = [np.zeros(0, np.uint32), everything]
            if owned:
                subsets += [np.flatnonzero(rng.random(owned) < f).astype(np.uint32) for f in (0.05, 0.5, 0.95)]
                subsets.append(np.array([owned - 1], np.uint32))
            for act in subsets:
                items = api.pass_items_active(W, H, spp, c0, c1, act, rank, world, R_)
                assert len(items) == len(act) * (c1 - c0)
                if not len(items):
                    continue
                per = items.reshape(c1 - c0, len(act), 4)
                for k in range(c1 - c0):  # chunk-major; inside a chunk the pixels follow the active list
                    assert np.array_equal(per[k, :, :2].astype(np.int64), pix[act])
                    assert (per[k, :, 2] == starts[c0 + k]).all() and (per[k, :, 3] == starts[c0 + k + 1]).all()
                # every (active pixel, sample in [starts[c0], starts[c1])) exactly once, no other pixel
                key = items[:, 1].astype(np.int64) * W + items[:, 0]
                assert set(key.tolist()) == set((pix[act, 1] * W + pix[act, 0]).tolist())
                seen = np.zeros(W * H, np.int64)
                np.add.at(seen, key, items[:, 3].astype(np.int64) - items[:, 2])
                assert (seen[np.unique(key)] == starts[c1] - starts[c0]).all()


def test_pass_items_active_rejects_bad_lists():
    W, H, spp = 16, 9, 64
    assert len(api.pass_items_active(W, H, spp, 0, 1, [0, 5, 7])) == 3
    for bad in ([5, 5], [7, 5], [0, W * H], [W * H + 3]):
        assert len(api.pass_items_active(W, H, spp, 0, 1, bad)) == 0, bad
    # a rank's list indexes its own pixels only
    owned = api.owned_rows(H, 1, 2, 1) * W
    assert len(api.pass_items_active(W, H, spp, 0, 1, [owned - 1], 1, 2, 1)) == 1
    assert len(api.pass_items_active(W, H, spp, 0, 1, [owned], 1, 2, 1)) == 0


def _lib_says(S, Q, N, K, rel, ab=0.0, ms=0):
    return api.adaptive_converged(S, Q, N, K, rel, ab, ms)


def test_converged_equals_the_numpy_statement_on_random_states():
    rng = np.random.default_rng(7)
    for _ in range(3000):
        K = int(rng.integers(0, 30))
        N = int(rng.integers(1, 4096))
        mean = rng.random(3) * rng.choice([1e-3, 1.0, 50.0])
        sigma = rng.random(3) * rng.choice([0.0, 1e-4, 0.1, 1.0, 10.0])
        S = mean * N
        Q = (sigma ** 2 * max(K - 1, 1) + mean * mean * N) * rng.choice([1.0, 1.0 - 1e-15, 1.0 + 1e-12])
        rel = float(rng.choice([0.0, 1e-3, 0.01, 0.03, 0.5]))
        ab = float(rng.choice([0.0, 0.0, 1e-4, 1e-2]))
        ms = int(rng.choice([0, 1, N, N + 1, 4096]))
        want = bool(R.converged(S, Q, N, K, rel, ab, ms))
        assert _lib_says(S, Q, N, K, rel, ab, ms) == want, (S, Q, N, K, rel, ab, ms)


def test_converged_edge_cases():
    N, K = 64, 8
    S = np.array([0.5, 0.25, 0.125]) * N
    Q = S * S / N  # zero variance: e2 = 0
    assert _lib_says(S, Q, N, K, 0.01) and R.converged(S, Q, N, K, 0.01)
    # Q - S*S/N a little below zero from rounding: clamped to zero, so still converged
    Qneg = np.nextafter(Q, -np.inf)
    assert ((Qneg - S * S / N) < 0).any()
    assert _lib_says(S, Qneg, N, K, 0.01) and R.converged(S, Qneg, N, K, 0.01)
    # one chunk: no variance estimate, never converged
    assert not _lib_says(S, Q, N, 1, 0.01) and not R.converged(S, Q, N, 1, 0.01)
    assert not _lib_says(S, Q, N, 0, 0.01)
    # below min_samples
    assert not _lib_says(S, Q, N, K, 0.01, 0.0, N + 1) and _lib_says(S, Q, N, K, 0.01, 0.0, N)
    # both tolerances 0: never, even at zero variance and zero mean
    assert not _lib_says(S, Q, N, K, 0.0, 0.0) and not _lib_says(np.zeros(3), np.zeros(3), N, K, 0.0, 0.0)
    assert _lib_says(np.zeros(3), np.zeros(3), N, K, 0.0, 1e-9)  # abs_error alone retires a black pixel
    # NaN anywhere in the state fails the test
    for arr in ("S", "Q"):
        for ch in range(3):
            s2, q2 = S.copy(), Q.copy()
            (s2 if arr == "S" else q2)[ch] = math.nan
            assert not _lib_says(s2, q2, N, K, 0.5, 1.0) and not R.converged(s2, q2, N, K, 0.5, 1.0)
    # at the boundary: e2 == tol^2 passes, one ulp above fails
    S1, N1, K1 = np.array([2.0, 2.0, 2.0]), 4, 5
    Q1 = np.array([1.0 + 0.16 * 16.0] * 3)  # d = Q - 1 = 2.56; e2 = 2.56 / 16 = 0.16 = 0.4^2 (in f64 arithmetic)
    e = R.e2(S1, Q1, N1, K1)[0]
    tol = math.sqrt(e)
    assert _lib_says(S1, Q1, N1, K1, 0.0, tol) == bool(e <= tol * tol) == R.converged(S1, Q1, N1, K1, 0.0, tol)
    assert _lib_says(S1, Q1, N1, K1, 0.0, np.nextafter(tol, 0)) == R.converged(S1, Q1, N1, K1, 0.0, np.nextafter(tol, 0))


def test_default_min_samples_is_the_first_boundary_at_or_above_an_eighth():
    assert api.default_min_samples(1024, 1920 * 1080) == 148  # chunks of 37: 4 x 37 >= 128
    assert api.default_min_samples(40, 64 * 36) == 6           # chunks of 2
    assert api.default_min_samples(1, 100) == 1


def run(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, cwd=ROOT, timeout=120)


@pytest.mark.parametrize("flag,value", [("--adaptive-error", "-0.1"), ("--adaptive-error", "nan"),
                                        ("--adaptive-error", "inf"), ("--adaptive-error", ""),
                                        ("--adaptive-error", "0.1x"), ("--adaptive-abs-error", "-1"),
                                        ("--adaptive-min-samples", "-3"), ("--adaptive-min-samples", "1.5")])
def test_adaptive_values_are_validated(tmp_path, flag, value):
    out = tmp_path / "v.png"
    args = ["render", QUADS, "-o", str(out), flag, value]
    if flag != "--adaptive-error":
        args += ["--adaptive-error", "0.01"]
    r = run(*args)
    assert r.returncode != 0 and "invalid value" in r.stderr and flag in r.stderr, r.stderr
    assert not out.exists()


def test_adaptive_is_refused_with_several_gpus_before_any_device(tmp_path):
    out = tmp_path / "p.png"
    r = run("render", QUADS, "-o", str(out), "--adaptive-error", "0.01", "--gpus", "2")
    assert r.returncode != 0 and "--adaptive-error" in r.stderr and "--gpus" in r.stderr, r.stderr
    assert "CUDA" not in r.stderr and "device" not in r.stderr
    assert not out.exists()
    for flag, v in (("--adaptive-abs-error", "0.1"), ("--adaptive-min-samples", "8")):
        r = run("render", QUADS, "-o", str(out), flag, v)
        assert r.returncode != 0 and "needs --adaptive-error" in r.stderr, r.stderr
        assert not out.exists()
    assert "--adaptive-error" in run("--help").stdout
