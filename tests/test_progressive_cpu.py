"""Progressive rendering on the host side: how passes cut the work (nrrt_pass_items runs the kernels' decode with a
pass's chunk offset), the CLI's --preview-every checks that come before any device is touched, and no CPU fallback."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from nr_ray_tracer_b200 import _abi as A
from nr_ray_tracer_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "nr_ray_tracer_b200", "bin", "nr-ray-tracer")
QUADS = os.path.join(ROOT, "scenes", "quads.toml")


def schedules(n_chunks):
    """Pass schedules as chunk boundaries [0, ..., n_chunks]: one pass, one per chunk, [1, rest], and an uneven one."""
    out = [[0, n_chunks], list(range(n_chunks + 1))]
    if n_chunks > 1:
        out.append([0, 1, n_chunks])
    if n_chunks > 4:
        out.append([0, 2, 3, n_chunks - 1, n_chunks])
    return out


@pytest.mark.parametrize("W,H,spp,world,R", [(16, 9, 5, 1, 8), (37, 23, 64, 1, 8), (37, 23, 64, 3, 1),
                                              (64, 36, 1000, 2, 8), (40, 30, 7, 8, 1), (9, 5, 3, 8, 8),
                                              (600, 400, 300, 4, 1)])
def test_passes_hand_out_every_owned_sample_once(W, H, spp, world, R):
    starts = api.chunk_starts(spp, W * H)
    n_chunks = len(starts) - 1
    for rank in range(world):
        full = api.work_items(W, H, spp, rank, world, R)
        owned = api.owned_rows(H, rank, world, R) * W
        assert len(full) == owned * n_chunks
        for bounds in schedules(n_chunks):
            got = [api.pass_items(W, H, spp, c0, c1, rank, world, R) for c0, c1 in zip(bounds, bounds[1:])]
            for (c0, c1), items in zip(zip(bounds, bounds[1:]), got):
                assert len(items) == owned * (c1 - c0)
                if len(items):  # the pass covers exactly samples [starts[c0], starts[c1]) of each of its pixels
                    assert items[:, 2].min() == starts[c0] and items[:, 3].max() == starts[c1]
                    assert set(items[:, 2].tolist()) <= set(starts) and set(items[:, 3].tolist()) <= set(starts)
            # item to pixel order inside a chunk, and the chunk order, are the one-shot render's: the passes put
            # together are the one-shot item list
            cat = np.concatenate(got) if got else np.zeros((0, 4), np.uint32)
            assert np.array_equal(cat, full), (rank, bounds)
        if owned == 0:  # a rank that owns no rows (more ranks than row-blocks) has no work in any pass
            continue
        # every (owned pixel, sample) exactly once: per pixel the spans tile [0, spp)
        key = full[:, 1].astype(np.int64) * W + full[:, 0]
        order = np.lexsort((full[:, 2], key))
        k, s0, s1 = key[order], full[order, 2], full[order, 3]
        first = np.r_[True, k[1:] != k[:-1]]
        last = np.r_[k[1:] != k[:-1], True]
        assert (s0[first] == 0).all() and (s1[last] == spp).all()
        assert (s1[:-1][~last[:-1]] == s0[1:][~first[1:]]).all()
        assert first.sum() == owned


def test_pass_items_rejects_ranges_past_the_last_chunk():
    n_chunks = len(api.chunk_starts(64, 16 * 9)) - 1
    assert api.lib().nrrt_pass_items(16, 9, 64, 0, 1, 8, n_chunks + 1, n_chunks + 2, 0, 0, None) == 0
    assert api.lib().nrrt_pass_items(16, 9, 64, 0, 1, 8, n_chunks, n_chunks, 0, 0, None) == 0
    assert api.lib().nrrt_pass_items(16, 9, 64, 0, 1, 8, 1, 1000, 0, 0, None) == 16 * 9 * (n_chunks - 1)


def test_owned_rows_matches_the_library():
    for H, world, R in [(9, 1, 8), (23, 3, 1), (36, 8, 8), (5, 8, 8), (1080, 8, 1)]:
        total = 0
        for rank in range(world):
            rows = api.owned_rows(H, rank, world, R)
            assert api.lib().nrrt_work_items(7, H, 1, rank, world, R, 0, 0, None) == rows * 7
            total += rows
        assert total == H


def run(*args):
    return subprocess.run([CLI, *args], capture_output=True, text=True, cwd=ROOT, timeout=120)


def test_preview_every_is_refused_with_several_gpus_before_any_device(tmp_path):
    out = tmp_path / "p.png"
    r = run("render", QUADS, "-o", str(out), "--preview-every", "4", "--gpus", "2")
    assert r.returncode != 0 and "--preview-every" in r.stderr and "--gpus" in r.stderr, r.stderr
    assert "CUDA" not in r.stderr and "device" not in r.stderr.replace("--preview-every", "")
    assert not out.exists()


@pytest.mark.parametrize("value", ["0", "-1", "1e3", "", "four", "4294967296"])
def test_preview_every_value_is_validated(tmp_path, value):
    out = tmp_path / "v.png"
    r = run("render", QUADS, "-o", str(out), "--preview-every", value)
    assert r.returncode != 0 and "invalid value" in r.stderr and "--preview-every" in r.stderr, r.stderr
    assert not out.exists()
    assert "--preview-every" in run("--help").stdout


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a box without a GPU")
def test_progressive_without_a_gpu_fails_loudly():
    cam = api.camera_build(A.CameraConfig(width=8, height=8, samples_per_pixel=4, ray_max_bounces=4,
                                          look_from=(0, 0, 1), look_at=(0, 0, 0), view_up=(0, 1, 0),
                                          field_of_view=1.0, focus_dist=1.0))
    with pytest.raises(api.NrrtError):
        api.Context(0).progressive(cam)
    h = C.c_void_p()
    assert api.lib().nrrt_accum_create(None, C.byref(cam), None, C.byref(h)) == A.ERR_INVALID and not h.value
