"""bench.py contract checks: the reference arm's JSON line, rank handling, --dump-outputs, and the refusal of the
product arm to produce a number without a GPU (no CPU fallback) — all without a GPU except the product arm's dump."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--width", "48", "--height", "27", "--spp", "4", "--ref-spp", "2", "--depth", "5"]


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          cwd=ROOT, env=e, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = run(["--impl", "reference", "--steps", "2", "--warmup", "1"] + SMALL)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "cornell-box-scene.json 48x27 4spp depth5" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_silently():
    r = run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"] + SMALL,
            env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_refused():
    r = run(["--impl", "reference", "--steps", "0"] + SMALL)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_reference_arm_dumps_its_last_step_reproducibly(tmp_path):
    """--dump-outputs DIR (relative to the caller's directory): the last timed step's image and segment count, the same
    bytes from run to run, and the image is the oracle's render of the benchmark scene at the given size."""
    for k in range(2):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                            "--warmup", "0", "--dump-outputs", f"out{k}"] + SMALL,
                           capture_output=True, text=True, cwd=tmp_path, timeout=600)
        assert r.returncode == 0, r.stderr
    img, segs = np.load(tmp_path / "out0" / "image.npy"), np.load(tmp_path / "out0" / "segments.npy")
    assert img.dtype == np.float32 and img.shape == (27, 48, 3) and segs.dtype == np.float64 and segs[0] > 0
    assert np.array_equal(img, np.load(tmp_path / "out1" / "image.npy"))
    assert np.array_equal(segs, np.load(tmp_path / "out1" / "segments.npy"))
    from oracle import oracle as O
    from tests.scenes_util import load
    g = load("cornell-box-scene.json", width=48, height=27, samples_per_pixel=2, ray_max_bounces=5)
    ref, cnt = O.OracleScene(g).render(O.camera_build(g.camera.to_builder_config()), seed=0)
    assert np.array_equal(img, ref) and segs[0] == cnt["segments"]


def test_dump_is_a_fixed_sample_within_the_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 4096 + 8 + 12 * 1000)   # two headers, the count, 1000 pixels
    img = np.random.default_rng(1).random((100, 50, 3), dtype=np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"image": img, "segments": np.array([7.0])})
    a = np.load(tmp_path / "a" / "image.npy")
    assert a.shape == (1000, 3) and np.array_equal(a, np.load(tmp_path / "b" / "image.npy"))
    assert np.isin(a[:, 0], img[..., 0]).all()
    assert np.load(tmp_path / "a" / "segments.npy").tolist() == [7.0]
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES


@pytest.mark.gpu
def test_product_arm_dumps_the_images_it_timed(gpu_ctx, tmp_path):
    """The device-resident step and the end-to-end Scene.render step both hand back the library's render of the
    benchmark scene with seed 0; --dump-outputs writes both, and the segment count, after the timed steps."""
    from nr_ray_tracer_b200 import api
    from tests.scenes_util import load
    r = run(["--steps", "2", "--warmup", "1", "--no-cpu", "--dump-outputs", str(tmp_path)] + SMALL)
    assert r.returncode == 0, r.stderr
    img = np.load(tmp_path / "image.npy")
    assert img.dtype == np.float32 and img.shape == (27, 48, 3)
    assert np.array_equal(img, np.load(tmp_path / "e2e_image.npy"))
    g = load("cornell-box-scene.json", width=48, height=27, samples_per_pixel=4, ray_max_bounces=5)
    scene = api.Scene(g, ctx=gpu_ctx)
    assert np.array_equal(img, scene.render(seed=0))
    assert np.load(tmp_path / "segments.npy").tolist() == [scene.last_stats["segments"]]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a box without a GPU")
def test_product_arm_refuses_to_run_without_a_gpu():
    r = run(["--steps", "1", "--warmup", "1", "--no-cpu"] + SMALL)
    assert r.returncode != 0
    assert not any(ln.startswith("{") and '"value"' in ln for ln in r.stdout.splitlines())
