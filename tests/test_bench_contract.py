"""bench.py contract: the reference arm prints ONE JSON line with the agreed keys; our arm refuses to run without a GPU
(no CPU fallback); --dump-outputs writes the frame of the last timed step."""
import importlib.util
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_reference_arm_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--splats", "20000", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and abs(d["value"] - 1000.0 / d["ms_per_step"]) < 1e-6
    assert d["config"]["workload"] == "train_1m_1080p" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_our_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                         timeout=300)
    assert res.returncode != 0 and "no CPU fallback" in (res.stderr + res.stdout)


def test_algorithmic_bytes_one_pass_and_slab():
    """SURVEY.md 8(d) byte model: the one-pass formula, and the slab path's own passes when the library reports slabs."""
    bench = _bench_module()
    st = dict(n_splats=1000, n_sorted=800, n_visible=600, n_tile_instances=5000, n_tiles=100, width=160, height=160,
              n_slabs=0, n_slabs_run=0, n_slab_entries=0, n_instances_kept=900)
    ab = bench.algorithmic_bytes(st)
    assert ab["sort"] == 20 * 1000 + 8 * 800 and ab["raster"] == 36 * 5000 + 4 * 160 * 160
    assert ab["total"] == ab["sort"] + ab["project"] + ab["bin"] + ab["raster"]
    st.update(n_slabs=3, n_slabs_run=2, n_slab_entries=700)
    sb = bench.algorithmic_bytes(st)
    assert sb["sort"] == 36 * 1000 and sb["project"] == 0
    assert sb["bin"] == 2 * 4 * 1000 + 700 * 86 + 80 * 900 + 8 * 100 * 2
    assert sb["total"] == sb["sort"] + sb["bin"] + sb["raster"]


def test_dump_outputs_frame_and_sample(tmp_path):
    """A 1080p frame is dumped whole; a 4K frame as a seeded pixel sample that fits the budget and is the same every run."""
    bench = _bench_module()
    rng = np.random.default_rng(7)
    small = rng.integers(0, 256, (1080, 1920, 4), dtype=np.uint8)
    out = bench.frame_outputs(small)
    assert list(out) == ["frame"] and out["frame"].dtype == np.float32 and np.array_equal(out["frame"], small)
    big = rng.integers(0, 256, (2160, 3840, 4), dtype=np.uint8)
    a, b = bench.frame_outputs(big), bench.frame_outputs(big.copy())
    assert sorted(a) == ["frame_pixel_index", "frame_pixels"]
    assert a["frame_pixels"].dtype == np.float32 and a["frame_pixel_index"].dtype == np.float64
    assert all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["frame_pixel_index"].astype(np.int64)
    assert np.all(np.diff(idx) > 0) and np.array_equal(a["frame_pixels"], big.reshape(-1, 4)[idx])
    bench.write_outputs(str(tmp_path / "d"), a)
    assert sum(os.path.getsize(tmp_path / "d" / f) for f in os.listdir(tmp_path / "d")) <= 64_000_000


def test_bench_writes_nothing_into_a_read_only_tree(tmp_path):
    """A read-only tree without built libraries: the bench compiles the oracle and the CUDA library in a temporary
    directory, loads them from there and leaves the tree as it was."""
    tree = tmp_path / "tree"
    tree.mkdir()
    shutil.copy2(BENCH, tree / "bench.py")
    for name in ("aframe-gaussian-splatting_b200", "include", "oracle"):  # the sources the bench loads or compiles
        shutil.copytree(os.path.join(ROOT, name), tree / name, ignore=shutil.ignore_patterns("*.so", "__pycache__"))
    before = sorted((d, tuple(sorted(f))) for d, _, f in os.walk(tree))
    for d, _, files in os.walk(tree):
        for f in files:
            os.chmod(os.path.join(d, f), 0o444)
        os.chmod(d, 0o555)
    try:
        ref = subprocess.run([sys.executable, str(tree / "bench.py"), "--impl", "reference", "--splats", "2000", "--steps", "1",
                              "--warmup", "1"], capture_output=True, text=True, timeout=300)
        assert ref.returncode == 0 and json.loads(ref.stdout)["value"] > 0, ref.stderr[-2000:]
        probe = ("import importlib, sys; sys.path.insert(0, sys.argv[1]); import bench; "
                 "gs = importlib.import_module('aframe-gaussian-splatting_b200'); print(bench.load_gsplat(gs)._name)")
        ours = subprocess.run([sys.executable, "-c", probe, str(tree)], capture_output=True, text=True, timeout=600)
        assert ours.returncode == 0, ours.stderr[-2000:]
        assert ours.stdout.strip().endswith("libgsplat_b200.so") and not ours.stdout.strip().startswith(str(tree))
        assert sorted((d, tuple(sorted(f))) for d, _, f in os.walk(tree)) == before
    finally:
        for d, _, _ in os.walk(tree):
            os.chmod(d, 0o755)


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(extra):
    res = subprocess.run([sys.executable, BENCH] + extra, capture_output=True, text=True, timeout=120)
    assert res.returncode == 2 and "error:" in res.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_timed_frame(gs, ctx, tmp_path):
    """--dump-outputs saves the frame the last of the --steps timed steps left on the device: a plain gs_render of the
    same seeded scene gives the same bytes."""
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, BENCH, "--splats", "20000", "--steps", "5", "--warmup", "1", "--no-other-configs",
                          "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 5
    assert os.listdir(out) == ["frame.npy"]
    got = np.load(out / "frame.npy")
    rows, frames, n, w, h = _bench_module().build_scene(gs, "train_1m_1080p", 20000)
    ctx.clear()
    ctx.push_splats(rows)
    exp = ctx.render(frames[0], fmt=gs.GS_FORMAT_RGBA8)
    assert got.dtype == np.float32 and got.shape == (h, w, 4) and np.array_equal(got, exp.astype(np.float32))
