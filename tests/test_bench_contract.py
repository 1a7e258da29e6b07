"""bench.py's host logic and the JSON-line contract of its reference arm (no GPU needed: the reference arm times the
oracle's cv2-backed driver on the host cores, which is the one place outside tests/ that may execute oracle/)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _args(argv):
    import bench
    old = sys.argv
    sys.argv = ["bench.py"] + argv
    try:
        return bench.parse_args()
    finally:
        sys.argv = old


def test_defaults_are_baseline_config_1_on_one_gpu():
    a = _args([])
    assert (a.gpus, a.impl, a.config_index) == (1, "ours", 1)
    assert a.warmup >= 3 and a.steps >= 1
    assert a.shape == [512, 1024, 1024] and a.sigma == (2.0, 2.0, 2.0) and (a.levels, a.winsize) == (3, 5)
    assert not a.customised and not a.no_of and not a.recompute_flow


def test_configs_follow_baseline_json():
    import bench
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        base = json.load(f)
    assert len(bench.CONFIGS) == len(base["configs"])
    a4 = _args(["--config", "cfg4"])
    assert a4.shape == [256, 2048, 2048] and a4.sigma == (4.0, 2.0, 2.0) and (a4.levels, a4.winsize) == (5, 9)
    assert a4.dtype == "uint8" and a4.config_index == 3
    assert _args(["--config", "cfg3"]).no_of
    assert _args(["--sigma", "1.5"]).customised and _args(["--recompute-flow"]).customised


def test_byte_model_matches_survey_formula():
    import bench
    # SURVEY.md section 8d: cfg 2 = 3 passes x 3811.2 B/voxel, cfg 4 = 15 221.9 B/voxel, no-OF = 8 B per pass
    assert bench.model_bytes_per_voxel((512, 1024, 1024), (2.0, 2.0, 2.0), 3, False) == pytest.approx(11433.6, abs=0.05)
    assert bench.model_bytes_per_voxel((256, 2048, 2048), (4.0, 2.0, 2.0), 5, False) == pytest.approx(15221.9, abs=0.05)
    assert bench.model_bytes_per_voxel((512, 1024, 1024), (2.0, 2.0, 2.0), 3, True) == 24.0
    # level cropping: a 64 x 256 slice stops at 32 x 128 (two extra levels), like cv2
    assert bench.level_sizes(64, 256, 3) == [(64, 256), (32, 128)]
    assert bench.level_sizes(1024, 1024, 3) == [(1024, 1024), (512, 512), (256, 256), (128, 128)]


def test_hash_keys_distinguish_modes():
    import bench
    keys = {bench.hash_key(_args(v), e) for v, e in (([], True), (["--recompute-flow"], True), (["--no-of"], True),
                                                     (["--no-of"], False), (["--config", "cfg4"], True))}
    assert len(keys) == 5
    with open(os.path.join(ROOT, "profiles", "expected_hashes.json")) as f:
        expected = json.load(f)
    assert bench.hash_key(_args([]), True) in expected and bench.hash_key(_args(["--config", "cfg5"]), True) in expected


def test_reference_arm_prints_the_contract_line():
    pytest.importorskip("cv2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--shape", "18", "48", "64",
                          "--sigma", "1", "--steps", "1", "--warmup", "0", "--cpu-slices", "2"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Mvoxel/s" and line["higher_is_better"] is True
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["config"]["shape"] == [18, 48, 64] and line["vs_baseline"] is None


def test_steps_and_dump_outputs_arguments():
    assert _args(["--steps", "7"]).steps == 7 and _args([]).dump_outputs is None
    assert _args(["--dump-outputs", "out"]).dump_outputs == "out"
    for bad in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        with pytest.raises(SystemExit):
            _args(bad)


def test_dump_sample_is_fixed_and_spans_the_volume():
    import bench
    assert np.array_equal(bench.dump_sample_index(1000), np.arange(1000))
    nvox = 512 * 1024 * 1024
    idx = bench.dump_sample_index(nvox)
    assert idx.size == bench.DUMP_VOXELS and 2 * idx.size * 4 <= 64 << 20     # zy + zyx in float32
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < nvox
    assert idx[-1] >= nvox - 2 * (nvox // idx.size)                          # reaches the end of the volume
    assert np.array_equal(idx, bench.dump_sample_index(nvox))


def _dump_worker(rank, world, port, shape, budget, out_dir):
    import torch
    import torch.distributed as dist
    import bench
    from flowdenoising_b200.dist import split_range
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        bench.DUMP_VOXELS = budget
        vol = np.arange(np.prod(shape), dtype=np.float32).reshape(shape)
        z0, z1 = split_range(shape[0], world, rank)
        bench.dump_outputs(out_dir, {"zyx": torch.from_numpy(vol[z0:z1].copy())}, shape, (z0, z1), rank, world)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,budget", [(1, 10_000), (1, 500), (3, 10_000), (3, 500)])
def test_dump_outputs_assembles_rank_slabs(tmp_path, monkeypatch, world, budget):
    """Whole volume within the budget (shaped [Z][Y][X]), else the seeded sample in index order; uneven Z-slabs."""
    import socket
    pytest.importorskip("torch")
    import torch.multiprocessing as mp
    import bench
    shape = (11, 13, 10)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_dump_worker, args=(world, port, shape, budget, str(tmp_path)), nprocs=world, join=True)
    got = np.load(tmp_path / "zyx.npy")
    vol = np.arange(np.prod(shape), dtype=np.float32).reshape(shape)
    monkeypatch.setattr(bench, "DUMP_VOXELS", budget)
    want = vol if vol.size <= budget else vol.ravel()[bench.dump_sample_index(vol.size)]
    assert got.dtype == np.float32 and got.shape == want.shape and np.array_equal(got, want)
