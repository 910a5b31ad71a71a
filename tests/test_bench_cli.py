"""bench.py contract pieces that can be checked without a GPU: the result is the ONLY thing on stdout (libraries such as NCCL print
banners on file descriptor 1 under torchrun), and the reference arm answers for models it has no CPU port for."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_result_line_is_alone_on_stdout():
    code = ("import bench, os; bench.reserve_stdout(); os.write(1, b'NCCL version x.y\\n'); print('python noise'); "
            "bench.emit({'metric': 'm', 'value': 1.0})")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=120)
    assert out.returncode == 0
    assert out.stdout.count("\n") == 1 and json.loads(out.stdout) == {"metric": "m", "value": 1.0}
    assert "NCCL version" in out.stderr and "python noise" in out.stderr


def _run_reference(extra):
    env = dict(os.environ, VQA_BENCH_TINY="1")          # tiny dims: the code path, not the 11 B-parameter model
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "3"] + extra, capture_output=True, text=True, cwd=ROOT,
                         timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout)


def test_reference_arm_measures_every_reported_pair():
    """`--impl reference` (CPU arm): one JSON line, impl=reference, a measured (not extrapolated) pairs/s whose timed region is
    ms_per_step x steps, the config-1 sub-object over the reference's 4 PNGs x 4 prompts, cores = what the process may really use."""
    line = _run_reference([])
    assert line["impl"] == "reference" and line["unit"] == "pairs/s" and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["steps"] == line["timing"]["pairs_timed"] == 3 and line["steps_requested"] == 3
    assert abs(line["ms_per_step"] * line["steps"] / 1000.0 * line["value"] - line["steps"]) < 1e-6 * line["steps"] + 1e-9
    assert "MEASURED" in line["cpu_baseline"]["sample"] and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    c1 = line["config1"]
    assert c1["pairs_timed"] == 16 and "4 reference PNGs x 4 prompts" in c1["sample"] and c1["pair_seconds_min"] <= c1["pair_seconds_median"]


def test_reference_arm_qwen_follows_the_reference_loop():
    line = _run_reference(["--model", "qwen2.5-vl-7b"])
    assert line["impl"] == "reference" and line["value"] > 0 and "generate(max_new_tokens=1" in line["cpu_baseline"]["sample"]
    assert line["steps"] == line["timing"]["pairs_timed"] == 3


def test_reference_arm_qwen_video_shapes():
    line = _run_reference(["--model", "qwen2.5-vl-7b", "--video"])
    assert line["impl"] == "reference" and line["value"] > 0 and "video" in line["metric"]
    line = _run_reference(["--model", "qwen2.5-vl-7b", "--video", "--video-size", "336"])
    assert line["value"] > 0


def test_host_threads_respects_affinity():
    import bench
    phys, logical = bench.host_threads()
    assert 1 <= phys <= logical == len(os.sched_getaffinity(0))


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, cwd=ROOT,
                         timeout=300, env=env)
    assert out.returncode == 0 and out.stdout == ""


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"], ["--ncu", "--dump-outputs", "d"]])
def test_arguments_without_a_timed_engine_step_are_refused(extra, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, cwd=tmp_path, timeout=120)
    assert out.returncode == 2 and out.stdout == "" and not os.listdir(tmp_path), out.stderr[-2000:]


def test_dump_outputs_writes_float32_and_a_fixed_sample_of_large_outputs(tmp_path, monkeypatch):
    import bench
    small, large = torch.linspace(0, 1, 7, dtype=torch.float64), torch.arange(1000, dtype=torch.float32)
    bench.dump_outputs(str(tmp_path / "a"), scores=small)
    got = np.load(tmp_path / "a" / "scores.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.float().numpy())
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 400)                     # room for 100 float32 values
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), scores=large)
    b, c = np.load(tmp_path / "b" / "scores.npy"), np.load(tmp_path / "c" / "scores.npy")
    assert b.dtype == np.float32 and b.nbytes <= 400 and len(b) == 100 and np.array_equal(b, c)
    assert np.all(np.diff(b) > 0) and set(b.tolist()) <= set(large.tolist())      # distinct elements, in index order


@pytest.mark.gpu
def test_dump_outputs_repeat_and_steps_are_the_timed_steps(tmp_path):
    """Two runs with the same arguments see the same seeded inputs: the dumped scores of the last timed step agree, and the JSON line
    reports exactly the requested number of timed steps."""
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    lines, dumps = [], []
    for steps in (1, 2):
        d = tmp_path / f"run{steps}"
        out = subprocess.run([sys.executable, "bench.py", "--model", "clip-flant5-xl", "--batch", "8", "--steps", str(steps), "--warmup", "1",
                              "--no-hf-baseline", "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, cwd=ROOT,
                             timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads(out.stdout))
        dumps.append(np.load(d / "scores.npy"))
    assert [ln["steps"] for ln in lines] == [1, 2]
    for ln, s in zip(lines, dumps):
        assert s.dtype == np.float32 and s.shape == (8,) and np.all(np.isfinite(s)) and np.all((s >= 0) & (s <= 1))
        assert np.allclose(s[:4], ln["sample_scores"], atol=1e-6)
    assert np.allclose(dumps[0], dumps[1], atol=1e-5), (dumps[0], dumps[1])
