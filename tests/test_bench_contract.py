"""bench.py contract checks that run without a GPU: the reference arm prints one well-formed JSON line (CPU oracle port,
the one place besides tests/ and smoke() that may execute oracle/), and our arm refuses to run without a B200."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=900):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    out = _run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1"], env={"LBC_CPU_THREADS": "8"})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["config"]["workload"] == "config2"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == dict(value=d["value"], unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)


def test_reference_arm_only_rank0_works_under_torchrun_env():
    out = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip() == ""


def test_reference_arm_times_the_requested_steps():
    out = _run(["--impl", "reference", "--steps", "21", "--warmup", "0", "--batch", "8"], env={"LBC_CPU_THREADS": "8"})
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")][-1])
    assert d["steps"] == 21 and d["warmup"] == 0
    assert d["cpu_baseline"]["batch8"]["timed_steps"] == 21 and d["cpu_baseline"]["like_for_like"] is None


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = _run(args)
        assert out.returncode == 2 and "error:" in out.stderr, args


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs writes the last timed step's outputs; --steps sets every timed loop; the same arguments give the
    same outputs, bit for bit: every reduction of the training step adds in a fixed order, so nothing differs between runs
    for Adam to amplify over the steps."""
    dumps = []
    for run in range(2):
        d = tmp_path / ("run%d" % run)
        out = _run(["--steps", "8", "--warmup", "2", "--batch", "8", "--no-cpu-baseline", "--dump-outputs", str(d)])
        assert out.returncode == 0, out.stderr[-2000:]
        res = json.loads([ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")][-1])
        assert res["steps"] == 8 and res["e2e"]["steps"] == 8
        a = {f.stem: np.load(f) for f in d.glob("*.npy")}
        assert sorted(a) == ["buffers", "grads_sample", "loss", "params_sample", "pred", "preds"]
        assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
        assert sum(v.nbytes for v in a.values()) <= 64 << 20
        assert a["pred"].shape == (8, 5, 2) and a["preds"].shape == (8, 4, 5, 2)
        assert a["params_sample"].shape == a["grads_sample"].shape == (1 << 20,)
        assert float(a["loss"]) == np.float32(res["last_loss"])
        assert np.abs(a["grads_sample"]).max() > 0
        dumps.append(a)
    for k in dumps[0]:
        assert np.array_equal(dumps[0][k], dumps[1][k]), (k, float(np.abs(dumps[0][k] - dumps[1][k]).max()))


def test_our_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    out = _run(["--steps", "1", "--warmup", "1"])
    assert out.returncode != 0
    assert "needs a B200" in out.stderr
