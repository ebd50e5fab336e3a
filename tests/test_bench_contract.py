"""bench.py output checks: the reference arm (`--impl reference`) prints ONE JSON line with the metric / unit / config
of BASELINE.json and the keys a reader of the result needs; N > 1 ranks other than 0 stay silent; `--dump-outputs` writes
the same float32 outputs for the same arguments (GPU)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return [l for l in p.stdout.splitlines() if l.strip()]


def test_reference_arm_json_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == base["metric"] and d["unit"] == "tok/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == []


def test_bad_arguments_are_refused():
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], cwd=ROOT, capture_output=True,
                           text=True, timeout=600)
        assert p.returncode == 2 and "error:" in p.stderr, (argv, p.stderr[-1000:])


def test_dump_outputs_keeps_a_fixed_row_sample_under_the_size_limit(tmp_path):
    dont_write = sys.dont_write_bytecode
    try:
        spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
        bench = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(bench)
    finally:
        sys.dont_write_bytecode = dont_write
    dec = torch.randn(1, 4096).to(torch.float16)
    pre = torch.randn(8192, 4096).to(torch.float16)  # 128 MiB as float32
    bench.dump_outputs(str(tmp_path), {"decode": dec, "prefill": pre})
    d, p = np.load(tmp_path / "decode.npy"), np.load(tmp_path / "prefill.npy")
    assert d.dtype == p.dtype == np.float32 and d.nbytes + p.nbytes <= bench.DUMP_BYTES
    assert np.array_equal(d, dec.float().numpy()) and np.array_equal(p, pre[::3].float().numpy())


@pytest.mark.gpu
def test_dump_outputs_are_the_same_for_the_same_arguments(tmp_path):
    outs = []
    for run in ("a", "b"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--layers", "2",
                            "--prefill-tokens", "128", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)],
                           cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads([ln for ln in p.stdout.splitlines() if ln.strip()][-1])
        assert line["steps"] == 3 and line["finite_outputs"]
        outs.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("decode", "prefill")})
    a, b = outs
    assert a["decode"].shape == (1, 4096) and a["prefill"].shape == (128, 4096)
    for n in a:
        assert a[n].dtype == np.float32 and np.isfinite(a[n]).all() and np.abs(a[n]).max() > 0
        assert np.array_equal(a[n], b[n]), n
