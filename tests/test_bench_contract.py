"""bench.py: the JSON line of the reference arm (CPU), and what --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
            "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(extra, env=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--cpu-sample-n", "48", "--no-ref-table"] + extra
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def test_reference_arm_json_line():
    lines = _run([])
    rec = json.loads(lines[-1])
    assert REQUIRED <= set(rec)
    assert rec["impl"] == "reference" and rec["unit"] == "pairs/s" and rec["higher_is_better"] is True
    assert rec["vs_baseline"] is None and rec["value"] > 0
    # the unmodified loss.py (source tree here, oracle/_ref on the GPU box) whenever it is reachable
    from oracle.ref_loader import reference_available
    assert rec["cpu_baseline"]["kind"] == ("reference" if reference_available() else "port")
    assert rec["cpu_baseline"]["cores"] >= 1 and "cpu_model" in rec
    assert rec["e2e"] == {"value": rec["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in rec["config"]


def test_reference_arm_falls_back_to_the_port_without_the_reference(tmp_path):
    env = dict(os.environ, SUPCON_REFERENCE_ROOT=str(tmp_path), SUPCON_REFERENCE_DISABLE="1")
    rec = json.loads(_run([], env=env)[-1])
    assert rec["cpu_baseline"]["kind"] == "port"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    assert _run(["--gpus", "2"], env=env) == []


def test_dump_outputs_keeps_a_fixed_sample_of_whole_rows(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_DZ_BYTES", 64 * 8 * 4)
    dz = torch.arange(200).repeat_interleave(8).reshape(200, 8).to(torch.bfloat16)    # row i holds i
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), torch.tensor(1.5), dz)
    a = np.load(tmp_path / "a" / "dz.npy")
    assert a.dtype == np.float32 and a.shape == (64, 8)
    assert (a == a[:, :1]).all() and (np.diff(a[:, 0]) > 0).all()          # whole rows, ascending, distinct
    assert np.array_equal(a, np.load(tmp_path / "b" / "dz.npy"))
    loss = np.load(tmp_path / "a" / "loss.npy")
    assert loss.dtype == np.float32 and float(loss) == 1.5
    bench.dump_outputs(str(tmp_path / "c"), torch.tensor(1.5), dz[:64])
    assert np.array_equal(np.load(tmp_path / "c" / "dz.npy"), dz[:64].float().numpy())


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_steps_loss_and_gradient(cuda_device, tmp_path):
    """The dumped loss and d loss / d z are those of the timed module call, on bench.py's seeded inputs."""
    from bench import synth
    from oracle import supcon_oracle as O
    n = 4096
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--batch-n", str(n), "--steps", "3", "--warmup", "1",
           "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    rec = json.loads(out.stdout.strip().splitlines()[-1])
    loss, dz = np.load(tmp_path / "loss.npy"), np.load(tmp_path / "dz.npy")
    assert loss.dtype == dz.dtype == np.float32 and dz.shape == (n, 256)
    assert float(loss) == pytest.approx(rec["loss"], rel=1e-6)
    z, y = synth(n, 256, torch.bfloat16)
    ref = O.closed_form(z.float(), y, temperature=0.07, similarity="cosine", topk_neg=15, alpha=0.0)
    assert float(loss) == pytest.approx(ref["loss"], rel=1e-4)
    assert float((torch.from_numpy(dz).double() - ref["dz"]).norm() / ref["dz"].norm()) < 1e-2
