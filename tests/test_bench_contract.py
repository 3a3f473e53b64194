"""The bench line contract, checked on the one arm that runs without a GPU: `bench.py --impl reference` (the reference's
step on the host cores, a bounded sample: the unmodified reference code when oracle/_ref/refpy_cpu is built, else the
oracle port).  Keys and invariants are the ones the driver reads."""
import json
import os
import tempfile
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import reference_step


@pytest.mark.parametrize("kind", ["reference", "port"])
def test_reference_arm_prints_one_contract_line(kind):
    if kind == "reference" and not reference_step.available():
        pytest.skip("oracle/_ref/refpy_cpu not built (python -m oracle.build_ref)")
    env = dict(os.environ, GG_CPU_KIND=kind)
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                           "--warmup", "0", "--cpu-batch", "1"], capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and lines[0].startswith("{"), "stdout must carry exactly ONE JSON line:\n" + proc.stdout[-2000:]
    line = json.loads(lines[0])
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert line["impl"] == "reference"
    assert line["metric"] == "gangealing_train_images_per_sec_256" and "images/sec at 256" in baseline["metric"]
    assert line["unit"] == "images/s" and line["higher_is_better"] is True and line["scaling"] == "weak"
    assert line["n_gpus"] == 1 and line["steps"] >= 1 and line["value"] > 0 and line["ms_per_step"] > 0
    assert line["vs_baseline"] is None and line["dtype"] == "f32" and line["data"] == "synthetic"
    assert isinstance(line["config"], dict) and "workload" in line["config"] and "model" not in line["config"]
    cpu = line["cpu_baseline"]
    assert cpu["kind"] == kind and cpu["cores"] >= 1 and cpu["value"] == line["value"] and cpu["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == line["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_non_zero_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                           "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert proc.returncode == 0
    assert not [l for l in proc.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_writes_the_same_arrays_on_every_run():
    """bench.py --dump-outputs DIR: float32 / float64 .npy files, 64 MB at most, and the same bits from two runs with the
    same arguments."""
    import numpy as np
    dumps = []
    with tempfile.TemporaryDirectory() as tmp:
        for run in range(2):
            out = os.path.join(tmp, "run%d" % run)
            proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0",
                                   "--batch", "4", "--no-extra", "--no-cpu-baseline", "--dump-outputs", out],
                                  capture_output=True, text=True, timeout=900, cwd=ROOT)
            assert proc.returncode == 0, proc.stderr[-2000:]
            line = json.loads(proc.stdout.strip().splitlines()[-1])
            assert line["steps"] == 2 and line["config"]["cudnn"].startswith("deterministic")
            files = sorted(os.listdir(out))
            assert files == ["loss_f.npy", "loss_p.npy", "loss_tv.npy", "stn_ema_params.npy", "stn_params.npy"]
            assert sum(os.path.getsize(os.path.join(out, f)) for f in files) <= 64 << 20
            arrays = {f: np.load(os.path.join(out, f)) for f in files}
            assert all(a.dtype in (np.float32, np.float64) and a.size > 0 for a in arrays.values())
            dumps.append(arrays)
    for f in dumps[0]:
        assert np.array_equal(dumps[0][f], dumps[1][f]), f
