"""bench.py's output contract, exercised on CPU through the reference arm (tiny shapes)."""
import json
import os
import subprocess
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "impl"}

pytestmark = pytest.mark.timeout(300)


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "pytensor_federated")),
                    reason="upstream package not installed (build() installs it into oracle/_ref)")
def test_reference_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    import numpy as np

    env = dict(os.environ, B200FED_REF_ALLOW_CPU="1")
    res = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "2000", "--features", "64",
         "--shards", "2", "--steps", "4", "--warmup", "3", "--dump-outputs", str(tmp_path)],
        cwd=ROOT, env=env, capture_output=True, text=True, timeout=240,
    )
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert REQUIRED <= set(line)
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["scaling"] == "strong"
    assert line["steps"] == 4 and line["warmup"] == 3 and line["value"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert "unmodified reference" in line["config"]["note"]
    logp, d_ic, d_beta = (np.load(tmp_path / f"{n}.npy") for n in ("logp", "grad_0", "grad_1"))
    assert logp.dtype == np.float64 and logp.shape == () and np.isfinite(logp)
    assert d_ic.shape == (1,) and d_beta.shape == (64,) and np.isfinite(d_beta).all()


@pytest.mark.gpu
def test_product_arm_times_exactly_steps_and_dumps_the_last_timed_result(tmp_path):
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import bench

    out = tmp_path / "dump"
    rows, features, shards, steps, warmup = 20000, 64, 2, 3, 2
    res = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(rows), "--features", str(features),
         "--shards", str(shards), "--steps", str(steps), "--warmup", str(warmup), "--dump-outputs", str(out)],
        cwd=ROOT, capture_output=True, text=True, timeout=240,
    )
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
    assert REQUIRED <= set(line) and line["verified"]
    # one fused launch per evaluation: the device-timed region ran exactly --steps evaluations
    assert line["gpu_launches"] == steps and line["e2e"]["steps"] == steps
    got = [np.load(out / f"{n}.npy") for n in ("logp", "grad_0", "grad_1")]
    assert [g.dtype for g in got] == [np.float64] * 3 and [g.shape for g in got] == [(), (1,), (features,)]
    # the same seeded workload: the timed steps evaluate thetas[warmup] (after the two verification draws)
    args = types.SimpleNamespace(config="glm", rows=rows, features=features, shards=shards, chains=1, kernel="auto")
    model, draw_theta, _ = bench.build_workload(args, 1, 0, torch.device("cuda", 0))
    theta = [draw_theta() for _ in range(2 + warmup + 1)][-1]
    want = model.unpack_result(np.asarray(model.reference_partial(theta, dtype=torch.float64)), model.call_context(theta))
    assert abs(got[0] - want[0]) <= 2e-4 * abs(want[0])
    for g, w in zip(got[1:], want[1:]):
        assert np.abs(g - w).max() <= 2e-4 * np.abs(w).max()


def test_reference_arm_reports_unavailable_instead_of_failing(tmp_path):
    """Without the install the arm must print {"impl": "reference", "unavailable": ...} and exit 0."""
    code = (
        "import sys, json; sys.path.insert(0, %r); import reference_arm as r; "
        "r._paths = lambda: None; "
        "import types; "
        "r.main(types.SimpleNamespace(shards=2, rows=10, features=64, steps=1, warmup=1, out=None))"
    ) % os.path.join(ROOT, "baseline")
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    res = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr[-1500:]
    line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][0])
    assert line["impl"] == "reference" and "unavailable" in line
