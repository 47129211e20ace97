"""bench.py contract: the reference arm prints ONE JSON line with the agreed keys (a bounded CPU run of the oracle
port), non-zero ranks of a torchrun launch stay silent, the CUDA arm refuses to run without a device instead of
falling back, and --dump-outputs writes what the CUDA arm's last timed step computed (on the GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.pop("RANK", None), e.pop("WORLD_SIZE", None), e.pop("LOCAL_RANK", None)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          env=e, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    res = _run(["--impl", "reference", "--steps", "2", "--warmup", "1"])
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "edges/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("GripNet fwd+bwd edges/sec") and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] >= 2 and d["gpu_launches"] == 0
    assert d["vs_baseline"] is None and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "epochs" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    res = _run(["--impl", "reference", "--gpus", "2", "--steps", "2"], env={"RANK": "1", "WORLD_SIZE": "2"}, timeout=120)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_dump_outputs_keeps_its_budget_and_samples_fixed_rows(tmp_path):
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    big = torch.randn(250_000, 80, generator=g)                    # 80 MB: over the whole budget alone
    big[:, 0] = torch.arange(big.size(0), dtype=torch.float32)     # row id in column 0
    named = [("loss", torch.tensor([0.5])), ("z", big), ("grad.w", torch.randn(16, 80, generator=g))]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), named)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["grad.w.npy", "loss.npy", "z.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 1000 * 1000
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "grad.w.npy"), named[2][1].numpy())
    z = np.load(tmp_path / "a" / "z.npy")
    rows = z[:, 0].astype(np.int64)
    assert 0 < len(rows) < big.size(0) and np.all(np.diff(rows) > 0)
    assert np.array_equal(z, big.numpy()[rows])


def test_reference_arm_refuses_dump_outputs(tmp_path):
    res = _run(["--impl", "reference", "--steps", "2", "--dump-outputs", str(tmp_path / "d")], timeout=120)
    assert res.returncode != 0 and res.stdout.strip() == ""
    assert "--dump-outputs applies to the CUDA arm" in res.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_of_two_runs_agree_and_line_up_with_the_model(tmp_path):
    """Two runs with the same arguments dump the same arrays; each file holds what its name says (the loss of
    the JSON line, the class probabilities, the final embedding) and there is one gradient per parameter."""
    import numpy as np
    import synthdata
    from gripnet_b200.pipelines import ChainModel
    dumps = []
    for d in ("a", "b"):
        res = _run(["--workload", "scaled-small", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path / d)])
        assert res.returncode == 0, res.stderr[-3000:]
        line = json.loads([l for l in res.stdout.splitlines() if l.strip()][-1])
        dump = {f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)}
        assert line["steps"] == 2 and dump["loss"].shape == (1,) and float(dump["loss"][0]) == line["loss"]
        dumps.append(dump)
    a, b = dumps
    c = synthdata.CHAIN_SMALL
    params = dict(ChainModel(c["n_a"], c["n_b"], c["n_c"], c["n_class"]).named_parameters())
    assert sorted(a) == sorted(b) and {"loss", "z", "score"} <= set(a)
    grads = {k[len("grad."):] for k in a if k.startswith("grad.")}
    assert grads == set(params) and len(a) == 3 + len(params)
    for k in grads:
        assert a["grad." + k].shape == tuple(params[k].shape) and np.isfinite(a["grad." + k]).all(), k
    assert a["score"].shape[1] == c["n_class"] and np.allclose(a["score"].sum(1), 1.0, atol=1e-5)
    assert a["z"].shape[0] == c["n_c"] and a["z"].shape[1] == params["mcip.weight"].shape[0]
    for k in a:
        assert a[k].dtype == np.float32 and a[k].shape == b[k].shape, k
        assert np.abs(a[k] - b[k]).max(initial=0.0) <= 1e-5 * np.abs(b[k]).max(initial=0.0), k


def test_cuda_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    res = _run(["--steps", "2"], timeout=300)
    assert res.returncode != 0 and res.stdout.strip() == ""
    assert "no CUDA device" in res.stderr and "no CPU fallback" in res.stderr
