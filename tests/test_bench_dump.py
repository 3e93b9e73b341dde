"""bench.py's output dump (``--dump-outputs``) and argument checks, on a CPU training session."""
import importlib.util
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _session_dump(bench, out_dir, steps=2):
    from distributeddeeplearning_b200.workloads.benchmark import BenchmarkSession

    s = BenchmarkSession("resnet18", 2, False)
    w0 = torch.cat([p.detach().reshape(-1).clone() for p in s.model.parameters()])
    for _ in range(steps):
        s.step()
    bench.dump_outputs(s, str(out_dir))
    return s, w0, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_seeded_float32_and_bounded(bench, tmp_path):
    s, w0, a = _session_dump(bench, tmp_path / "a")
    _, _, b = _session_dump(bench, tmp_path / "b")
    assert sorted(a) == ["bn_stats", "loss", "weights"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 64 << 20
    for k in a:                                   # same arguments, same inputs: identical outputs (CPU is deterministic)
        assert np.array_equal(a[k], b[k]), k
    assert a["loss"].shape == () and float(a["loss"]) == float(s.last_loss)
    # resnet18's 11.7 M weights exceed the cap: a sorted fixed sample of the UPDATED weights
    idx = np.sort(np.random.default_rng(0).choice(w0.numel(), bench.DUMP_WEIGHT_SAMPLES, replace=False))
    w = torch.cat([p.detach().reshape(-1) for p in s.model.parameters()]).numpy()
    assert np.array_equal(a["weights"], w[idx]) and not np.array_equal(a["weights"], w0.numpy()[idx])
    bn = sum(m.running_mean.numel() + m.running_var.numel() for m in s.model.modules()
             if isinstance(getattr(m, "running_mean", None), torch.Tensor))
    assert a["bn_stats"].shape == (bn,)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"]])
def test_bench_rejects_empty_timed_region(bench, monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse()


@pytest.mark.parametrize("argv", [["--impl", "reference", "--warmup", "0"],
                                  ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_reference_arm_argument_rules(bench, monkeypatch, argv):
    """The reference arm times from the last warm-up step's event (needs one) and has no output dump."""
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse()


def test_bench_reference_arm_fails_without_staged_script(bench, monkeypatch, tmp_path, capsys):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference"])
    a = bench.parse()
    monkeypatch.setattr(bench, "REF_SCRIPT", str(tmp_path / "missing.py"))
    assert bench.run_reference(a) != 0
    assert "missing" in capsys.readouterr().err


def test_reference_script_staging(tmp_path):
    """build() copies the upstream benchmark script byte for byte; without an upstream checkout it keeps the staged copy."""
    sys.path.insert(0, ROOT)
    from oracle import reference

    up = tmp_path / "upstream"
    src = up / reference.UPSTREAM_SCRIPT
    src.parent.mkdir(parents=True)
    src.write_bytes(b"print('upstream benchmark')\n")
    dst = tmp_path / "_ref"
    assert "staged" in reference.stage(str(up), str(dst))
    assert (dst / reference.SCRIPT).read_bytes() == src.read_bytes()
    assert "keeping" in reference.stage(str(tmp_path / "nowhere"), str(dst))
    assert (dst / reference.SCRIPT).read_bytes() == src.read_bytes()
    assert "unavailable" in reference.stage(str(tmp_path / "nowhere"), str(tmp_path / "empty"))
