"""GPU tests (B200): every native kernel vs a plain PyTorch fp32 reference of the same op, the fused engine,
whole-model gradients, and the bench/smoke entry points.  Each group runs in a subprocess (tools/gpu_diag.py) so a
device-side trap in one kernel cannot poison the CUDA context of the others."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _group(name, timeout=600, env=None):
    e = dict(os.environ)
    e.update(env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gpu_diag.py"), "--group", name], cwd=ROOT,
                       capture_output=True, text=True, timeout=timeout, env=e)
    out = r.stdout + r.stderr
    tail = "\n".join(l for l in out.splitlines() if "FAIL" in l or "Error" in l)[:3000] + "\n...\n" + out[-3000:]
    assert r.returncode == 0, tail
    assert "FAIL" not in r.stdout, tail


@pytest.mark.parametrize("group", ["elementwise", "gemm", "conv_fwd", "conv_dgrad", "conv_wgrad", "linear", "bn", "sgd", "zoo", "zoograd", "conv_generic", "graph", "fp8", "benchshape"])
def test_kernel_group(group):
    """Default configuration: the per-shape autotuner picks among the kernel variants (a variant that dead-locks on a
    shape makes the group fail: gpu_diag reports the tuner's rejections and any pipeline timeout).  `benchshape` runs
    EVERY variant on batch-256 ResNet-50 layers with an element-wise (atol + rtol*|ref|) check; `fp8` covers the
    e4m3 / e5m2 operand path."""
    _group(group)


@pytest.mark.parametrize("mode", ["2", "3", "4"])
def test_deep_ring_kernel_forced(mode):
    """The deep-ring kernel (one CTA / one cta_group::2 pair per SM, chunked epilogue) forced onto every TMA-fed shape:
    2 = CTA pairs wherever possible, 3 = single CTAs with up to 256-wide tiles, 4 = single CTAs, tiles <= 128 wide."""
    for group in ("gemm", "conv_fwd", "conv_dgrad", "conv_generic"):
        _group(group, timeout=300, env={"DDL_CONV_DEEP": mode, "DDL_CONV_AUTOTUNE": "0"})


def test_persistent_kernel_forced():
    """The CL = 0 persistent kernel (two CTAs per SM, double-buffered TMEM) forced onto every TMA-fed shape — in the
    benchmark step it is chosen only for layers with >= 7 waves of tiles, which the small test shapes never reach."""
    for group in ("gemm", "conv_fwd", "conv_dgrad", "conv_generic"):
        _group(group, timeout=300, env={"DDL_CONV_PERSISTENT": "2", "DDL_CONV_DEEP": "0", "DDL_CONV_AUTOTUNE": "0"})


@pytest.mark.parametrize("mode", ["1", "2"])
def test_cluster_pair_kernels(mode):
    """Thread-block-cluster variants of the persistent conv kernel, forced onto every TMA-fed shape: 1 = CTA pairs that
    TMA-multicast the weight tile, 2 = cta_group::2 pair MMAs (M = 256 across two SMs, half of B per SM)."""
    for group in ("gemm", "conv_dgrad"):
        _group(group, timeout=300, env={"DDL_CONV_CLUSTER": mode, "DDL_CONV_PERSISTENT": "2"})


def test_whole_model_gradients():
    _group("model", timeout=900)


def test_native_module_loaded_and_counts_launches():
    code = ("import torch, sys; sys.path.insert(0, %r)\n"
            "from distributeddeeplearning_b200 import _ext\n"
            "from distributeddeeplearning_b200.ops import native as nv\n"
            "n0 = _ext.launch_count(); x = nv.philox_images(2, 8, 8, 1); torch.cuda.synchronize()\n"
            "assert _ext.launch_count() == n0 + 1\n"
            "import distributeddeeplearning_b200._C as m; print(m.__file__)\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip().endswith("_C.so")


def test_smoke_entry():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "__graft_entry__.py"), "smoke"], cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    assert "smoke ok" in r.stdout


def test_bench_contract_small():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--batch-size", "32"],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    out = json.loads(line)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"):
        assert key in out, key
    assert out["value"] > 0 and out["gpu_launches"] > 0 and out["e2e"]["value"] > 0
    assert out["e2e"]["h2d_bytes_per_step"] == 32 * 224 * 224 * 3 + 32 * 8


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs: the loss and (sampled) updated weights of the last timed step, float32, at most 64 MB."""
    import numpy as np

    def bench(steps, d):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                            "--batch-size", "16", "--no-e2e", "--dump-outputs", str(d)],
                           cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
        return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])

    d = tmp_path / "dump"
    out, out4 = bench(2, d), bench(4, tmp_path / "dump4")
    # --steps sets the number of timed steps: the timed region's kernel launches double from 2 to 4 steps
    assert out["steps"] == 2 and out["gpu_launches"] > 0 and out4["gpu_launches"] == 2 * out["gpu_launches"]
    a = {f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))}
    assert sorted(a) == ["bn_stats", "loss", "weights"] and all(v.dtype == np.float32 for v in a.values())
    assert sum((d / f).stat().st_size for f in os.listdir(d)) <= 64 << 20
    assert float(a["loss"]) == pytest.approx(out["final_loss"], rel=1e-6)
    assert a["weights"].size == 1 << 22 and np.isfinite(a["weights"]).all() and np.isfinite(a["bn_stats"]).all()


def _launch(module, argv, gpus, env=None, timeout=900):
    import io

    sys.path.insert(0, ROOT)
    from distributeddeeplearning_b200.cli import launcher

    out, err = io.StringIO(), io.StringIO()
    e = {"PYTHONPATH": ROOT}
    e.update(env or {})
    res = launcher.launch(module, argv, gpus=gpus, record=False, stdout=out, stderr=err, timeout=timeout, env=e)
    return res, out.getvalue(), err.getvalue()


def test_imagenet_trainer_synthetic_gpu(tmp_path):
    """Reference PyTorch_imagenet trainer surface on the native kernels: LR warm-up, epoch log lines, checkpoint."""
    res, out, err = _launch("distributeddeeplearning_b200.workloads.imagenet",
                            ["--epochs", "1", "--batch_size", "16", "--model", "resnet50",
                             "--save_filepath", str(tmp_path / "ck-{epoch}.pt")], gpus=1, env={"FAKE_DATA_LENGTH": "64"})
    assert res.returncode == 0, (out + err)[-3000:]
    assert "Training epoch 0 took" in out and "Total images/sec:" in out
    assert (tmp_path / "ck-1.pt").exists()


def test_hvd_trainer_checkpoint_resume_gpu(tmp_path):
    """Reference PyTorch_hvd trainer: checkpoints every epoch, second launch resumes from the latest one; the per-step
    metric allreduces ride in the last gradient bucket (FusedSGD.piggyback)."""
    fmt = str(tmp_path / "checkpoint-{epoch}.pth.tar")
    common = ["--batch-size", "16", "--model", "resnet50", "--synthetic-length", "32", "--checkpoint-format", fmt,
              "--log-dir", str(tmp_path / "logs")]
    for epochs in ("1", "2"):
        res, out, err = _launch("distributeddeeplearning_b200.workloads.hvd_imagenet", ["--epochs", epochs] + common, gpus=1)
        assert res.returncode == 0, (out + err)[-3000:]
    assert os.path.exists(fmt.format(epoch=1)) and os.path.exists(fmt.format(epoch=2))


def test_cuda_graph_replay_matches_eager():
    """The captured step (forward, backward with side-stream weight gradients, fused SGD buckets) replays to the same
    loss trajectory as the eager step."""
    code = ("import sys, torch; sys.path.insert(0, %r)\n"
            "from distributeddeeplearning_b200.parallel import dist\n"
            "from distributeddeeplearning_b200.workloads.benchmark import BenchmarkSession\n"
            "dist.init()\n"
            "def run(graph):\n"
            "    torch.manual_seed(0)\n"
            "    s = BenchmarkSession('resnet18', 16, True, lr=0.05, momentum=0.9)\n"
            "    out = [float(s.step()) for _ in range(3)]\n"
            "    if graph: assert s.enable_graph(warmup=1), 'capture failed'\n"
            "    else: out.append(float(s.step()))\n"
            "    out += [float(s.step()) for _ in range(4)]\n"
            "    return out[-4:]\n"
            "a, b = run(False), run(True)\n"
            "print(a, b)\n"
            # bf16 steps are not bit-reproducible run to run (atomics order): 5 % bounds that; a capture bug is far off
            "assert all(abs(x - y) < 5e-2 * max(1.0, abs(x)) for x, y in zip(a, b)), (a, b)\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]


def test_multi_rank_fused_engine():
    """NVLink peer-memory engine on however many GPUs the box has (>= 2): P2P + NVLS transports, fp32 + bf16 wire,
    piggy-backed scalars, artificial block / rank skew, debug invariants, and the one-step equivalence of an N-rank
    ResNet-50 step on identical data with a single-rank step (parallel/selfcheck.py)."""
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (bench.py runs the same checks before timing whenever it is launched on N > 1)")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", "29731", os.path.join(ROOT, "tools", "comm_test.py"),
                        "--no-sweep", "--model-check"], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ENGINE CHECKS: all ok" in r.stdout, (r.stdout + r.stderr)[-3000:]


@pytest.mark.parametrize("native_hooks", ["1", "0"])
def test_single_rank_local_engine_equals_torch_sgd(native_hooks):
    """One-GPU part of the engine contract: a FusedSGD step (world 1, `local` mode included) applies exactly
    torch.optim.SGD's update, and its state_dict round-trips through torch.optim.SGD's loader and back — with the
    native StepLauncher sequencing the bucket launches (default) and with the Python sequencing (DDL_NATIVE_HOOKS=0)."""
    code = ("import sys, torch; sys.path.insert(0, %r)\n"
            "from distributeddeeplearning_b200.parallel import dist\n"
            "from distributeddeeplearning_b200.parallel.engine import FusedSGD\n"
            "dist.init()\n"
            "torch.manual_seed(0)\n"
            "shapes = [(64, 3, 7, 7), (10, 64), (10,), (32, 16, 3, 3)]\n"
            "ps = [torch.nn.Parameter(torch.randn(s, device='cuda')) for s in shapes]\n"
            "qs = [torch.nn.Parameter(p.detach().clone()) for p in ps]\n"
            "a = FusedSGD(ps, lr=0.1, momentum=0.9, weight_decay=1e-3, local=True)\n"
            "b = torch.optim.SGD(qs, lr=0.1, momentum=0.9, weight_decay=1e-3)\n"
            "for it in range(3):\n"
            "    for p, q in zip(ps, qs):\n"
            "        g = torch.randn_like(q)\n"
            "        p.grad.add_(g.view_as(p.grad)); q.grad = g.clone(); p._ddl_ready()\n"
            "    a.step(); b.step()\n"
            "torch.cuda.synchronize()\n"
            "for p, q in zip(ps, qs): assert torch.allclose(p, q, rtol=1e-5, atol=1e-6), (p - q).abs().max()\n"
            "sd = a.state_dict()\n"
            "assert sd['param_groups'][0]['params'] == [0, 1, 2, 3] and set(sd['state']) == {0, 1, 2, 3}\n"
            "c = torch.optim.SGD([torch.nn.Parameter(q.detach().clone()) for q in qs], lr=0.5)\n"
            "c.load_state_dict(sd)                                  # torch accepts the fused engine's checkpoint\n"
            "for i, q in enumerate(c.param_groups[0]['params']):\n"
            "    assert torch.allclose(c.state[q]['momentum_buffer'].cuda(), b.state[qs[i]]['momentum_buffer'], rtol=1e-5, atol=1e-6)\n"
            "a2 = FusedSGD([torch.nn.Parameter(q.detach().clone()) for q in qs], lr=0.1, momentum=0.9, local=True)\n"
            "a2.load_state_dict(b.state_dict())                     # and the engine accepts torch's\n"
            "m = a2.state_dict()['state']\n"
            "for i in range(4): assert torch.allclose(m[i]['momentum_buffer'].cuda(), b.state[qs[i]]['momentum_buffer'], rtol=1e-5, atol=1e-6)\n"
            "assert (a._launcher is not None) == (%r == '1')\n"
            "print('engine == torch.optim.SGD')\n" % (ROOT, native_hooks))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env=dict(os.environ, DDL_NATIVE_HOOKS=native_hooks))
    assert r.returncode == 0 and "engine == torch.optim.SGD" in r.stdout, (r.stdout + r.stderr)[-3000:]


def test_fp8_loss_curve_tracks_bf16():
    """BASELINE config #3: 200 ResNet-50 steps with fp8 tensor-core operands follow the bf16 loss curve."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fp8_parity.py"), "--steps", "200", "--batch", "32"],
                       cwd=ROOT, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0 and "FP8 PARITY: ok" in r.stdout, (r.stdout + r.stderr)[-3000:]
