#!/usr/bin/env python
"""Headline benchmark: ResNet-50 synthetic-ImageNet training throughput (images/sec, device-timed,
max over ranks) — the metric/config BASELINE.json names ("PyTorch_benchmark ResNet-50 bf16 synthetic,
batch 256/GPU").

    python bench.py --gpus N --steps K --warmup W            # this repo (N>1: run under torchrun, or
                                                             #  bench.py re-launches itself with the local launcher)
    python bench.py --impl reference --gpus N ...            # the reference's unmodified script (oracle/_ref, staged by build())

Prints ONE JSON line on rank 0.  Timed region = exactly K full training steps (forward, loss,
backward, fused allreduce + SGD update) between barrier + cuda.synchronize on both sides, CUDA events
on the launching stream, max over ranks.  Per-step working set (>5 GB of activations at batch 256)
exceeds the 126 MB L2, so no explicit L2 flush is needed ("l2": "working_set_exceeds_l2").
``e2e`` repeats the measurement through the public API with, every step, a host->device copy of that
step's inputs from pinned memory (uint8 NHWC images, the decoded-JPEG format, + int64 labels) and a
device->host read of the step's loss.

``--dump-outputs DIR`` writes, after the K timed steps (before ``e2e`` trains on), what the last timed step handed
back on rank 0 as float32 ``.npy`` files (see ``dump_outputs``).  Model init and the synthetic batch are seeded, so
two builds run with the same arguments can be compared output for output.  The bf16 step is not bit-reproducible
(fp32 atomics order: profiles/step_reproducibility.md), so compare against the spread of two runs of the same build.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

REF_SCRIPT = os.path.join(HERE, "oracle", "_ref", "pytorch_synthetic_benchmark.py")      # oracle/reference.py
METRIC = "resnet50_synthetic_train_images_per_sec"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", choices=["ours", "reference"], default="ours")
    p.add_argument("--model", default="resnet50")
    p.add_argument("--batch-size", type=int, default=256, help="per-GPU batch (BASELINE config: 256)")
    p.add_argument("--no-e2e", action="store_true", help="skip the end-to-end (H2D/D2H per step) measurement")
    p.add_argument("--fp16-allreduce", action="store_true")
    p.add_argument("--no-selfcheck", action="store_true",
                   help="N>1: skip the engine self-checks that run before the timed region")
    p.add_argument("--cuda-graph", choices=["on", "off"], default=os.environ.get("DDL_BENCH_GRAPH", "on"),
                   help="replay the whole training step from one captured CUDA graph (falls back to eager if capture fails)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the loss and updated weights of the last timed step to DIR/<name>.npy")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if a.impl == "reference" and a.warmup < 1:
        p.error("--impl reference times from the end of the last warm-up step: --warmup must be >= 1")
    if a.impl == "reference" and a.dump_outputs:
        p.error("--dump-outputs applies to this repo's arm only, not --impl reference")
    return a


DUMP_WEIGHT_SAMPLES = 1 << 22       # 16 MiB of float32; ResNet-50 has 25.6 M weights (102 MB)


def dump_outputs(session, out_dir: str) -> None:
    """Write what ``session.step()`` hands back to a caller, as float32 ``out_dir/<name>.npy``:

    * ``loss``: the last step's loss (0-d);
    * ``weights``: the updated fp32 master weights, every parameter flattened in ``model.parameters()`` order; above
      ``DUMP_WEIGHT_SAMPLES`` elements, the elements at a fixed sorted sample of indices (numpy seed 0);
    * ``bn_stats``: every floating-point buffer (BatchNorm running means / variances) flattened in ``model.buffers()``
      order."""
    import numpy as np
    import torch

    session.sync()
    w = torch.cat([p.detach().reshape(-1).float() for p in session.model.parameters()])
    if w.numel() > DUMP_WEIGHT_SAMPLES:
        idx = np.sort(np.random.default_rng(0).choice(w.numel(), DUMP_WEIGHT_SAMPLES, replace=False))
        w = w[torch.from_numpy(idx).to(w.device)]
    bufs = [b.detach().reshape(-1).float() for b in session.model.buffers() if b.is_floating_point()]
    out = {"loss": session.last_loss.detach().float().reshape(()), "weights": w,
           "bn_stats": torch.cat(bufs) if bufs else torch.zeros(0)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------
# clock sampling during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        """``gpu_index`` is the CUDA ordinal; nvidia-smi wants the PHYSICAL GPU, which differs under CUDA_VISIBLE_DEVICES:
        address it by UUID."""
        self.gpu, self.proc, self.path = str(gpu_index), None, f"/tmp/ddl_clocks_{os.getpid()}.csv"
        try:
            import torch

            uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            probe = subprocess.run(["nvidia-smi", "-i", uuid, "--query-gpu=index", "--format=csv,noheader"],
                                   capture_output=True, text=True, timeout=20)
            if probe.returncode == 0 and probe.stdout.strip().isdigit():
                self.gpu = uuid                      # else: keep the ordinal (right whenever no device remapping is active)
        except Exception:
            pass
        self.t0 = None

    def mark(self):
        """Start of the timed region: only samples taken from here on are reported.  The sampler itself is started
        before the warm-up so that nvidia-smi's start-up (NVML attach takes driver locks for ~100 ms and was seen to
        stall kernel launches) falls outside the timed steps."""
        self.t0 = time.time()

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", self.gpu], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        rows = []
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    ts = time.mktime(time.strptime(c[0].split(".")[0], "%Y/%m/%d %H:%M:%S")) + float("0." + c[0].split(".")[1])
                except (ValueError, IndexError):
                    ts = None
                rows.append((ts, c))
            os.unlink(self.path)
        except OSError:
            pass
        inside = [c for ts, c in rows if self.t0 is None or ts is None or ts >= self.t0 - 0.2]
        for c in (inside or [c for _, c in rows]):
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch

    from distributeddeeplearning_b200 import _ext
    from distributeddeeplearning_b200.ops import native
    from distributeddeeplearning_b200.parallel import dist
    from distributeddeeplearning_b200.workloads.benchmark import BenchmarkSession

    dist.init()
    rank, world = dist.rank(), dist.size()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (use workloads.benchmark --no-cuda for the CPU plumbing mode)")
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()               # early: nvidia-smi's start-up must not overlap the timed steps (see mark())
    # ---- multi-GPU correctness, visible to whoever reads the JSON line (N>1, before anything is timed) ------------
    # check_engine: per-rank DIFFERENT gradients through the fused allreduce+SGD kernels (NVLS and P2P transports, fp32
    # and bf16 wire, with and without artificial block skew) against the same maths in torch, replicas bit-identical.
    # step_equivalence: a real ResNet-50 step (per-rank different batches): the engine's new weights == w - lr * mean_r(g_r)
    # with the per-rank gradients gathered independently over NCCL; plus the run-to-run noise floor of a single-rank step.
    engine_check, equivalence = None, None
    if world > 1 and not a.no_selfcheck:
        from distributeddeeplearning_b200.parallel import Compression, selfcheck

        oks, names = [], []
        ok, had_mc, name = selfcheck.check_engine(None, Compression.none)
        oks.append(ok); names.append(name)
        for use_mc, wire, skew in ((None, Compression.bf16, 0), (None, Compression.none, 30000),
                                   (None, Compression.bf16, 30000)) + (
                                   ((False, Compression.none, 0), (False, Compression.bf16, 30000)) if had_mc else ()):
            ok, _, name = selfcheck.check_engine(use_mc, wire, skew_ns=skew)
            oks.append(ok); names.append(name)
        engine_check = {"status": "ok" if all(oks) else "FAIL", "variants": len(oks),
                        "failed": [n for n, o in zip(names, oks) if not o]}
        equivalence = selfcheck.step_equivalence("resnet50", 32)
        torch.cuda.empty_cache()
    same_data = os.environ.get("DDL_BENCH_SAME_DATA", "0") == "1"      # experiment hook: every rank trains on rank 0's batch
    session = BenchmarkSession(a.model, a.batch_size, True, a.fp16_allreduce, data_seed_offset=0 if same_data else rank)
    B, dev = a.batch_size, session.device
    graphed = session.enable_graph() if a.cuda_graph == "on" else False

    def region(step_fn, steps, warmup, tail=None, on_start=None):
        for _ in range(warmup):
            step_fn()
        if tail is not None:
            tail()
        dist.barrier()
        torch.cuda.synchronize()
        if on_start is not None:
            on_start()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = _ext.launch_count()
        start.record()
        for _ in range(steps):
            step_fn()
        if tail is not None:
            tail()                     # host has read the result of the last timed step before the clock stops
        stop.record()
        torch.cuda.synchronize()
        dist.barrier()
        ms = dist.allreduce_scalar(start.elapsed_time(stop), op="max")
        return ms, _ext.launch_count() - launches0

    # ---- device-timed headline ------------------------------------------------------------------
    ms, launches = region(session.step, a.steps, a.warmup, on_start=sampler.mark)
    clocks = sampler.stop() if rank == 0 else {}
    loss = float(session.last_loss)
    value = world * B * a.steps / (ms / 1e3)
    if a.dump_outputs:
        if rank == 0:
            dump_outputs(session, a.dump_outputs)
        dist.barrier()                 # the other ranks enter the e2e region's collectives only once rank 0 is done

    # ---- end to end: per-step H2D of the inputs from pinned memory + D2H of the loss --------------
    e2e = None
    if not a.no_e2e:
        size = 224 if not a.model.startswith("inception") else 299
        pool = 4
        g = torch.Generator().manual_seed(1234 + rank)
        host_x = [torch.randint(0, 256, (B, size, size, 3), dtype=torch.uint8, generator=g).pin_memory() for _ in range(pool)]
        host_y = [torch.randint(0, 1000, (B,), dtype=torch.int64, generator=g).pin_memory() for _ in range(pool)]
        mean = torch.tensor([0.485, 0.456, 0.406], device=dev)
        std = torch.tensor([0.229, 0.224, 0.225], device=dev)
        copy_stream = torch.cuda.Stream()
        host_loss = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        state = {"i": 0, "next": None, "losses": [], "pending": None}

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                xd = host_x[i % pool].to(dev, non_blocking=True)
                yd = host_y[i % pool].to(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return xd, yd, ev

        def e2e_step():
            i = state["i"]
            if state["next"] is None:
                state["next"] = prefetch(i)
            xd, yd, ev = state["next"]
            torch.cuda.current_stream().wait_event(ev)
            state["next"] = prefetch(i + 1)            # overlaps this step's compute
            x = native.u8_nhwc_to_nhwc4(xd, mean, std)
            xd.record_stream(torch.cuda.current_stream())
            yd.record_stream(torch.cuda.current_stream())
            l = session.step(x, yd)
            # D2H read of EVERY step's loss: the copy is enqueued now, the host consumes it one step later so the
            # CPU keeps launching step i+1 while step i drains (the last one is consumed by flush_e2e below)
            buf = host_loss[i & 1]
            buf.copy_(l.reshape(1), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            if state["pending"] is not None:
                pev, pbuf = state["pending"]
                pev.synchronize()
                state["losses"].append(float(pbuf[0]))
            state["pending"] = (ev, buf)
            state["i"] = i + 1

        def flush_e2e():
            if state["pending"] is not None:
                pev, pbuf = state["pending"]
                pev.synchronize()
                state["losses"].append(float(pbuf[0]))
                state["pending"] = None

        ms_e, _ = region(e2e_step, a.steps, max(3, a.warmup // 2), tail=flush_e2e)
        e2e = {"value": world * B * a.steps / (ms_e / 1e3), "unit": "images/sec",
               "h2d_bytes_per_step": world * (B * size * size * 3 + B * 8), "d2h_bytes_per_step": world * 4,
               "ms_per_step": ms_e / a.steps}
    if hasattr(session.optimizer, "check_errors"):
        session.optimizer.check_errors()
    checksum = None
    if world > 1:
        from distributeddeeplearning_b200.parallel import selfcheck

        checksum = selfcheck.replica_checksum(session.optimizer)      # after ALL steps: replicas still bit-identical?

    from distributeddeeplearning_b200.ops import fp8 as _fp8

    dtype = "bf16"
    if _fp8.enabled():          # DDL_PRECISION=fp8 experiment runs (the headline stays bf16)
        dtype = "fp8 operands (e4m3/e5m2%s) for forward/dgrad convs with K >= %d, bf16 elsewhere" % (
            ", MX block scales on 1x1 forward" if _fp8.MX else "", _fp8.MIN_K)
    if rank == 0:
        base = None
        try:
            with open(os.path.join(HERE, "BASELINE.json")) as f:
                pub = json.load(f).get("published", {})
            base = pub.get("value") if isinstance(pub, dict) else None
        except Exception:
            pass
        out = {"metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": a.steps,
               "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": (value / base) if base else None, "dtype": dtype, "data": "synthetic",
               "impl": "ours", "final_loss": loss,
               "config": {"model": a.model, "global_batch": world * B, "per_gpu_batch": B, "image": "224x224x3",
                          "seq_len": None, "parallelism": f"dp{world}", "optimizer": "sgd lr=0.01 (fused allreduce+update)",
                          "weights": "random-init, fp32 master + bf16 compute", "l2": "working_set_exceeds_l2",
                          "cuda_graph": bool(graphed),
                          "engine": session.optimizer.describe() if hasattr(session.optimizer, "describe") else "generic"},
               "clocks": clocks, "e2e": e2e, "gpu_launches": launches}
        out["config"]["data_seed"] = ("identical on all ranks (DDL_BENCH_SAME_DATA=1)" if same_data else
                                      "per-rank (seed + rank): ranks train on different batches")
        if world > 1:
            out["engine_check"] = engine_check["status"] if engine_check else "skipped"
            out["engine_check_detail"] = engine_check
            out["step_equivalence"] = equivalence
            out["weight_checksum"] = checksum
        print(json.dumps(out), flush=True)
    dist.shutdown()


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own script, unmodified, through its own CLI
# ------------------------------------------------------------------------------------------------
def run_reference(a):
    def unavailable(why):
        print(f"bench.py --impl reference: {why}", file=sys.stderr, flush=True)
        return 1

    if not os.path.isfile(REF_SCRIPT):
        return unavailable(f"{REF_SCRIPT} is missing; build() stages it from an upstream checkout (oracle/reference.py)")
    try:
        import torch
        import torchvision  # noqa: F401
    except Exception as e:  # pragma: no cover
        return unavailable(f"torch/torchvision import failed: {e}")
    if not torch.cuda.is_available():
        return unavailable("no CUDA device")
    sys.path.insert(0, os.path.join(HERE, "baseline", "hvd_shim"))
    import runpy

    import horovod.torch as hvd

    hvd.init()
    rank, world = hvd.rank(), hvd.size()
    argv = [REF_SCRIPT, "--model", a.model, "--batch-size", str(a.batch_size), "--num-warmup-batches", str(a.warmup),
            "--num-batches-per-iter", str(a.steps), "--num-iters", "1"]
    if a.fp16_allreduce:
        argv.append("--fp16-allreduce")
    old_argv, sys.argv = sys.argv, argv
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
    import contextlib
    import io

    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            runpy.run_path(REF_SCRIPT, run_name="__main__")      # the reference's own code path, start to finish
    finally:
        sys.argv = old_argv
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else {}
    ev = hvd.STEP_EVENTS
    if len(ev) < a.warmup + a.steps:
        return unavailable(f"reference ran {len(ev)} steps, expected {a.warmup + a.steps}")
    ms = ev[a.warmup - 1].elapsed_time(ev[a.warmup + a.steps - 1])      # the K steps after the last warm-up step
    steps = a.steps
    t = torch.tensor([ms], device="cuda")
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms = float(t.item())
    if rank == 0:
        value = world * a.batch_size * steps / (ms / 1e3)
        # The script's OWN end-to-end number: it host-times `timeit(benchmark_step)` through its public CLI and prints
        # "Total img/sec on N GPU(s): X" (pytorch_synthetic_benchmark.py:112-126).  Its stock path keeps ONE fixed batch
        # resident on the device (:81-84), so no input bytes cross PCIe per step and the loss is never read back.
        import re

        e2e = None
        m = re.search(r"Total img/sec on \d+ \S+: ([0-9.]+)", buf.getvalue())
        if m:
            e2e = {"value": float(m.group(1)), "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "how": "the reference script's own host-timed 'Total img/sec' line (its public CLI, stock data path: "
                          "one fixed device-resident batch, no per-step copies)"}
        print(json.dumps({"e2e": e2e, "metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": a.steps,
                          "warmup": a.warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "fp32 (cuDNN TF32 convs: torch default)", "data": "synthetic",
                          "impl": "reference",
                          "config": {"model": a.model, "global_batch": world * a.batch_size, "parallelism": f"dp{world}",
                                     "script": "PyTorch_benchmark/src/pytorch_synthetic_benchmark.py (unmodified)",
                                     "stack": f"torch {torch.__version__} + torchvision + cuDNN + NCCL via horovod shim",
                                     "stdout_tail": buf.getvalue().strip().splitlines()[-3:]},
                          "clocks": clocks}), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return 0


def main():
    a = parse()
    launched = "RANK" in os.environ and "WORLD_SIZE" in os.environ
    if a.gpus > 1 and not launched:
        # convenience: re-launch ourselves on N ranks with the repo's own launcher
        from distributeddeeplearning_b200.cli.launcher import free_port

        port = free_port()
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__), *sys.argv[1:]]
        return subprocess.call(cmd)
    if a.impl == "reference":
        return run_reference(a)
    run_ours(a)
    return 0


if __name__ == "__main__":
    sys.exit(main())
