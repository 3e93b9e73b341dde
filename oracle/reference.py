"""Stage the upstream project's synthetic benchmark for ``bench.py --impl reference`` into ``oracle/_ref/`` (git-ignored).

The upstream project (Microsoft's DistributedDeepLearning cookiecutter template) is not pip-installable and pins a
runtime (horovod 0.15.2, torch 1.0.0, CUDA 9) with no sm_100 build, so the reference arm runs its
``PyTorch_benchmark/src/pytorch_synthetic_benchmark.py`` byte for byte, unmodified, against ``baseline/hvd_shim``.
``build()`` calls ``stage()``.  The upstream checkout is found at ``$DDL_REFERENCE_ROOT``, else in a directory named
``reference`` next to this repository.  Without one, ``stage()`` keeps what ``oracle/_ref/`` already holds, and the
reference arm exits with an error if the script is not there.
"""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
SCRIPT = "pytorch_synthetic_benchmark.py"
UPSTREAM_SCRIPT = os.path.join("{{cookiecutter.project_name}}", "PyTorch_benchmark", "src", SCRIPT)


def upstream_root() -> str:
    return os.environ.get("DDL_REFERENCE_ROOT") or os.path.join(os.path.dirname(ROOT), "reference")


def stage(src_root: str = None, dst: str = DST) -> str:
    """Copy the upstream benchmark script into ``dst``; returns a one-line account of what was done."""
    root = src_root or upstream_root()
    src = os.path.join(root, UPSTREAM_SCRIPT)
    out = os.path.join(dst, SCRIPT)
    if not os.path.isfile(src):
        return f"reference benchmark: no upstream checkout at {root}; " + (
            f"keeping {out}" if os.path.isfile(out) else "bench.py --impl reference is unavailable")
    os.makedirs(dst, exist_ok=True)
    shutil.copyfile(src, out + ".tmp")
    os.replace(out + ".tmp", out)
    return f"reference benchmark: staged {out}"


if __name__ == "__main__":
    print(stage(sys.argv[1] if len(sys.argv) > 1 else None))
