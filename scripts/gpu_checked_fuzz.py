"""Builds the library with -DHMK_CHECKED (in-kernel bounds assertions, hmk_common.h) next to the normal one and runs the
bulk-kernel and batch-table tests, the randomised differential tier, the boundary tests, the clinkage tests (dense and sparse path) and the nearest-partner tests against it (HMK_LIB selects the library the
host layer loads).  A failing assertion prints `file:line: ... Assertion ... failed` from the device and the call
returns HMK_STATUS_CUDA, so the test fails with the line in the log.  compute-sanitizer is not available on the pool.

usage (on a GPU box): python scripts/gpu_checked_fuzz.py [extra pytest args]     -> gpurun_out/checked_fuzz.log"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hammock_b200 import build as hb_build      # noqa: E402


def main():
    lib = os.path.join(ROOT, "hammock_b200", "libhammock_b200_checked.so")
    hb_build.build(force=True, defines=["HMK_CHECKED"], out=lib)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    env = dict(os.environ, HMK_LIB=lib)
    cmd = [sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "tests/test_bulk_kernels.py", "tests/test_batch_tables.py",
           "tests/test_gpu_fuzz.py",
           "tests/test_gpu_boundary.py", "tests/test_clinkage.py", "tests/test_clinkage_large.py", "tests/test_gpu_parity.py",
           "tests/test_p1_pipeline.py", "tests/test_nearest.py"] + sys.argv[1:]
    with open(os.path.join(ROOT, "gpurun_out", "checked_fuzz.log"), "w") as log:
        log.write("library: " + lib + "\n$ " + " ".join(cmd) + "\n")
        log.flush()
        rc = subprocess.call(cmd, cwd=ROOT, env=env, stdout=log, stderr=subprocess.STDOUT)
        log.write(f"exit code {rc}\n")
    os.remove(lib)
    print(open(os.path.join(ROOT, "gpurun_out", "checked_fuzz.log")).read()[-3000:])
    return rc


if __name__ == "__main__":
    sys.exit(main())
