"""Record tests/golden/parity/*.npz from the reference's own CUDA rasterizer: what the reference-parity tests of
tests/test_gpu_parity.py compare against.

Run on a B200 with the native library and the reference's build (oracle/build_ref.py -> oracle/_ref/) in place:
    python tests/golden/make_golden_parity.py --out <dir> [--sample N]
then copy <dir>/*.npz into tests/golden/parity/.  It runs tests/test_gpu_parity.py with BRS_RECORD_PARITY set, so
that every compared call runs the reference on the same inputs, records the reference's results and compares this
library with them live (parity_lib.Recorded).  Nothing is written unless every test passes.  `--sample N` shortens
every sampled array of the records to its first N elements (parity_lib.sample_index keeps a shortened sample a
valid one), to keep the files small.

`--shorten N FILE...` shortens existing records the same way without a GPU.
"""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def shorten(path: str, n: int) -> None:
    """Keep the first n elements of every sampled array of one record file.  Arrays stored whole are at most
    parity_lib.FULL (256) elements long and so stay as they are (parity_lib needs the native library; this does not)."""
    assert n >= 256, "--sample must be at least parity_lib.FULL (256)"
    with np.load(path) as z:
        data = {k: z[k] for k in z.files}
    for k, v in data.items():
        if v.ndim == 1 and v.dtype == np.float32 and k + ".norm" in data:
            data[k] = v[:n]
    np.savez_compressed(path, **data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="directory the records are written to")
    ap.add_argument("--sample", type=int, default=0, help="shorten sampled arrays to this many elements")
    ap.add_argument("--shorten", type=int, default=0, help="shorten the sampled arrays of FILE... to this many elements")
    ap.add_argument("files", nargs="*")
    a = ap.parse_args()
    if a.shorten:
        for f in a.files:
            shorten(f, a.shorten)
        return 0
    if not a.out:
        ap.error("--out is required")
    with tempfile.TemporaryDirectory() as tmp:
        env = dict(os.environ, BRS_RECORD_PARITY=tmp)
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", os.path.join(ROOT, "tests", "test_gpu_parity.py")],
                           cwd=ROOT, env=env)
        if r.returncode != 0:
            print("not recorded: this library does not pass against the reference", file=sys.stderr)
            return r.returncode
        os.makedirs(a.out, exist_ok=True)
        for f in sorted(os.listdir(tmp)):
            path = os.path.join(a.out, f)
            shutil.move(os.path.join(tmp, f), path)
            if a.sample:
                shorten(path, a.sample)
            print(f, os.path.getsize(path), "bytes", flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
