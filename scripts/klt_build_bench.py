"""Go / no-go microbenchmark of the two matrix builds of klt_quad_kernel (scripts/klt_build_bench.cu): writes staged tiles
(random, extreme and cut from two consecutive C3 synthetic 4K frames) to a temporary directory, builds the .cu there for
sm_100a and runs it.  Prints the card, its power limit and SM clock, and the .cu's JSON line (per-round device time of
each build, their ratio, mismatched doubles).  Exit status 1 when any of the 50 doubles of any feature differs."""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
from sfmgpu import synth  # noqa: E402

N_EACH = 32 * 148 * 14  # one resident wave of the Gram build per tile family


def tile(t1, t0):
    """448 bytes as staged: 14 rows of 16 bytes per image (I1 first), bytes 14 and 15 zero."""
    out = np.zeros((2, 14, 16), np.uint8)
    out[0, :, :14], out[1, :, :14] = t1, t0
    return out


def tiles():
    rng = np.random.default_rng(2026)
    out = [tile(rng.integers(0, 256, (14, 14)), rng.integers(0, 256, (14, 14))) for _ in range(N_EACH)]
    cb = (np.indices((14, 14)).sum(0) % 2 * 255).astype(np.uint8)
    full, zero = np.full((14, 14), 255, np.uint8), np.zeros((14, 14), np.uint8)
    ext = [(full, full), (zero, zero), (full, zero), (zero, full), (cb, cb), (cb, 255 - cb), (255 - cb, cb), (cb, full), (zero, cb)]
    out += [tile(*ext[i % len(ext)]) for i in range(N_EACH)]
    f0, f1 = synth.frame(20261018, 0, 3840, 2160), synth.frame(20261018, 1, 3840, 2160)
    ys, xs = rng.integers(0, 2160 - 14, N_EACH), rng.integers(0, 3840 - 14, N_EACH)
    out += [tile(f1[y:y + 14, x:x + 14], f0[y:y + 14, x:x + 14]) for y, x in zip(ys, xs)]
    return np.stack(out)


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        exe, data = os.path.join(tmp, "klt_build_bench"), os.path.join(tmp, "tiles.bin")
        tiles().tofile(data)
        subprocess.run(["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-fmad=false",
                        "--expt-relaxed-constexpr", "-o", exe, os.path.join(ROOT, "scripts", "klt_build_bench.cu")], check=True)
        return subprocess.run([exe, data, str(reps)]).returncode


if __name__ == "__main__":
    sys.exit(main())
