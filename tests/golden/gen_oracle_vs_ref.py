"""Writes tests/golden/oracle_vs_ref.npz: the outputs of every case of tests/test_oracle_vs_ref.py, so that the module's
comparisons run where the compiled reference is not built.  Records with the compiled reference (oracle/_ref) when it is
built, else with the restatement; the key "recorded_with" says which.  Inputs are reproducible from seeds, so only
outputs are stored (compressed, < 1 MB).   python tests/golden/gen_oracle_vs_ref.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle  # noqa: E402
import test_oracle_vs_ref as t  # noqa: E402


def main():
    chk, kind = oracle.best()
    g = {"recorded_with": np.array(kind)}
    for key, outputs in t.cases(oracle.port()).items():
        out = outputs(chk)
        g[f"{key}#n"] = np.array(len(out))
        for i, a in enumerate(out):
            g[f"{key}#{i}"] = np.asarray(a)
    out = os.path.join(ROOT, "tests", "golden", "oracle_vs_ref.npz")
    np.savez_compressed(out, **g)
    print(f"wrote {out}: {os.path.getsize(out)} bytes, {len(g)} arrays, recorded with the {kind}")


if __name__ == "__main__":
    main()
