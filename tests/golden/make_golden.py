"""Generate the golden fixtures under tests/golden/ from the REFERENCE ITSELF.

Needs the original project's sources, by default its checkout next to this repository:
`python tests/golden/make_golden.py` (`REFERENCE=<their directory>` points elsewhere).
It compiles attention.c and attention-mpi.c unmodified into oracle/_ref (oracle/Makefile),
calls their own attention() on seeded N(0,1) inputs and stores the outputs: the serial program
(`/serial`), the MPI program on one rank (`/mpi`) and on MPI_RANKS ranks through the shim
(`/mpi<MPI_RANKS>`, run by reference_result.c).  The inputs are not stored: they are regenerated
from (shape, seed, gain) by oracle.make_inputs, and a checksum of the inputs guards against RNG drift.
"""
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle import oracle  # noqa: E402

# (name, m, n, dk, dv, seed, score_gain)
CASES = [
    ("c1_like", 64, 96, 64, 64, 11, 1.0),
    ("odd_dims", 33, 13, 80, 48, 12, 1.0),
    ("tiny", 7, 5, 3, 9, 13, 1.0),
    ("d128", 48, 300, 128, 128, 14, 1.0),
    ("one_key", 5, 1, 16, 8, 15, 1.0),
    ("peaky", 40, 257, 64, 64, 16, 8.0),
    ("wide_v", 17, 70, 32, 200, 17, 1.0),
]
MPI_RANKS = 3      # more ranks than keys in `one_key` and `tiny`: empty and ragged shards


def reference_mpi_result(exe, tmp, Q, K, V, ranks):
    data, res = Path(tmp, "case.bin"), Path(tmp, "result.bin")
    oracle.write_data_file(data, Q, K, V, np.zeros((Q.shape[0], V.shape[1])))
    subprocess.run([str(exe), str(data), str(res)], check=True, env={**os.environ, "MPI_SHIM_NP": str(ranks)})
    return np.fromfile(res, dtype=np.float64).reshape(Q.shape[0], V.shape[1])


def main() -> None:
    oracle.build()
    if not (oracle.REF_DIR / "libattention_mpi.so").exists():
        raise SystemExit("the reference was not compiled: set REFERENCE to the directory of the original project's sources")
    subprocess.run(["make", "-s", "-C", str(oracle.HERE), "golden_driver"], check=True)   # the Makefile's compiler
    exe = oracle.REF_DIR / "reference_result"
    out = {}
    meta = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, m, n, dk, dv, seed, gain in CASES:
            Q, K, V = oracle.make_inputs(m, n, dk, dv, seed, gain)
            out[name + "/serial"] = oracle.reference_attention(Q, K, V, "serial")
            out[name + "/mpi"] = oracle.reference_attention(Q, K, V, "mpi")
            out[f"{name}/mpi{MPI_RANKS}"] = reference_mpi_result(exe, tmp, Q, K, V, MPI_RANKS)
            meta[name] = dict(m=m, n=n, dk=dk, dv=dv, seed=seed, gain=gain,
                              checksum=float(Q.sum() + 2 * K.sum() + 3 * V.sum()))
    here = Path(__file__).resolve().parent
    np.savez_compressed(here / "reference_outputs.npz", **out)
    (here / "cases.json").write_text(json.dumps(meta, indent=1))
    print("wrote", here / "reference_outputs.npz", "and cases.json")


if __name__ == "__main__":
    main()
