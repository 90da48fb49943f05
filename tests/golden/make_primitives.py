"""Write tests/golden/primitives_fixture.npz: the outputs of every per-level AMG primitive (spmv, Jacobi sweeps, residual,
stored residual, restriction, prolongation) and of the coarse solve on the bundled fixture, HEM (0) and Beck (1)
hierarchies, from the seeded inputs of oracle_bindings.primitive_outputs.  Each output is stored at a fixed sample of at
most 512 rows ("<coarsening>:<level>/<op>", rows under "...@rows"), which keeps the file far below 1 MB.

    python tests/golden/make_primitives.py --source ref      # the reference's own code (oracle/_ref must be built)
    python tests/golden/make_primitives.py --source oracle   # the C restatement (oracle/sparsh_oracle.c)

The file records its source.  test_primitives_against_live_reference compares the restatement with it on every run.
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle_bindings import CSR, Oracle, OracleAmg, OracleOps, RefAmg, have_ref, primitive_outputs  # noqa: E402

SAMPLE = 512


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--source", choices=["ref", "oracle"], default="ref")
    args = ap.parse_args()
    if args.source == "ref" and not have_ref():
        sys.exit("oracle/_ref/libsparsh_ref.so is missing: build it with `make -C oracle ref`")
    z = np.load(os.path.join(HERE, "fixture_poisson_P1.npz"))
    n = len(z["rowptr"]) - 1
    A = CSR(n, n, z["rowptr"], z["colindex"], z["val"])
    out = {"source": np.array("the reference's own code (oracle/_ref)" if args.source == "ref" else
                              "the C restatement (oracle/sparsh_oracle.c)")}
    for coarsening in (0, 1):
        if args.source == "ref":
            ops = RefAmg(A, coarsening)
            H = ops.hierarchy()
        else:
            H = OracleAmg(A, coarsening).hierarchy()
            ops = OracleOps(Oracle.get(), H)
        for key, v in primitive_outputs(H, ops).items():
            rows = np.sort(np.random.default_rng(0).choice(len(v), min(len(v), SAMPLE), replace=False)).astype(np.int32)
            out[f"{coarsening}:{key}"] = v[rows]
            out[f"{coarsening}:{key}@rows"] = rows
    path = os.path.join(HERE, "primitives_fixture.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, f"({os.path.getsize(path)} bytes, {len(out) // 2} outputs)")


if __name__ == "__main__":
    main()
