"""Golden data for the CPU tests of the host-side helpers, from the REAL reference: its `kkt_resid_reg`
(batch.py:228-241) on the seeded problem of tests/test_kkt_cpu.py (inputs + outputs -> tests/golden/kkt_resid_reg.npz)
and what its qpth/util.py helpers return on the inputs of oracle.cases.util_results (-> tests/golden/util_ref.json).
TEST INFRASTRUCTURE ONLY; needs a reference checkout (QPTH_REFERENCE, see oracle/ref_runner.py).

  python oracle/gen_golden_host.py
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_runner  # noqa: E402
from oracle.cases import util_results  # noqa: E402
from tests.test_kkt_cpu import _problem  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def main():
    _, rb = ref_runner.load()
    from qpth import util as R
    p, eps = _problem(seed=1), 1e-7
    res = rb.kkt_resid_reg(p["Q"], torch.diag_embed(p["d"]), p["G"], p["A"], eps, p["dx"], p["ds"], p["dz"], p["dy"],
                           p["rx"], p["rs"], p["rz"], p["ry"])
    np.savez_compressed(os.path.join(OUT, "kkt_resid_reg.npz"), eps=np.float64(eps), **{k: v.numpy() for k, v in p.items()},
                        **{k: v.numpy() for k, v in zip(("resx", "ress", "resz", "resy"), res)})
    with open(os.path.join(OUT, "util_ref.json"), "w") as fh:
        json.dump(util_results(R), fh)
        fh.write("\n")
    print("wrote kkt_resid_reg.npz, util_ref.json to", OUT)


if __name__ == "__main__":
    main()
