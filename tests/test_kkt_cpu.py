"""CPU checks of the host-side pieces of qpth_b200/kkt.py and qpth_b200/layers.py (no GPU): the residual of the regularised
KKT system against a densely assembled matrix and against the real reference's outputs (tests/golden/kkt_resid_reg.npz,
oracle/gen_golden_host.py), and the golden files the GPU tests of both modules read."""
import os

import numpy as np
import pytest
import torch


def _problem(B=3, n=7, m=5, e=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    M = r(B, n, n)
    return dict(Q=M @ M.transpose(1, 2), G=r(B, m, n), A=r(B, e, n), d=torch.rand(B, m, generator=g, dtype=torch.float64) + 0.1,
                rx=r(B, n), rs=r(B, m), rz=r(B, m), ry=r(B, e), dx=r(B, n), ds=r(B, m), dz=r(B, m), dy=r(B, e))


def test_kkt_resid_reg_matches_dense_assembly():
    from qpth_b200 import kkt
    p, eps = _problem(), 1e-3
    res = kkt.kkt_resid_reg(p["Q"], p["d"], p["G"], p["A"], eps, p["dx"], p["ds"], p["dz"], p["dy"], p["rx"], p["rs"], p["rz"], p["ry"])
    B, n, m, e = 3, 7, 5, 2
    for i in range(B):
        K = np.zeros((n + 2 * m + e, n + 2 * m + e))
        Q, G, A, d = (p[k][i].numpy() for k in ("Q", "G", "A", "d"))
        K[:n, :n] = Q; K[:n, n + m:n + 2 * m] = G.T; K[:n, n + 2 * m:] = A.T
        K[n:n + m, n:n + m] = np.diag(d); K[n:n + m, n + m:n + 2 * m] = np.eye(m)
        K[n + m:n + 2 * m, :n] = G; K[n + m:n + 2 * m, n:n + m] = np.eye(m); K[n + m:n + 2 * m, n + m:n + 2 * m] = -eps * np.eye(m)
        K[n + 2 * m:, :n] = A; K[n + 2 * m:, n + 2 * m:] = -eps * np.eye(e)
        v = np.concatenate([p[k][i].numpy() for k in ("dx", "ds", "dz", "dy")])
        rhs = np.concatenate([p[k][i].numpy() for k in ("rx", "rs", "rz", "ry")])
        want = K @ v + rhs
        got = np.concatenate([t[i].numpy() for t in res])
        assert np.abs(got - want).max() < 1e-12
    # the diagonal-matrix form of D (the reference's calling convention) gives the same
    res2 = kkt.kkt_resid_reg(p["Q"], torch.diag_embed(p["d"]), p["G"], p["A"], eps, p["dx"], p["ds"], p["dz"], p["dy"],
                             p["rx"], p["rs"], p["rz"], p["ry"])
    assert all(torch.equal(a, b) for a, b in zip(res, res2))


def test_kkt_resid_reg_matches_reference_golden(golden_dir):
    """The reference's kkt_resid_reg (batch.py:228-241) on _problem(seed=1), inputs and outputs stored."""
    from qpth_b200 import kkt
    g = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(golden_dir, "kkt_resid_reg.npz")).items()}
    ours = kkt.kkt_resid_reg(g["Q"], g["d"], g["G"], g["A"], float(g["eps"]), g["dx"], g["ds"], g["dz"], g["dy"],
                             g["rx"], g["rs"], g["rz"], g["ry"])
    for a, k in zip(ours, ("resx", "ress", "resz", "resy")):
        assert float((a - g[k]).abs().max()) < 1e-12


def test_golden_files_of_the_kkt_and_layer_tests_exist(golden_dir):
    for name in ("kkt_small", "kkt_c3", "kkt_ineq_only", "kkt_singular", "layer_small", "layer_cls"):
        z = np.load(os.path.join(golden_dir, name + ".npz"))
        assert all(np.isfinite(z[k]).all() for k in z.files)


def test_kkt_and_layers_refuse_cpu_tensors():
    from qpth_b200 import kkt
    from qpth_b200.layers import OptNetQP
    p = _problem()
    with pytest.raises(AssertionError):
        kkt.factor_solve_kkt(p["Q"], p["d"], p["G"], p["A"], p["rx"], p["rs"], p["rz"], p["ry"])
    with pytest.raises(AssertionError):
        OptNetQP()(torch.eye(4, dtype=torch.float64), torch.ones(3, 4, dtype=torch.float64), torch.zeros(4, dtype=torch.float64),
                   torch.ones(3, dtype=torch.float64), torch.zeros(2, 4, dtype=torch.float64))
