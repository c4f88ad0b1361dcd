"""Calibration of the trajectory checks of tests/test_gpu_zz_trajectory.py on the CPU.

The GPU test compares every kernel family's per-iteration trace and truncated solves with oracle/kernel_model.py at
fixed tolerances. Here the oracle (oracle/pdipm_oracle.py: the reference's LU arithmetic, an independent implementation)
is put through the same comparison helpers at every shape of the family table: it meets those tolerances, so they are
not tighter than two correct fp64 implementations agree. The exit-rule replay helper is checked against the model's own
exit decisions, and the family table against the plans the library chooses.
"""
import os

import numpy as np
import pytest

from oracle import pdipm_oracle as orc
from tests import trajectory_jobs as tj


def _oracle_traces(tr, B):
    """The oracle's per-QP trace (solved one QP at a time) as a list of (iterations, 4) arrays."""
    out = []
    for row in tr:
        if row["it"] == 0:
            out.append([])
        out[-1].append((row["pri"][0], row["dual"][0], row["mu"][0], row["resids"][0]))
    assert len(out) == B
    return [np.array(t) for t in out]


def _pad(traces, n):
    arr = np.full((len(traces), n, 4), np.nan)
    for i, t in enumerate(traces):
        arr[i, :len(t)] = t[:, :4]
    return arr


@pytest.mark.parametrize("shape", tj.ALL_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_oracle_meets_the_trajectory_tolerances(shape):
    """(T) and (K) with the oracle standing in for a kernel, under the reference's literal exit rules on both sides.
    Without equality constraints the two agree within a few percent of the tolerances. With them the oracle forms
    A Q^-1 A^T through LU (cond(Q) reaches 1e7..1e8 at these shapes) and its primal residual and nu carry that error:
    up to 40x the trace tolerance and 5x the nu tolerance, so those shapes are held to 50x. The kernels implement the
    model's whitened Cholesky form and are held to 1x everywhere."""
    loose = 1.0 if shape[3] == 0 else 50.0
    pr = tj.family_problem(shape)
    B = shape[0]
    tr = []
    ref = orc.qp_solve(*(pr[k] for k in tj.KEYS), pr["dl"], per_qp=True, trace=tr)
    model = tj.model_solve(pr, stall_tol=np.inf, tie=1.0)
    assert all(t[3, 3] > 1e-6 for t in model["trace"])          # well posed: still far from converged at iteration 3
    traces = _oracle_traces(tr, B)
    # (iteration counts are not compared: under the literal rules the exit depends on where each implementation's
    # residual lands at the rounding floor, eps = 1e-12 or three non-improving iterations)
    worst = tj.trace_errors(_pad(traces, 20), ref["info"]["iters"], model["trace"], iters_slack=None)
    assert worst <= loose, worst
    for mi in tj.TRUNCATED:
        o = orc.qp_solve(*(pr[k] for k in tj.KEYS), pr["dl"], per_qp=True, maxIter=mi)
        got = dict(zhat=o["zhat"], lam=o["lam"], slacks=o["slacks"], nus=o["nus"], grads=o["grads"],
                   best_resid=o["info"]["best_resids"])
        m = tj.model_solve(pr, trace=False, stall_tol=np.inf, tie=1.0, maxIter=mi)
        assert (o["info"]["iters"] == mi).all() and (m["iters"] == mi).all()
        r = tj.truncated_errors(got, m)
        assert max(r.values()) <= loose, (mi, r)


def test_exit_replay_reproduces_the_model():
    """replay_exit on the model's own trace gives the model's iteration count, returned iterate and reported residual
    (the tied, later iterate's residual, not the running minimum) for every option combination of the exit grid."""
    tied = 0
    for shape in [(6, 20, 15, 5), (8, 50, 50, 10)]:
        pr = tj.family_problem(shape)
        for eps, nil, mi, tie in tj.X_GRID:
            m = tj.model_solve(pr, dl=False, eps=eps, notImprovedLim=nil, maxIter=mi, tie=tie)
            for i, t in enumerate(m["trace"]):
                rows = _pad([t], mi)[0]
                n, ret = tj.replay_exit(rows, eps, nil, mi, tie)
                assert (n, ret) == (m["iters"][i], m["best_iter"][i]), (shape, eps, nil, mi, tie, i)
                assert int(t[-1, 4]) == ret
                assert m["best_resids"][i] == t[ret, 3]
                tied += int(t[ret, 3] > t[:n, 3].min())
    assert tied > 0          # the grid reaches the BEST_TIE rule


def test_replay_handles_each_exit():
    """Hand-made traces: improvement, tie, stall (only below STALL_TOL), eps, mu > 1e32, NaN and maxIter."""
    def rows(res, mu=None):
        mu = [1.0] * len(res) if mu is None else mu
        return np.array([[0.0, 0.0, m, r] for r, m in zip(res, mu)])
    # stall ignored above STALL_TOL: runs to maxIter; the tie keeps the later iterate
    assert tj.replay_exit(rows([1.0, 2.0, 3.0, 1.2, 5.0]), 1e-12, 1, 5, 1.5) == (5, 3)
    assert tj.replay_exit(rows([1.0, 2.0, 3.0, 1.2, 5.0]), 1e-12, 1, 5, 1.0) == (5, 0)
    # stall below STALL_TOL after notImprovedLim non-improving iterations
    assert tj.replay_exit(rows([1e-5, 1e-7, 2e-7, 3e-7, 4e-7, 1e-9]), 1e-12, 3, 6, 1.0) == (5, 1)
    assert tj.replay_exit(rows([1e-5, 1e-7, 1.2e-7, 3e-7, 4e-7, 1e-9]), 1e-12, 3, 6, 1.5) == (5, 2)
    # eps, mu > 1e32, NaN
    assert tj.replay_exit(rows([1.0, 1e-3, 1e-7]), 1e-6, 3, 20, 1.5) == (3, 2)
    assert tj.replay_exit(rows([1.0, 2.0, 3.0], mu=[1.0, 1e33, 1.0]), 1e-12, 3, 20, 1.5) == (2, 0)
    assert tj.replay_exit(rows([1.0, 0.5, np.nan, 0.1]), 1e-12, 3, 20, 1.5) == (3, 1)


def test_options_and_family_table_match_the_library():
    """The job tables name the plans the library chooses (plan_init is host code): every family's shape under its
    environment and mode selects the kernels the GPU test asserts on."""
    from qpth_b200 import _lib, qp as qpmod
    assert (tj.STALL_TOL, tj.BEST_TIE) == (qpmod.STALL_TOL, qpmod.BEST_TIE)
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libqpth_b200.so not built")

    def plan(env, shape, two):
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            return _lib.plan_for(*shape[1:], two=two)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    for fam, (env, mode, shapes, want) in tj.FAMILIES.items():
        for shape in shapes:
            p = plan(env, shape, mode == "throughput")
            assert {k: getattr(p, k) for k in want} == want, (fam, shape)
    for name, (env, shape, want) in tj.SPD_CASES.items():
        p = plan(env, shape, False)
        assert {k: getattr(p, k) for k in want} == want, name


@pytest.mark.parametrize("pattern", sorted(tj.LAYOUTS))
def test_layout_problems_are_the_expanded_problem(pattern):
    """The shared-input problem and its expansion are the same QPs, each strictly feasible (the model converges)."""
    shared, full = tj.layout_problem(pattern, 5, 12, 9, 3, seed=1)
    dims = dict(Q=3, p=2, G=3, h=2, A=3, b=2)
    for k in tj.KEYS:
        unb = shared[k].ndim == dims[k] - 1
        assert unb == (k in tj.LAYOUTS[pattern]), k
        assert full[k].shape[0] == 5 and np.array_equal(full[k][3], shared[k] if unb else shared[k][3])
    m = tj.model_solve(full, trace=False, dl=False)
    assert m["best_resids"].max() < 1e-8
