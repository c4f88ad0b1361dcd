"""Every solve-kernel family on the way to the answer, not only at it (tests/trajectory_jobs.py has the tables and the
helpers): the per-iteration trace and truncated solves against oracle/kernel_model.py, iteration counts and returned
residuals against a replay of the exit rule on the kernel's own trace, shared-input layouts against the expanded
problem, and the SPD check of each setup kernel.

All GPU work runs in ONE child process with a timeout (python -m tests.trajectory_jobs); this process only compares on
the CPU. Every test asserts the plan fields of the plan the solves actually used (recorded from st.plan by the child).
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pdipm_oracle as orc
from tests import trajectory_jobs as tj
from tests.parity import GTOL, ZTOL, rel_rows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD_TIMEOUT_S = 420


@pytest.fixture(scope="module")
def child_results(tmp_path_factory):
    out_dir = str(tmp_path_factory.mktemp("trajectory"))
    note = ""
    try:
        r = subprocess.run([sys.executable, "-m", "tests.trajectory_jobs", out_dir], cwd=ROOT, timeout=CHILD_TIMEOUT_S,
                           capture_output=True, text=True)
        if r.returncode != 0:
            note = "child exited with %d: %s" % (r.returncode, (r.stderr or "")[-2000:])
    except subprocess.TimeoutExpired:
        note = "child killed after %d s (a job hung)" % CHILD_TIMEOUT_S
    return out_dir, note


def _load(child_results, job):
    out_dir, note = child_results
    path = os.path.join(out_dir, job + ".npz")
    if not os.path.exists(path):
        err = os.path.join(out_dir, job + ".err")
        why = open(err).read()[-3000:] if os.path.exists(err) else ("no result: " + (note or "job never ran"))
        pytest.fail("%s: %s" % (job, why), pytrace=False)
    return dict(np.load(path))


def _report(what, **vals):
    """Append the worst error / tolerance ratios of a check to the JSON-lines file named by QPB200_TRAJECTORY_REPORT
    (if set; best effort)."""
    path = os.environ.get("QPB200_TRAJECTORY_REPORT")
    if not path:
        return
    try:
        with open(path, "a") as fh:
            fh.write(json.dumps(dict(check=what, **{k: float(v) for k, v in vals.items()})) + "\n")
    except OSError:
        pass


def _assert_plan(run, want, what):
    got = tj.plan_dict(run["plan"])
    assert {k: got[k] for k in want} == want, (what, got)


@functools.lru_cache(maxsize=None)
def _model(shape, **opts):
    return tj.model_solve(tj.family_problem(shape), **opts)


@pytest.mark.parametrize("case", sorted(tj.CASES))
def test_trace_matches_kernel_model(case, child_results):
    """(T) qp.TRACE with the default options: pri, dual, mu and resid at every iteration whose model residual is above
    1e-6, within 1e-8 relative + 1e-12 of the initial residual; the iteration count within 2 of the model's."""
    fam, shape = tj.CASES[case]
    run = tj.get_run(_load(child_results, "T_" + case), "t")
    _assert_plan(run, tj.FAMILIES[fam][3], case)
    m = _model(shape, dl=False)
    assert all(t[3, 3] > 1e-6 for t in m["trace"]), "problem converges too fast to pin a trajectory"
    tr, iters = run["trace"], run["iters"]
    assert tr.shape == (shape[0], 20, 4)
    for i in range(shape[0]):                 # written exactly for the iterations run
        assert np.isnan(tr[i, iters[i]:]).all() and np.isfinite(tr[i, :iters[i]]).all(), i
    worst = tj.trace_errors(tr, iters, m["trace"])
    _report("T " + case, worst=worst)
    assert worst <= 1.0, worst


@pytest.mark.parametrize("case", sorted(tj.CASES))
def test_truncated_solves_match_kernel_model(case, child_results):
    """(K) maxIter 1 (the initial point), 2 (one predictor-corrector step) and 4: exactly that many iterations; z, lambda,
    s, nu and the returned residual within 1e-8 of the model's truncated solve; the backward pass from the truncated
    iterate (moderate d = lambda / s) within 1e-7 of the model's."""
    fam, shape = tj.CASES[case]
    d = _load(child_results, "K_" + case)
    worst = {}
    for mi in tj.TRUNCATED:
        run = tj.get_run(d, "k%d" % mi)
        _assert_plan(run, tj.FAMILIES[fam][3], case)
        assert (run["iters"] == mi).all(), (mi, run["iters"])
        r = tj.truncated_errors(run, _model(shape, trace=False, maxIter=mi))
        for k, v in r.items():
            worst[k] = max(worst.get(k, 0.0), v)
    _report("K " + case, **worst)
    assert max(worst.values()) <= 1.0, worst


@pytest.mark.parametrize("case", sorted(tj.CASES))
def test_exit_rule_replay(case, child_results):
    """(X) over the (eps, notImprovedLim, maxIter, BEST_TIE) grid: the iteration count equals the documented rule replayed
    on the kernel's own trace, and the reported residual is that trace's entry for the replayed returned iterate, bit for
    bit. With eps = 1e-6 the exit iteration equals the model's wherever the model's residuals stay 10x clear of eps."""
    fam, shape = tj.CASES[case]
    d = _load(child_results, "X_" + case)
    compared = 0
    for ci, (eps, nil, mi, tie) in enumerate(tj.X_GRID):
        run = tj.get_run(d, "x%d" % ci)
        _assert_plan(run, tj.FAMILIES[fam][3], case)
        assert run["trace"].shape == (shape[0], mi, 4)
        for i in range(shape[0]):
            n, ret = tj.replay_exit(run["trace"][i], eps, nil, mi, tie)
            assert run["iters"][i] == n, (eps, nil, mi, tie, i, run["iters"][i], n)
            assert run["best_resid"][i] == run["trace"][i, ret, 3], (eps, nil, mi, tie, i)
            assert np.isnan(run["trace"][i, n:]).all()
        if eps == 1e-6:
            m = _model(shape, trace=True, dl=False, eps=eps, notImprovedLim=nil, maxIter=mi, tie=tie)
            for i, t in enumerate(m["trace"]):
                r = t[:, 3]
                if np.all((r > 10 * eps) | (r < eps / 10)):
                    compared += 1
                    assert run["iters"][i] == m["iters"][i], (eps, nil, mi, tie, i)
    _report("X " + case, qps_compared_with_model=compared)


@pytest.mark.parametrize("case", sorted(tj.CASES))
def test_shared_input_layouts(case, child_results):
    """(L) P1 (Q, G, h, A shared: one system), P2 (only Q), P3 (G, h), P4 (p, h, b) against the same problem expanded to a
    full batch through the same family: z, lambda, s and batched gradients within 1e-12, batch-mean gradients within
    1e-10 of .mean(0) of the expanded ones, the expanded run against the oracle; P1 with only p and h requiring grad
    gives exactly the all-gradient run's gradients and None for the others."""
    fam, shape = tj.CASES[case]
    d = _load(child_results, "L_" + case)
    B, nz, nineq, neq = shape
    worst = dict(same=0.0, mean=0.0, z_oracle=0.0, g_oracle=0.0)
    for pi, pat in enumerate(sorted(tj.LAYOUTS)):
        shared, full = tj.layout_problem(pat, B, nz, nineq, neq, seed=tj.shape_seed(shape) + 50 + pi)
        s, e = tj.get_run(d, pat + "s"), tj.get_run(d, pat + "e")
        _assert_plan(s, tj.FAMILIES[fam][3], case)
        _assert_plan(e, tj.FAMILIES[fam][3], case)
        _check_layout(pat, s, e, full, worst)
        if pat == "P1":
            ph = tj.get_run(d, pat + "ph")
            _assert_plan(ph, tj.FAMILIES[fam][3], case)
            assert [g is None for g in ph["grads"]] == [True, False, True, False, True, True]
            assert np.array_equal(ph["grads"][1], s["grads"][1]) and np.array_equal(ph["grads"][3], s["grads"][3])
            assert np.array_equal(ph["zhat"], s["zhat"])
    _report("L " + case, **worst)


def _check_layout(pat, s, e, full, worst, n_oracle=16):
    for k in ("zhat", "lam", "slacks", "nus"):
        if e[k] is not None:
            r = rel_rows(s[k], e[k]).max()
            worst["same"] = max(worst["same"], r / 1e-12)
            assert r <= 1e-12, (pat, k, r)
    for j, key in enumerate(tj.KEYS):
        gs, ge = s["grads"][j], e["grads"][j]
        if ge is None:
            assert gs is None, (pat, key)
            continue
        if key in tj.LAYOUTS[pat]:      # un-batched input: its gradient is the batch mean
            ref = ge.mean(0)
            r = np.linalg.norm(gs - ref) / np.linalg.norm(ref)
            worst["mean"] = max(worst["mean"], r / 1e-10)
            assert gs.shape == ref.shape and r <= 1e-10, (pat, key, r)
        else:
            r = rel_rows(gs, ge, floor=1e-4).max()
            worst["same"] = max(worst["same"], r / 1e-12)
            assert r <= 1e-12, (pat, key, r)
    n = min(n_oracle, e["zhat"].shape[0])
    ref = orc.qp_solve(*(full[k][:n] for k in tj.KEYS), full["dl"][:n], per_qp=True)
    rz = rel_rows(e["zhat"][:n], ref["zhat"]).max()
    worst["z_oracle"] = max(worst["z_oracle"], rz / ZTOL)
    assert rz <= ZTOL, (pat, rz)
    for g, r in zip(e["grads"], ref["grads"]):
        if r is None:
            assert g is None
            continue
        rg = rel_rows(g[:n], r, floor=1e-4).max()
        worst["g_oracle"] = max(worst["g_oracle"], rg / GTOL)
        assert rg <= GTOL, (pat, rg)


def test_one_shared_system_in_auto_mode(child_results):
    """(L) the OptNet training setup: one shared system (P1) at C2 size with a batch 13 above the SM count (not a
    multiple of 16: the tail of the batch-mean kernels) in auto mode takes the three-QPs-per-SM kernel and agrees with
    the expanded problem and the oracle."""
    d = _load(child_results, "L_auto")
    B = int(d["B"])
    shared, full = tj.layout_problem("P1", B, *tj.AUTO_SHAPE, seed=401)
    s, e = tj.get_run(d, "P1s"), tj.get_run(d, "P1e")
    for run in (s, e):
        _assert_plan(run, dict(tiny=0, pf=1, pf_three=1), "auto")
    worst = dict(same=0.0, mean=0.0, z_oracle=0.0, g_oracle=0.0)
    _check_layout("P1", s, e, full, worst)
    _report("L auto B=%d" % B, **worst)


@pytest.mark.parametrize("name", sorted(tj.SPD_CASES))
def test_spd_check_per_setup_kernel(name, child_results):
    """(S) each setup kernel flags exactly the indefinite Q of a batch of 5 (index 0, 2 or 4) and QPFunction raises
    'Q is not SPD.', also when the indefinite Q is the shared one; an SPD Q with condition number 1e10 is not flagged."""
    env, shape, want = tj.SPD_CASES[name]
    d = _load(child_results, "S_" + name)
    for idx in tj.SPD_BAD_INDEX:
        assert {k: tj.plan_dict(d["plan%d" % idx])[k] for k in want} == want, name
        expect = np.zeros(shape[0], dtype=np.int32)
        expect[idx] = 1
        assert np.array_equal(d["flags%d" % idx], expect), (idx, d["flags%d" % idx])
        assert int(d["raised%d" % idx]) == 1, idx
    assert int(d["raised_shared"]) == 1
    assert {k: tj.plan_dict(d["plan_cond"])[k] for k in want} == want, name
    assert np.array_equal(d["flags_cond"], np.zeros(shape[0], dtype=np.int32)), d["flags_cond"]
