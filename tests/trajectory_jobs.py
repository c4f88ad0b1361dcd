"""Newton trajectories, truncated solves, exit rules, shared-input layouts and the SPD check of every solve-kernel family.

Final-answer parity cannot see most bugs in a Newton loop: an interior-point method corrects a subtly wrong step and
still converges, only more slowly. So this module pins what the kernels compute ON THE WAY against
`oracle/kernel_model.py` (the numpy model of their arithmetic):
  (T) the per-iteration trace the kernels write (pri, dual, mu, resid) against the model's, iteration by iteration;
  (K) solves truncated at maxIter 1, 2, 4 (the initial point, one predictor-corrector step, ...) and the backward pass
      from the truncated iterate, where d = lambda / s is moderate;
  (X) iteration counts and the returned residual against a replay of the documented exit rule on the kernel's own trace;
  (L) shared-input layouts (one system, only Q shared, ...) against the same problem expanded to a full batch;
  (S) the 'Q is not SPD.' check of each setup kernel.

It holds the job tables, the problem builders and the numpy comparison helpers (used by tests/test_trajectory_cpu.py on
any machine and by tests/test_gpu_zz_trajectory.py), and the GPU side: `python -m tests.trajectory_jobs <out_dir>` runs
every job on cuda:0 in one process and writes <out_dir>/<job>.npz (or <job>.err with the traceback), so that a fault in
a configuration cannot take the rest of the GPU suite with it.
"""
import os
import sys
import traceback

import numpy as np

KEYS = ("Q", "p", "G", "h", "A", "b")
# plan fields recorded for every solve (from st.plan: the plan the solve actually used)
PLAN_FIELDS = ("tiny", "pf", "pf_global", "pf_two", "pf_three", "pf_threads", "fast", "coop", "smem_resident",
               "setup_pf", "setup_fast")

# family -> (environment, qp.MODE, shapes (B, nz, nineq, neq), plan fields the solve must have used)
PF_SHAPES = [(8, 100, 100, 0), (8, 50, 50, 10)]
FAMILIES = {
    "tiny":     ({}, "auto", [(6, 20, 15, 5)], dict(tiny=1)),
    "pf_one":   ({}, "latency", PF_SHAPES, dict(tiny=0, pf=1, pf_global=0, pf_two=0, pf_three=0)),
    "pf_two":   ({"QPB200_MAXQPS": "2"}, "throughput", PF_SHAPES, dict(tiny=0, pf=1, pf_two=1, pf_three=0)),
    "pf_three": ({}, "throughput", PF_SHAPES, dict(tiny=0, pf=1, pf_two=0, pf_three=1)),
    "pf_l2":    ({}, "latency", [(4, 181, 49, 8)], dict(tiny=0, pf=1, pf_global=1, pf_threads=256, pf_two=0, pf_three=0)),
    "pf_512":   ({}, "auto", [(4, 124, 190, 8)], dict(tiny=0, pf=1, pf_threads=512, pf_two=0, pf_three=0)),
    "r1_fast":  ({"QPB200_PF": "0", "QPB200_COOP": "0"}, "auto", [(8, 100, 100, 0)], dict(tiny=0, pf=0, fast=1, coop=0)),
    "r1_coop":  ({"QPB200_PF": "0", "QPB200_COOP": "1"}, "auto", [(8, 100, 100, 0)], dict(tiny=0, pf=0, fast=1, coop=1)),
    "r1_smem":  ({"QPB200_PF": "0"}, "auto", [(6, 20, 120, 0)], dict(tiny=0, pf=0, fast=0, smem_resident=1)),
    "global":   ({}, "auto", [(3, 120, 260, 0)], dict(tiny=0, pf=0, smem_resident=0)),
}


def case_id(family, shape):
    return "%s_%dx%dx%dx%d" % ((family,) + tuple(shape))


CASES = {case_id(f, sh): (f, sh) for f, (_, _, shapes, _) in FAMILIES.items() for sh in shapes}
ALL_SHAPES = sorted({sh for _, (_, _, shapes, _) in FAMILIES.items() for sh in shapes})


def shape_seed(shape):
    return 300 + ALL_SHAPES.index(tuple(shape))


def family_problem(shape):
    """The (fully batched) problem every family runs at `shape`: the same for every family that shares the shape."""
    from qpth_b200.problems import random_qp_batch
    return random_qp_batch(*shape, seed=shape_seed(shape))


# the solver options of qpth_b200.qp (kept in sync by test_trajectory_cpu.py)
STALL_TOL = 1e-6
BEST_TIE = 1.5
TRUNCATED = (1, 2, 4)
# (eps, notImprovedLim, maxIter, BEST_TIE): every value of each option, the defaults first
X_GRID = [(1e-12, 3, 20, 1.5), (1e-12, 1, 20, 1.5), (1e-12, 3, 40, 1.0), (1e-12, 1, 40, 1.0), (1e-12, 3, 3, 1.0),
          (1e-6, 3, 20, 1.5), (1e-6, 1, 40, 1.0), (1e-6, 3, 3, 1.5),
          (0.0, 3, 40, 1.5), (0.0, 1, 40, 1.5), (0.0, 3, 20, 1.0), (0.0, 1, 3, 1.0)]
# shared-input layouts: the inputs passed un-batched
LAYOUTS = {"P1": ("Q", "G", "h", "A"), "P2": ("Q",), "P3": ("G", "h"), "P4": ("p", "h", "b")}
# P1 (one shared system) once more in auto mode with a batch above the SM count: the OptNet training setup
AUTO_SHAPE = (100, 100, 0)
AUTO_EXTRA = 13

# setup kernel -> (environment, shape, plan fields that select it in pre_factor_impl)
SPD_CASES = {
    "k_setup_tiny":   ({}, (5, 20, 15, 5), dict(tiny=1)),
    "k_setup_fast":   ({}, (5, 100, 100, 0), dict(tiny=0, setup_pf=0, setup_fast=1)),
    "k_setup_pf":     ({}, (5, 50, 50, 10), dict(tiny=0, pf=1, setup_pf=1)),
    "k_setup_smem":   ({"QPB200_PF": "0"}, (5, 150, 20, 0), dict(tiny=0, pf=0, setup_fast=0, smem_resident=1)),
    "k_setup_global": ({}, (5, 120, 260, 0), dict(tiny=0, pf=0, setup_fast=0, smem_resident=0)),
}
SPD_BAD_INDEX = (0, 2, 4)


# ---- problems ------------------------------------------------------------------------------------------------------

def layout_problem(pattern, B, nz, nineq, neq, seed):
    """(shared, expanded): `shared` passes the inputs LAYOUTS[pattern] un-batched, `expanded` is the same problem with
    every input batched. Strictly feasible for every QP: h >= G z0_i + s0 and b_i = A_i z0_i."""
    sk = LAYOUTS[pattern]
    rs = np.random.RandomState(seed)

    def spd():
        L = rs.rand(nz, nz)
        return L @ L.T + 1e-3 * np.eye(nz)

    Q = spd() if "Q" in sk else np.stack([spd() for _ in range(B)])
    G = rs.randn(nineq, nz) if "G" in sk else rs.randn(B, nineq, nz)
    A = rs.randn(neq, nz) if "A" in sk else rs.randn(B, neq, nz)
    p = rs.randn(nz) if "p" in sk else rs.randn(B, nz)
    Ab = np.broadcast_to(A, (B, neq, nz))
    z0 = rs.randn(B, nz)
    if "b" in sk:
        b = rs.randn(neq)
        if neq > 0:       # z0_i: a point with A_i z0_i = b
            z0 = np.stack([np.linalg.lstsq(Ab[i], b, rcond=None)[0] for i in range(B)])
    else:
        b = np.einsum("ben,bn->be", Ab, z0)
    gz = np.einsum("bmn,bn->bm", np.broadcast_to(G, (B, nineq, nz)), z0)
    h = gz.max(0) + rs.rand(nineq) if "h" in sk else gz + rs.rand(B, nineq)
    dl = rs.randn(B, nz)
    shared = dict(Q=Q, p=p, G=G, h=h, A=A, b=b, dl=dl)
    dims = dict(Q=3, p=2, G=3, h=2, A=3, b=2)
    expanded = {k: (np.broadcast_to(v[None], (B,) + v.shape).copy() if (k in dims and v.ndim == dims[k] - 1) else v)
                for k, v in shared.items()}
    return shared, expanded


def indefinite_Q(Q):
    """Q with its smallest eigenvalue replaced by -1e-2 ||Q||_2."""
    w, V = np.linalg.eigh(Q)
    w[0] = -1e-2 * w[-1]
    M = (V * w) @ V.T
    return 0.5 * (M + M.T)


def ill_conditioned_Q(n, rs, cond=1e10):
    V, _ = np.linalg.qr(rs.randn(n, n))
    M = (V * np.logspace(0.0, -np.log10(cond), n)) @ V.T
    return 0.5 * (M + M.T)


# ---- the kernel model and numpy comparison helpers ------------------------------------------------------------------

def model_solve(prob, trace=True, dl=True, **opts):
    """oracle/kernel_model.py with the kernels' exit rules (STALL_TOL, BEST_TIE unless given). Returns the stacked
    outputs plus `trace`: a list of (iterations, 5) arrays (pri, dual, mu, resid, returned-iterate index)."""
    from oracle import kernel_model as km
    opts.setdefault("stall_tol", STALL_TOL)
    opts.setdefault("tie", BEST_TIE)
    tr = [] if trace else None
    o = km.qp_solve(*(prob[k] for k in KEYS), dl=prob["dl"] if dl else None, trace=tr, **opts)
    if trace:
        o["trace"] = [np.array(t, dtype=np.float64).reshape(-1, 5) for t in tr]
    if dl:
        g = o["grads"]
        o["grads"] = tuple(g.get(k) for k in ("dQ", "dp", "dG", "dh", "dA", "db"))
    return o


def trace_errors(got, got_iters, model_trace, rtol=1e-8, atol0=1e-12, floor=1e-6, iters_slack=2):
    """(T): ratio |got - model| / (rtol |model| + atol0 resid_0) per QP, over the four trace fields at every iteration
    whose model residual is >= floor. got: (B, >= iterations, 4). Raises AssertionError if the kernel stopped before
    the last such iteration or its iteration count differs from the model's by more than iters_slack (None: not
    checked). Returns the worst ratio."""
    worst = 0.0
    for i, mt in enumerate(model_trace):
        rows = np.nonzero(mt[:, 3] >= floor)[0]
        assert len(rows) > 0, (i, "model residual below the floor at the initial point")
        last = rows.max()
        assert got_iters[i] > last, (i, "kernel stopped at iteration %d before the model's %d" % (got_iters[i], last + 1))
        assert iters_slack is None or abs(int(got_iters[i]) - len(mt)) <= iters_slack, \
            (i, "iterations", int(got_iters[i]), len(mt))
        ref = mt[rows, :4]
        tol = rtol * np.abs(ref) + atol0 * mt[0, 3]
        r = np.abs(np.asarray(got[i])[rows, :4] - ref) / tol
        assert np.all(np.isfinite(r)), (i, "non-finite trace entry")
        worst = max(worst, float(r.max()))
    return worst


def truncated_errors(got, ref, ztol=1e-8, gtol=1e-7):
    """(K): per-quantity worst ratio error / tolerance of a truncated solve against the model's (rel_rows per QP;
    gradients with the denominator floored at 1e-4 of the batch maximum). got / ref: dicts with zhat, lam, slacks,
    nus, best_resid(s), grads (6-tuple)."""
    from tests.parity import rel_rows
    out = {}
    for k in ("zhat", "lam", "slacks", "nus"):
        if ref.get(k) is None:
            assert got.get(k) is None, k
            continue
        out[k] = float(rel_rows(got[k], ref[k]).max()) / ztol
    gb = np.asarray(got["best_resid"]); rb = np.asarray(ref["best_resids"] if "best_resids" in ref else ref["best_resid"])
    out["best_resid"] = float((np.abs(gb - rb) / np.abs(rb)).max()) / ztol
    for name, g, r in zip(("dQ", "dp", "dG", "dh", "dA", "db"), got["grads"], ref["grads"]):
        if r is None:
            assert g is None, name
            continue
        out[name] = float(rel_rows(g, r, floor=1e-4).max()) / gtol
    return out


def replay_exit(trace, eps, notImprovedLim, maxIter, tie, stall_tol=STALL_TOL):
    """The kernels' documented exit rule (DESIGN.md section 2) replayed on one QP's trace rows (pri, dual, mu, resid):
    strict improvement resets the not-improved count; an iterate within `tie` of the best is returned instead of it;
    stop after notImprovedLim non-improving iterations once best < stall_tol, when best < eps, when mu > 1e32, at a NaN
    or infinite residual, or after maxIter iterations. Returns (iterations, index of the returned iterate)."""
    best, n_not, ret = 0.0, 0, 0
    for it in range(maxIter):
        mu, resid = float(trace[it][2]), float(trace[it][3])
        improved = it == 0 or resid < best
        if improved:
            best, n_not = resid, 0
        else:
            n_not += 1
        if improved or resid < tie * best:
            ret = it
        if (n_not == notImprovedLim and best < stall_tol) or best < eps or mu > 1e32:
            return it + 1, ret
        if not np.isfinite(resid):
            return it + 1, ret
    return maxIter, ret


# ---- the GPU side ---------------------------------------------------------------------------------------------------

DEV = "cuda:0"


def _solve(prob, eps=1e-12, notImprovedLim=3, maxIter=20, requires=KEYS, backward=True):
    import torch
    from qpth_b200 import QPFunction
    t = {}
    for k in KEYS:
        v = np.asarray(prob[k], dtype=np.float64)
        if v.size == 0:
            t[k] = torch.Tensor().to(DEV).double()
        else:
            t[k] = torch.tensor(v, dtype=torch.float64, device=DEV, requires_grad=(k in requires))
    f = QPFunction(eps=eps, verbose=-1, notImprovedLim=notImprovedLim, maxIter=maxIter)
    z = f(*(t[k] for k in KEYS))
    st = f.last_solve()
    out = dict(zhat=z.detach().cpu().numpy(), lam=st.lam.cpu().numpy(), slacks=st.slacks.cpu().numpy(),
               nus=None if st.nus is None else st.nus.cpu().numpy(), iters=st.iters.cpu().numpy(),
               best_resid=st.best_resid.cpu().numpy(), trace=None if st.trace is None else st.trace.cpu().numpy(),
               plan=np.array([getattr(st.plan, fld) for fld in PLAN_FIELDS], dtype=np.int64))
    if backward:
        B = out["zhat"].shape[0]
        z.backward(torch.tensor(np.asarray(prob["dl"]).reshape(B, -1), dtype=torch.float64, device=DEV))
        out["grads"] = tuple(None if (not t[k].requires_grad or t[k].grad is None) else t[k].grad.cpu().numpy()
                             for k in KEYS)
    return out


def _put(rec, prefix, out):
    for k, v in out.items():
        if k == "grads":
            for i, g in enumerate(v):
                if g is not None:
                    rec["%s_g%d" % (prefix, i)] = np.asarray(g)
        elif v is not None:
            rec["%s_%s" % (prefix, k)] = np.asarray(v)


def get_run(d, prefix):
    """Inverse of _put on a loaded .npz: the dict of one solve (grads a 6-tuple with None where absent)."""
    out = {}
    for k in ("zhat", "lam", "slacks", "nus", "iters", "best_resid", "trace", "plan", "error"):
        key = "%s_%s" % (prefix, k)
        out[k] = d[key] if key in d else None
    g = tuple(d["%s_g%d" % (prefix, i)] if ("%s_g%d" % (prefix, i)) in d else None for i in range(6))
    out["grads"] = g if any(x is not None for x in g) else None
    return out


def plan_dict(arr):
    return dict(zip(PLAN_FIELDS, (int(x) for x in arr)))


def _job_T(prob):
    from qpth_b200 import qp as qpmod
    qpmod.TRACE = True
    try:
        rec = {}
        _put(rec, "t", _solve(prob, backward=False))
        return rec
    finally:
        qpmod.TRACE = False


def _job_K(prob):
    rec = {}
    for mi in TRUNCATED:
        _put(rec, "k%d" % mi, _solve(prob, maxIter=mi))
    return rec


def _job_X(prob):
    from qpth_b200 import qp as qpmod
    rec = {}
    qpmod.TRACE = True
    try:
        for ci, (eps, nil, mi, tie) in enumerate(X_GRID):
            qpmod.BEST_TIE = tie
            _put(rec, "x%d" % ci, _solve(prob, eps=eps, notImprovedLim=nil, maxIter=mi, backward=False))
    finally:
        qpmod.TRACE = False
        qpmod.BEST_TIE = BEST_TIE
    return rec


def _job_L(shape):
    B, nz, nineq, neq = shape
    rec = {}
    for pi, pat in enumerate(sorted(LAYOUTS)):
        shared, expanded = layout_problem(pat, B, nz, nineq, neq, seed=shape_seed(shape) + 50 + pi)
        _put(rec, pat + "s", _solve(shared))
        _put(rec, pat + "e", _solve(expanded))
        if pat == "P1":
            _put(rec, pat + "ph", _solve(shared, requires=("p", "h")))
    return rec


def _job_L_auto():
    import torch
    from qpth_b200 import _lib
    B = _lib.sm_count(torch.device(DEV).index or 0) + AUTO_EXTRA
    shared, expanded = layout_problem("P1", B, *AUTO_SHAPE, seed=401)
    rec = dict(B=np.array(B))
    _put(rec, "P1s", _solve(shared))
    _put(rec, "P1e", _solve(expanded))
    return rec


def _raw_spd_flags(shape, Q):
    """qpb200_pre_factor_kkt alone (no solve) on Q (B, nz, nz); returns the per-system spd flags and the plan used."""
    import ctypes
    import torch
    from qpth_b200 import _lib
    B, nz, nineq, neq = shape
    lib = _lib.load()
    plan = _lib.plan_for(nz, nineq, neq)
    rs = np.random.RandomState(7)
    f64 = dict(dtype=torch.float64, device=DEV)
    tt = lambda a: torch.tensor(a, **f64).contiguous()
    Qd, Gd = tt(Q), tt(rs.randn(B, nineq, nz))
    Ad = tt(rs.randn(B, neq, nz)) if neq > 0 else None
    L = torch.empty(B * plan.L_elems, **f64)
    W = torch.empty(B * plan.W_elems, **f64)
    K = torch.empty(B * plan.K_elems, **f64)
    scr = torch.empty(B * plan.setup_scratch_elems, **f64) if plan.setup_scratch_elems > 0 else None
    spd = torch.full((B,), -1, dtype=torch.int32, device=DEV)
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)
    _lib.check(lib.qpb200_pre_factor_kkt(ctypes.byref(plan), B, P(Qd), nz * nz, P(Gd), nineq * nz, P(Ad), neq * nz,
                                         P(L), P(W), P(K), P(spd), P(scr),
                                         ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return spd.cpu().numpy(), np.array([getattr(plan, fld) for fld in PLAN_FIELDS], dtype=np.int64)


def _raises_not_spd(prob):
    """QPFunction (check_Q_spd on): 1 if it raised 'Q is not SPD.', 0 if it returned; anything else propagates."""
    try:
        _solve(prob, backward=False)
    except RuntimeError as exc:
        if "Q is not SPD." in str(exc):
            return 1
        raise
    return 0


def _job_S(shape):
    from qpth_b200.problems import random_qp_batch
    B, nz, nineq, neq = shape
    base = random_qp_batch(*shape, seed=500 + nz)
    rec = {}
    for idx in SPD_BAD_INDEX:
        pr = dict(base)
        pr["Q"] = base["Q"].copy()
        pr["Q"][idx] = indefinite_Q(base["Q"][idx])
        rec["flags%d" % idx], rec["plan%d" % idx] = _raw_spd_flags(shape, pr["Q"])
        rec["raised%d" % idx] = np.array(_raises_not_spd(pr))
    pr = dict(base)
    pr["Q"] = indefinite_Q(base["Q"][0])                     # the shared (un-batched) Q is the indefinite one
    rec["raised_shared"] = np.array(_raises_not_spd(pr))
    rs = np.random.RandomState(600 + nz)
    Qc = np.stack([ill_conditioned_Q(nz, rs) for _ in range(B)])
    rec["flags_cond"], rec["plan_cond"] = _raw_spd_flags(shape, Qc)
    return rec


def jobs():
    """[(job name, environment, qp.MODE, thunk returning the record to save)] in execution order."""
    out = []
    for cid, (fam, shape) in CASES.items():
        env, mode, _, _ = FAMILIES[fam]
        out.append(("T_" + cid, env, mode, lambda shape=shape: _job_T(family_problem(shape))))
        out.append(("K_" + cid, env, mode, lambda shape=shape: _job_K(family_problem(shape))))
        out.append(("X_" + cid, env, mode, lambda shape=shape: _job_X(family_problem(shape))))
        out.append(("L_" + cid, env, mode, lambda shape=shape: _job_L(shape)))
    out.append(("L_auto", {}, "auto", _job_L_auto))
    for name, (env, shape, _) in SPD_CASES.items():
        out.append(("S_" + name, env, "auto", lambda shape=shape: _job_S(shape)))
    return out


def main(out_dir, only=None):
    from qpth_b200 import qp as qpmod
    for name, env, mode, thunk in jobs():
        if only and not any(s in name for s in only):
            continue
        saved = {k: os.environ.get(k) for k in env}
        try:
            os.environ.update(env)
            qpmod.MODE = mode
            np.savez(os.path.join(out_dir, name + ".npz"), **thunk())
        except BaseException:      # noqa: BLE001 - recorded for the parent, the next job still runs
            with open(os.path.join(out_dir, name + ".err"), "w") as fh:
                fh.write(traceback.format_exc())
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        with open(os.path.join(out_dir, "progress.txt"), "a") as fh:
            fh.write(name + "\n")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2:])
