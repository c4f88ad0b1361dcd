"""numpy model of the ARITHMETIC the CUDA kernels use (TEST INFRASTRUCTURE ONLY).

Not the reference's algorithm restated (that is `pdipm_oracle.py`) but the
B200 design's reformulation, kept here so tests can separate "the
reformulation changes the answer" from "the kernel has a bug":

* per-QP semantics: every QP is solved as the reference solves an nBatch=1
  call (exit tests of `batch.py:140` applied to that QP alone);
* whitened variables x~ = L^T x with Q = L L^T (Cholesky instead of the
  reference's pivoted LU): G~ = G L^-T, A~ = A L^-T, p~ = L^-1 p, so that
  Q^-1 disappears from `solve_kkt` (batch.py:349-372) and
  R = G Q^-1 G^T = G~ G~^T (batch.py:396-399);
* the (neq+nineq) block system is eliminated with Cholesky blocks
  L11 = chol(A~ A~^T), L21 = G~ A~^T L11^-T, L22 = chol(R - L21 L21^T + D^-1)
  (the SPD counterpart of the block LU in batch.py:402-424,435-470).
The dual residual norm is mapped back (||L r~x|| = ||Qx + p + G^T z + A^T y||)
so `resids` (batch.py:107) means the same thing as in the reference.
"""
import numpy as np
import scipy.linalg as sla


def _tri(L, b, trans=False):
    return sla.solve_triangular(L, b, lower=True, trans=1 if trans else 0, check_finite=False)


def _chol(S):
    # non-raising Cholesky: a failed pivot yields NaN like the kernel's rsqrt of a negative number
    n = S.shape[0]
    L = np.array(S, dtype=np.float64)
    with np.errstate(all="ignore"):
        for k in range(n):
            L[k, k] = np.sqrt(L[k, k])
            L[k + 1:, k] /= L[k, k]
            L[k + 1:, k + 1:] -= np.outer(L[k + 1:, k], L[k + 1:, k])
    return np.tril(L)


def setup(Q, G, A):
    n = Q.shape[0]
    e = A.shape[0]
    try:
        L = np.linalg.cholesky(Q)
        ok = True
    except np.linalg.LinAlgError:
        L = _chol(Q); ok = False
    Gt = _tri(L, G.T).T
    f = dict(L=L, Gt=Gt, ok=ok, e=e)
    R = Gt @ Gt.T
    if e > 0:
        At = _tri(L, A.T).T
        L11 = _chol(At @ At.T)
        L21 = _tri(L11, (Gt @ At.T).T).T
        R = R - L21 @ L21.T
        f.update(At=At, L11=L11, L21=L21)
    f["R"] = R
    return f


def _solve_kkt(f, L22, d, t, rs, rz, ry):
    Gt = f["Gt"]
    hz = Gt @ t + rs / d - rz
    if f["e"] > 0:
        At, L11, L21 = f["At"], f["L11"], f["L21"]
        hy = At @ t - ry
        u1 = _tri(L11, -hy)
        u2 = _tri(L22, -hz - L21 @ u1)
        wz = _tri(L22, u2, trans=True)
        wy = _tri(L11, u1 - L21.T @ wz, trans=True)
        dxt = -t - Gt.T @ wz - At.T @ wy
    else:
        wz = _tri(L22, _tri(L22, -hz), trans=True)
        wy = None
        dxt = -t - Gt.T @ wz
    ds = (-rs - wz) / d
    return dxt, ds, wz, wy


def _step(v, dv):
    a = -v / dv
    a = np.where(dv > 0, np.inf, a)          # the fill value max(1.0, a.max()) (batch.py:212) is >= every entry
    st = a.min()
    return 1.0 if st == np.inf else st       # every dv > 0: the fill is max(1.0, negative) = 1.0 at nBatch=1


def solve_one(Q, p, G, h, A, b, eps=1e-12, notImprovedLim=3, maxIter=20, stall_tol=np.inf, use_eps=True, tie=1.0, noise=None,
              trace=None):
    """One QP with the kernels' per-QP exit rules. `trace` (a list) receives one tuple per iteration:
    (pri, dual, mu, resid, ret_it) - the four values the kernels write to their trace buffer (pri = |rz| + |ry|,
    dual = |L r~x|) and the index of the iterate that would be returned if the loop stopped there.
    `best_resid` is the residual of the returned iterate, as the kernels report it: on a BEST_TIE tie that is the
    later, tied iterate's residual, not the running minimum `min_resid` the exit tests use."""
    m, n = G.shape
    f = setup(Q, G, A)
    e = f["e"]
    L, Gt = f["L"], f["Gt"]
    At = f.get("At")
    pt = _tri(L, p)
    with np.errstate(all="ignore"):
        d = np.ones(m)
        L22 = _chol(f["R"] + np.diag(1.0 / d))
        xt, s, z, y = _solve_kkt(f, L22, d, pt, np.zeros(m), -h, -b if e > 0 else None)
        if s.min() < 0:
            s = s - (s.min() - 1)
        if z.min() < 0:
            z = z - (z.min() - 1)
        best = None
        nNot = 0
        iters = 0
        for it in range(maxIter):
            iters = it + 1
            rxt = xt + pt + Gt.T @ z + (At.T @ y if e > 0 else 0.0)
            rz = Gt @ xt + s - h
            ry = At @ xt - b if e > 0 else None
            mu = abs((s * z).sum() / m)
            pri = np.linalg.norm(rz) + (np.linalg.norm(ry) if e > 0 else 0.0)
            dual = np.linalg.norm(L @ rxt)
            resid = pri + dual + m * mu
            if noise is not None:
                resid = resid + abs(noise.randn()) * 3e-13
            d = z / s
            L22 = _chol(f["R"] + np.diag(1.0 / d))
            if best is None:
                best = dict(resid=resid, ret_resid=resid, xt=xt.copy(), s=s.copy(), z=z.copy(),
                            y=None if y is None else y.copy(), it=it)
                minres = resid
                nNot = 0
            elif resid < minres:
                best = dict(resid=resid, ret_resid=resid, xt=xt.copy(), s=s.copy(), z=z.copy(),
                            y=None if y is None else y.copy(), it=it)
                minres = resid
                nNot = 0
            else:
                nNot += 1
                if resid < tie * minres:     # within the tie factor of the minimum: prefer the later iterate
                    best = dict(resid=minres, ret_resid=resid, xt=xt.copy(), s=s.copy(), z=z.copy(),
                                y=None if y is None else y.copy(), it=it)
            if trace is not None:
                trace.append((pri, dual, mu, resid, best["it"]))
            if (nNot == notImprovedLim and best["resid"] < stall_tol) or (use_eps and best["resid"] < eps) or mu > 1e32:
                break
            if not np.isfinite(resid):
                break        # every later iterate is NaN too; `best` cannot change (batch.py:126)
            dxa, dsa, dza, dya = _solve_kkt(f, L22, d, rxt, z, rz, ry)
            alpha = min(_step(z, dza), _step(s, dsa), 1.0)
            sig = (((s + alpha * dsa) * (z + alpha * dza)).sum() / (s * z).sum()) ** 3
            rs_c = (-mu * sig + dsa * dza) / s
            dxc, dsc, dzc, dyc = _solve_kkt(f, L22, d, np.zeros(n), rs_c, np.zeros(m),
                                            np.zeros(e) if e > 0 else None)
            dx, ds, dz = dxa + dxc, dsa + dsc, dza + dzc
            alpha = min(0.999 * min(_step(z, dz), _step(s, ds)), 1.0)
            xt = xt + alpha * dx; s = s + alpha * ds; z = z + alpha * dz
            if e > 0:
                y = y + alpha * (dya + dyc)
    x = _tri(L, best["xt"], trans=True)
    return dict(x=x, lam=best["z"], s=best["s"], nu=best["y"], f=f, iters=iters,
                best_resid=best["ret_resid"], min_resid=best["resid"], best_iter=best["it"])


def backward_one(sol, dl):
    f = sol["f"]
    L = f["L"]
    m = f["Gt"].shape[0]
    e = f["e"]
    with np.errstate(all="ignore"):
        d = np.maximum(sol["lam"], 1e-8) / np.maximum(sol["s"], 1e-8)
        L22 = _chol(f["R"] + np.diag(1.0 / d))
        t = _tri(L, dl)
        dxt, _, dlam, dnu = _solve_kkt(f, L22, d, t, np.zeros(m), np.zeros(m),
                                       np.zeros(e) if e > 0 else None)
        dx = _tri(L, dxt, trans=True)
    x, lam = sol["x"], sol["lam"]
    g = dict(dQ=0.5 * (np.outer(dx, x) + np.outer(x, dx)), dp=dx,
             dG=np.outer(dlam, x) + np.outer(lam, dx), dh=-dlam)
    if e > 0:
        g["dA"] = np.outer(dnu, x) + np.outer(sol["nu"], dx)
        g["db"] = -dnu
    return g


def qp_solve(Q, p, G, h, A, b, dl=None, trace=None, **opts):
    """Batched (all inputs batched) wrapper; returns stacked outputs like pdipm_oracle.qp_solve.
    `trace` (a list) receives one per-QP trace list (see solve_one) per QP."""
    B = Q.shape[0]
    sols = []
    for i in range(B):
        tr = None if trace is None else []
        sols.append(solve_one(Q[i], p[i], G[i], h[i], A[i], b[i], trace=tr, **opts))
        if trace is not None:
            trace.append(tr)
    out = dict(zhat=np.stack([s["x"] for s in sols]), lam=np.stack([s["lam"] for s in sols]),
               slacks=np.stack([s["s"] for s in sols]),
               nus=np.stack([s["nu"] for s in sols]) if A.shape[1] > 0 else None,
               iters=np.array([s["iters"] for s in sols]),
               best_resids=np.array([s["best_resid"] for s in sols]),
               best_iter=np.array([s["best_iter"] for s in sols]))
    if dl is not None:
        gs = [backward_one(s, dl[i]) for i, s in enumerate(sols)]
        out["grads"] = {k: np.stack([g[k] for g in gs]) for k in gs[0]}
    return out
