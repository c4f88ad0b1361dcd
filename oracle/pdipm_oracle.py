"""CPU oracle: numpy/scipy restatement of qpth's batched dense PDIPM (TEST INFRASTRUCTURE ONLY).

This file restates, function by function, the algorithm of the reference
(`/root/reference`, locuslab/qpth @ 528e9f6) for the hot path
`QPFunction()(Q,p,G,h,A,b)` forward + backward.  It exists to CHECK the CUDA
product in `qpth_b200/`; nothing in the product may import it.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs use it.

Parity status: PINNED.  `oracle/gen_golden.py` imports the real reference in
the build container, runs it on seeded problems and commits its outputs under
`tests/golden/`; `tests/test_oracle.py` checks this restatement against those
vectors (z*, lambda, s, nu and all six gradients).

Arithmetic notes.  The reference's factorizations live in PyTorch -> LAPACK
getrf/getrs with partial pivoting (`qpth/solvers/pdipm/batch.py:8-20`); here
they are `scipy.linalg.lu_factor/lu_solve` (same LAPACK routines, different
BLAS build), so results agree to rounding, not bit for bit.  The reference's
block-LU bookkeeping (`batch.py:402-424,450-470`: packed S_LU with re-pivoted
S_LU_21) is restated as the block elimination it implements: LU(A Q^-1 A^T)
once, LU(R + D^-1) per call with R the Schur complement of that block.
"""
import numpy as np
import scipy.linalg as sla

INACC_ERR = "qpth warning: Returning an inaccurate and potentially incorrect solution."


class _Singular(Exception):
    pass


def _lu(x):
    """`lu_hack` on CPU (batch.py:8-20): pivoted LU; exact-zero pivot raises like torch.linalg.lu_factor."""
    lu, piv = sla.lu_factor(x, check_finite=False)
    if np.any(np.diag(lu) == 0.0):
        raise _Singular()
    return lu, piv


def _lus(f, rhs):
    return sla.lu_solve(f, rhs, check_finite=False)


def expand_param(X, nBatch, nDim):
    """util.py:44-50."""
    X = np.asarray(X)
    if X.ndim in (0, nDim) or X.size == 0:
        return X, False
    if X.ndim == nDim - 1:
        return np.broadcast_to(X[None], (nBatch,) + X.shape), True
    raise RuntimeError("Unexpected number of dimensions.")


def extract_nbatch(Q, p, G, h, A, b):
    """util.py:53-59."""
    for prm, dim in zip((Q, p, G, h, A, b), (3, 2, 3, 2, 3, 2)):
        if np.asarray(prm).ndim == dim:
            return np.asarray(prm).shape[0]
    return 1


class Factors:
    """What `pre_factor_kkt` returns (batch.py:375-429), per QP."""

    def __init__(self, Q, G, A):
        B, m, n = G.shape
        e = A.shape[1] if A.size > 0 else 0
        self.B, self.n, self.m, self.e = B, n, m, e
        self.Q_LU, self.A_LU, self.T_LU = [], [], [None] * B
        self.R = np.empty((B, m, m))
        self.GiA = [None] * B      # G Q^-1 A^T
        for i in range(B):
            qlu = _lu(Q[i])                               # batch.py:380
            self.Q_LU.append(qlu)
            R = G[i] @ _lus(qlu, G[i].T)                  # batch.py:396-399
            if e > 0:
                invQ_AT = _lus(qlu, A[i].T)               # batch.py:403
                A_invQ_AT = A[i] @ invQ_AT                # batch.py:404
                G_invQ_AT = G[i] @ invQ_AT                # batch.py:405
                alu = _lu(A_invQ_AT)                      # batch.py:407
                self.A_LU.append(alu)
                T = _lus(alu, G_invQ_AT.T)                # batch.py:414-415
                R = R - G_invQ_AT @ T                     # batch.py:424
                self.GiA[i] = G_invQ_AT
            self.R[i] = R

    def factor_kkt(self, d):
        """batch.py:435-470: LU of R + diag(1/d), per QP. Raises _Singular like the reference."""
        for i in range(self.B):
            T = self.R[i].copy()
            T[np.diag_indices(self.m)] += 1.0 / d[i]
            self.T_LU[i] = _lu(T)

    def solve_kkt(self, G, A, d, rx, rs, rz, ry):
        """batch.py:349-372 with the block-LU of S applied as block elimination."""
        B, n, m, e = self.B, self.n, self.m, self.e
        dx = np.empty((B, n)); ds = np.empty((B, m)); dz = np.empty((B, m))
        dy = np.empty((B, e)) if e > 0 else None
        for i in range(B):
            invQ_rx = _lus(self.Q_LU[i], rx[i])                        # :353
            hz = G[i] @ invQ_rx + rs[i] / d[i] - rz[i]                 # :355-358
            if e > 0:
                hy = A[i] @ invQ_rx - ry[i]
                # w = -S^-1 [hy; hz], S = [[S11, S12],[S21, R' + S21 S11^-1 S12 + D^-1]]
                u = _lus(self.A_LU[i], -hy)                            # S11^-1 (-hy)
                wz = _lus(self.T_LU[i], -hz - self.GiA[i] @ u)
                wy = u - _lus(self.A_LU[i], self.GiA[i].T @ wz)
            else:
                wz = _lus(self.T_LU[i], -hz)                           # :360
            g1 = -rx[i] - wz @ G[i]                                    # :362
            if e > 0:
                g1 = g1 - wy @ A[i]                                    # :363-364
                dy[i] = wy
            dx[i] = _lus(self.Q_LU[i], g1)                             # :367
            ds[i] = (-rs[i] - wz) / d[i]                               # :365,368
            dz[i] = wz
        return dx, ds, dz, dy


def get_step(v, dv):
    """batch.py:210-213 including the batch-global fill value and Python max() NaN behaviour."""
    with np.errstate(all="ignore"):
        a = -v / dv
        amax = a.max()
        fill = amax if amax > 1.0 else 1.0     # python max(1.0, t): t only if t > 1.0
        a = np.where(dv > 0, fill, a)
        return a.min(axis=1)


def forward(Q, p, G, h, A, b, F, eps=1e-12, verbose=0, notImprovedLim=3, maxIter=20, trace=None):
    """batch.py:47-207 (KKTSolvers.LU_PARTIAL branch). Returns best x, y, z, s and info."""
    B, m, n = G.shape
    e = F.e
    with np.errstate(all="ignore"):
        d = np.ones((B, m))
        F.factor_kkt(d)                                                    # :61-62
        x, s, z, y = F.solve_kkt(G, A, d, p, np.zeros((B, m)), -h,
                                 -b if e > 0 else None)                    # :63-66
        x = x.copy(); s = s.copy(); z = z.copy()
        M = s.min(axis=1); I = M < 0
        s[I] -= (M[I] - 1)[:, None]                                        # :77-81
        M = z.min(axis=1); I = M < 0
        z[I] -= (M[I] - 1)[:, None]                                        # :83-87

        best = dict(resids=None, x=None, z=None, s=None, y=None)
        best_iter = np.full(B, -1)
        nNotImproved = 0
        iters_run = 0
        for it in range(maxIter):
            iters_run = it + 1
            Gx = np.einsum("bmn,bn->bm", G, x)
            rx = np.einsum("bm,bmn->bn", z, G) + np.einsum("bnk,bk->bn", Q, x) + p   # :94-97
            if e > 0:
                rx = rx + np.einsum("be,ben->bn", y, A)
            rs = z
            rz = Gx + s - h                                                # :99
            ry = np.einsum("ben,bn->be", A, x) - b if e > 0 else None      # :100-101
            mu = np.abs((s * z).sum(1) / m)                                # :102
            z_resid = np.sqrt((rz * rz).sum(1))
            y_resid = np.sqrt((ry * ry).sum(1)) if e > 0 else 0.0
            pri_resid = y_resid + z_resid
            dual_resid = np.sqrt((rx * rx).sum(1))
            resids = pri_resid + dual_resid + m * mu                       # :107
            d = z / s                                                      # :109
            try:
                F.factor_kkt(d)                                            # :110-113
            except _Singular:
                break
            if verbose == 1:
                print("iter: {}, pri_resid: {:.5e}, dual_resid: {:.5e}, mu: {:.5e}".format(
                    it, pri_resid.mean(), dual_resid.mean(), mu.mean()))
            if best["resids"] is None:                                     # :118-124
                best["resids"] = resids.copy()
                best["x"], best["z"], best["s"] = x.copy(), z.copy(), s.copy()
                best["y"] = y.copy() if y is not None else None
                best_iter[:] = it
                nNotImproved = 0
            else:
                I = resids < best["resids"]                                # :126 (False for NaN)
                if I.sum() > 0:
                    nNotImproved = 0
                else:
                    nNotImproved += 1
                best["resids"][I] = resids[I]
                best["x"][I] = x[I]; best["z"][I] = z[I]; best["s"][I] = s[I]
                if e > 0:
                    best["y"][I] = y[I]
                best_iter[I] = it
            if trace is not None:
                trace.append(dict(it=it, resids=resids.copy(), mu=mu.copy(), pri=np.broadcast_to(pri_resid, (B,)).copy(),
                                  dual=dual_resid.copy(),
                                  x=x.copy(), s=s.copy(), z=z.copy()))
            bmax = best["resids"].max()
            mumin = mu.min()
            if nNotImproved == notImprovedLim or bmax < eps or mumin > 1e32:   # :140
                break
            dx_aff, ds_aff, dz_aff, dy_aff = F.solve_kkt(G, A, d, rx, rs, rz, ry)   # :150
            alpha = np.minimum(np.minimum(get_step(z, dz_aff), get_step(s, ds_aff)), 1.0)  # :160-162
            t1 = s + alpha[:, None] * ds_aff
            t2 = z + alpha[:, None] * dz_aff
            t3 = (t1 * t2).sum(1)
            t4 = (s * z).sum(1)
            sig = (t3 / t4) ** 3                                           # :164-168
            rs_c = (-(mu * sig)[:, None] + ds_aff * dz_aff) / s            # :171
            dx_cor, ds_cor, dz_cor, dy_cor = F.solve_kkt(
                G, A, d, np.zeros((B, n)), rs_c, np.zeros((B, m)),
                np.zeros((B, e)) if e > 0 else None)                       # :180
            dx = dx_aff + dx_cor; ds = ds_aff + ds_cor; dz = dz_aff + dz_cor
            dy = dy_aff + dy_cor if e > 0 else None
            alpha = np.minimum(0.999 * np.minimum(get_step(z, dz), get_step(s, ds)), 1.0)  # :189-191
            x = x + alpha[:, None] * dx                                    # :200-203
            s = s + alpha[:, None] * ds
            z = z + alpha[:, None] * dz
            y = y + alpha[:, None] * dy if e > 0 else None
    inaccurate = bool(best["resids"] is not None and np.nanmax(best["resids"]) > 1.0)
    info = dict(iters=iters_run, best_resids=best["resids"], best_iter=best_iter,
                inaccurate=inaccurate)
    return best["x"], best["y"], best["z"], best["s"], info


def backward(Q, G, A, F, zhat, lam, slacks, nus, dl, expanded):
    """qp.py:128-182. `expanded` = (Q_e, p_e, G_e, h_e, A_e, b_e) flags for the .mean(0) rule."""
    B, m, n = G.shape
    e = F.e
    with np.errstate(all="ignore"):
        d = np.maximum(lam, 1e-8) / np.maximum(slacks, 1e-8)               # qp.py:148
        F.factor_kkt(d)                                                    # qp.py:150
        dx, _, dlam, dnu = F.solve_kkt(G, A, d, dl, np.zeros((B, m)), np.zeros((B, m)),
                                       np.zeros((B, e)) if e > 0 else None)   # qp.py:151-155
        dps = dx
        dGs = dlam[:, :, None] * zhat[:, None, :] + lam[:, :, None] * dx[:, None, :]   # :158
        dhs = -dlam
        if e > 0:
            dAs = dnu[:, :, None] * zhat[:, None, :] + nus[:, :, None] * dx[:, None, :]
            dbs = -dnu
        else:
            dAs, dbs = None, None
        dQs = 0.5 * (dx[:, :, None] * zhat[:, None, :] + zhat[:, :, None] * dx[:, None, :])  # :174
    Q_e, p_e, G_e, h_e, A_e, b_e = expanded
    out = [dQs, dps, dGs, dhs, dAs, dbs]
    for k, flag in enumerate((Q_e, p_e, G_e, h_e, A_e, b_e)):
        if flag and out[k] is not None:
            out[k] = out[k].mean(0)                                        # qp.py:159-177
    return tuple(out)


def qp_solve(Q, p, G, h, A, b, dl=None, eps=1e-12, verbose=0, notImprovedLim=3, maxIter=20,
             check_Q_spd=True, per_qp=False, trace=None):
    """`QPFunction(...)(Q,p,G,h,A,b)` + `.backward(dl)` (qp.py:23-182) on numpy arrays.

    per_qp=True solves each QP as its own nBatch=1 call (the reference's
    semantics without its batch-global exit tests / get_step fill value).
    Returns dict(zhat, lam, slacks, nus, grads=(dQ,dp,dG,dh,dA,db) or None, info).
    """
    Q_, p_, G_, h_, A_, b_ = [np.asarray(v, dtype=np.float64) for v in (Q, p, G, h, A, b)]
    B = extract_nbatch(Q_, p_, G_, h_, A_, b_)
    Qe, Q_e = expand_param(Q_, B, 3)
    pe, p_e = expand_param(p_, B, 2)
    Ge, G_e = expand_param(G_, B, 3)
    he, h_e = expand_param(h_, B, 2)
    Ae, A_e = expand_param(A_, B, 3)
    be, b_e = expand_param(b_, B, 2)
    if check_Q_spd:
        try:
            for i in range(B if not Q_e else 1):
                np.linalg.cholesky(Qe[i])
        except np.linalg.LinAlgError:
            raise RuntimeError("Q is not SPD.")                            # qp.py:81-85
    _, m, n = Ge.shape
    e = Ae.shape[1] if Ae.size > 0 else 0
    assert e > 0 or m > 0

    def run(sl):
        Qs, ps, Gs, hs = Qe[sl], pe[sl], Ge[sl], he[sl]
        As = Ae[sl] if e > 0 else np.zeros((Gs.shape[0], 0, n))
        bs = be[sl] if e > 0 else np.zeros((Gs.shape[0], 0))
        F = Factors(Qs, Gs, As)
        x, y, z, s, info = forward(Qs, ps, Gs, hs, As, bs, F, eps, verbose, notImprovedLim,
                                   maxIter, trace)
        return F, x, y, z, s, info

    if not per_qp:
        F, x, y, z, s, info = run(slice(0, B))
        grads = None
        if dl is not None:
            As = Ae if e > 0 else np.zeros((B, 0, n))
            grads = backward(Qe, Ge, As, F, x, z, s, y, np.asarray(dl, dtype=np.float64).reshape(B, n),
                             (Q_e, p_e, G_e, h_e, A_e, b_e))
        return dict(zhat=x, lam=z, slacks=s, nus=y, grads=grads, info=info)

    xs, ys, zs, ss, infos, per = [], [], [], [], [], []
    dl = None if dl is None else np.asarray(dl, dtype=np.float64).reshape(B, n)
    for i in range(B):
        F, x, y, z, s, info = run(slice(i, i + 1))
        xs.append(x); ys.append(y); zs.append(z); ss.append(s); infos.append(info)
        if dl is not None:
            As = Ae[i:i + 1] if e > 0 else np.zeros((1, 0, n))
            per.append(backward(Qe[i:i + 1], Ge[i:i + 1], As, F, x, z, s, y, dl[i:i + 1],
                                (False,) * 6))
    x = np.concatenate(xs); z = np.concatenate(zs); s = np.concatenate(ss)
    y = np.concatenate(ys) if e > 0 else None
    grads = None
    if dl is not None:
        grads = []
        for k, flag in enumerate((Q_e, p_e, G_e, h_e, A_e, b_e)):
            if per[0][k] is None:
                grads.append(None)
                continue
            g = np.concatenate([pp[k] for pp in per])
            grads.append(g.mean(0) if flag else g)
        grads = tuple(grads)
    info = dict(iters=np.array([f["iters"] for f in infos]),
                best_resids=np.concatenate([f["best_resids"] for f in infos]),
                best_iter=np.concatenate([f["best_iter"] for f in infos]),
                inaccurate=any(f["inaccurate"] for f in infos))
    return dict(zhat=x, lam=z, slacks=s, nus=y, grads=grads, info=info)
