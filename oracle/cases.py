"""Golden-case recipes shared by `oracle/gen_golden.py` and `tests/` (TEST INFRASTRUCTURE ONLY).

Every case is rebuilt from seeds; the committed fixtures under tests/golden/
hold the reference's outputs for exactly these inputs plus an input checksum.
"""
import numpy as np

from qpth_b200.problems import random_qp_batch, cls_layer_problem, c5_shard


def checksum(prob):
    return float(sum(np.abs(np.asarray(prob[k], dtype=np.float64)).sum() for k in ("Q", "p", "G", "h", "A", "b")))


def proj(n):
    return np.cos(np.arange(1, n + 1, dtype=np.float64))


def shared_problem(seed=3, B=6, n=12, m=8, e=3):
    """Q, G, h, A un-batched; p, b batched -> exercises the .mean(0) rule (qp.py:159-177)."""
    pr = random_qp_batch(1, n, m, e, seed=seed)
    rs = np.random.RandomState(seed + 100)
    z0 = rs.randn(B, n)
    out = dict(Q=pr["Q"][0], G=pr["G"][0], A=pr["A"][0],
               h=pr["h"][0] + 1.0, p=rs.randn(B, n), b=z0 @ pr["A"][0].T, dl=rs.randn(B, n))
    return out


def unbatched_problem(seed=4, n=9, m=6, e=2):
    pr = random_qp_batch(1, n, m, e, seed=seed)
    return {k: v[0] for k, v in pr.items()}


def testpy_problem(nz=10, neq=2, nineq=3, Qscale=1., Gscale=1., Ascale=1.):
    """test.py:42-66 (`get_grads`): npr.seed(1), nBatch=1, loss 0.5||z - truez||^2."""
    npr = np.random.RandomState(1)
    L = npr.randn(nz, nz)
    Q = Qscale * L.dot(L.T)
    G = Gscale * npr.randn(nineq, nz)
    z0 = npr.randn(nz)
    s0 = npr.rand(nineq)
    h = G.dot(z0) + s0
    A = Ascale * npr.randn(neq, nz)
    b = A.dot(z0)
    p = npr.randn(1, nz)
    truez = npr.randn(1, nz)
    return dict(Q=Q, p=p, G=G, h=h, A=A, b=b, truez=truez)



def sweep_spec(i):
    """Deterministic recipe of sweep case i (dims, conditioning, activity), i in range(N_SWEEP)."""
    rs = np.random.RandomState(7000 + i)
    nz = int(rs.randint(5, 121))
    nineq = int(rs.randint(1, 105))
    neq = int(rs.choice([0, 0, 1, 3, 8, 20]))
    neq = min(neq, max(0, nz - 1))                        # A must keep full row rank
    logk = float([0, 0, 2, 4, 6, 8][i % 6])               # condition number of Q: 10**logk .. (generic when 0)
    active = bool((i // 6) % 2)                           # pull the unconstrained optimum far outside: many active rows
    B = 4 if nz * nineq > 4000 else 6
    return dict(nz=nz, nineq=nineq, neq=neq, logk=logk, active=active, B=B, seed=7000 + i)


N_SWEEP = 48


def sweep_problem(i):
    """Randomised parity sweep (VERDICT r1 item 1b): nz 5..120, nineq 1..104, neq 0..20, Q with a prescribed
    condition number up to 1e8 (orthogonal basis x log-spaced spectrum), tight slacks / large p so that the
    active set is close to nz on the `active` cases.  Everything batched, strictly feasible by construction."""
    sp = sweep_spec(i)
    rs = np.random.RandomState(sp["seed"])
    B, n, m, e = sp["B"], sp["nz"], sp["nineq"], sp["neq"]
    Q = np.empty((B, n, n))
    for k in range(B):
        if sp["logk"] > 0:
            U, _ = np.linalg.qr(rs.randn(n, n))
            ev = np.logspace(0.0, -sp["logk"], n)
            Qk = (U * ev) @ U.T
            Q[k] = 0.5 * (Qk + Qk.T)
        else:
            L = rs.rand(n, n)
            Q[k] = L @ L.T + 1e-3 * np.eye(n)
    G = rs.randn(B, m, n)
    z0 = rs.randn(B, n)
    s0 = rs.rand(B, m) * (0.05 if sp["active"] else 1.0)
    p = rs.randn(B, n) * (30.0 if sp["active"] else 1.0)
    if sp["logk"] > 0:
        p = p * 10.0 ** (-sp["logk"] / 2)                 # keep |Q^-1 p| moderate for ill-conditioned Q
    h = np.einsum("bmn,bn->bm", G, z0) + s0
    A = rs.randn(B, e, n)
    b = np.einsum("ben,bn->be", A, z0)
    dl = rs.randn(B, n)
    return dict(Q=Q, p=p, G=G, h=h, A=A, b=b, dl=dl)


def sudoku_structured_problem(seed=31, B=12, n=64, e=40):
    """The structure of example-sudoku.ipynb:305-323 (the OptNet sudoku layer for 4 x 4 boards): Q = 0.1 I (diagonal),
    G = -I, h = 0 (z >= 0), a SHARED dense A with b = A z0 for a strictly positive z0, batched p. This is the problem
    class the reference's sparse path (SpQPFunction, dead code) was written for; here it goes through the dense kernels
    (order of the reduced system: 40 + 64 = 104)."""
    rs = np.random.RandomState(seed)
    A = rs.randn(e, n)
    z0 = rs.rand(n) + 0.1
    return dict(Q=0.1 * np.eye(n), p=-rs.rand(B, n), G=-np.eye(n), h=np.zeros(n), A=A, b=A @ z0, dl=rs.randn(B, n))


def util_results(U):
    """What the helpers of qpth/util.py (`U`: qpth_b200.util, or the reference's module) return on fixed inputs, as
    JSON data: batch sizes, expandParam's (shape, stride, expanded), get_sizes, bdiag."""
    import torch
    e, Q, q, p, h = torch.Tensor(), torch.zeros(3, 4, 4), torch.zeros(4, 4), torch.zeros(4), torch.zeros(3)
    G, A = torch.zeros(4, 3, 5), torch.zeros(4, 2, 5)
    out = {"extract_nBatch": [U.extract_nBatch(Q, p, G[:3, :, :4], h, e, e), U.extract_nBatch(q, p, G[0, :, :4], h, e, e)],
           "expandParam": [], "get_sizes": list(U.get_sizes(G, A)),
           "bdiag": U.bdiag(torch.arange(6.).view(2, 3)).tolist()}
    for X, nd in ((Q, 3), (q, 3), (p, 2), (e, 3), (torch.tensor(1.0), 2)):
        Y, expanded = U.expandParam(X, 3, nd)
        out["expandParam"].append([list(Y.shape), list(Y.stride()), bool(expanded)])
    return out


def _testpy(tag_kw):
    def build():
        return testpy_problem(**tag_kw)
    return build


# name -> (builder, full_mats)
CASES = {
    "c1": (lambda: random_qp_batch(4, 10, 5, 0, seed=0), True),
    "eq_small": (lambda: random_qp_batch(8, 20, 15, 5, seed=1), True),
    "ineq_only_wide": (lambda: random_qp_batch(5, 7, 19, 0, seed=2), True),
    "shared": (shared_problem, True),
    "unbatched": (unbatched_problem, True),
    "c2": (lambda: random_qp_batch(128, 100, 100, 0, seed=0), False),
    "c3_b64": (lambda: random_qp_batch(64, 50, 50, 10, seed=0), False),
    "c4": (lambda: cls_layer_problem(64, 200, 200, seed=0), True),
    "c4_small": (lambda: cls_layer_problem(8, 40, 40, seed=0), True),
    "testpy_dp": (_testpy(dict(neq=2, nineq=3, Qscale=100., Gscale=100., Ascale=100.)), True),
    "testpy_dG": (_testpy(dict(neq=0, nineq=3)), True),
    "testpy_dA": (_testpy(dict(neq=3, nineq=1)), True),
    # ---- round 2: BASELINE.json configs at their full sizes, the kernel-selection bands, the randomised sweep
    "c3": (lambda: random_qp_batch(1024, 50, 50, 10, seed=0), False),
    "c5_shard0": (lambda: c5_shard(0), False),
    "band_smem": (lambda: random_qp_batch(6, 20, 120, 0, seed=21), True),        # fast=0, smem_resident=1
    "band_smem_eq": (lambda: random_qp_batch(6, 24, 116, 4, seed=22), True),
    "band_setup": (lambda: random_qp_batch(6, 150, 20, 0, seed=23), False),      # fast=1, setup_fast=0
    "band_setup_eq": (lambda: random_qp_batch(6, 140, 24, 3, seed=24), False),
    "sudoku_structured": (sudoku_structured_problem, True),                     # SURVEY 8f.4: diagonal Q, G = -I, shared A
}
for _i in range(N_SWEEP):
    CASES["sweep%02d" % _i] = ((lambda i=_i: sweep_problem(i)), True)

# cases whose reference run takes more than a few seconds on CPU (kept out of the CPU oracle-vs-golden loops)
BIG = ("c2", "c4", "c3", "c5_shard0")


def load_case(name, golden_dir):
    """Rebuild the inputs of golden case `name` and load the reference's outputs for it."""
    import os
    build, full_mats = CASES[name]
    prob = build()
    dlp = os.path.join(golden_dir, name + "_dl.npy")
    if os.path.exists(dlp):
        prob["dl"] = np.load(dlp)
    gold = dict(np.load(os.path.join(golden_dir, name + ".npz")))
    cs = checksum(prob)
    assert abs(cs - float(gold["input_checksum"])) <= 1e-9 * abs(cs), \
        "golden inputs no longer reproduce from the seed (numpy RandomState changed?)"
    return prob, gold, full_mats
