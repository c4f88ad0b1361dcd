"""CPU-only checks of the C-ABI boundary: the library builds, loads, and exports every symbol the
header declares; plan sizes are sane. No compute calls (no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from qpth_b200 import build, _lib
    build.build()
    return _lib.load()


def test_header_symbols_all_exported(lib):
    from qpth_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "qpth_b200.h")).read()
    declared = set(re.findall(r"\b(qpb200_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))


def test_version_and_error_strings(lib):
    assert lib.qpb200_version() >= 100
    assert lib.qpb200_error_string(0) == b"ok"
    assert b"nineq" in lib.qpb200_error_string(2)


def test_plan_shapes(lib):
    from qpth_b200 import _lib
    p = _lib.plan_for(100, 100, 0)
    assert (p.ms, p.neq_pad, p.smem_resident) == (100, 0, 1)
    assert p.solve_smem_bytes <= 232448 and p.ldw % 8 == 4 and p.lds % 8 == 4
    p = _lib.plan_for(50, 50, 10)
    assert (p.neq_pad, p.ms) == (16, 66)
    p = _lib.plan_for(200, 200, 0)         # product-form "large problem" kernels: factor in shared memory, W / L from L2
    assert p.smem_resident == 0 and (p.pf, p.pf_global, p.pf2_ok) == (1, 1, 0) and p.pf_smem_bytes <= 232448 - 1024
    assert p.solve_scratch_elems == 0 and p.setup_pf == 1 and p.setup_scratch_elems == 0 and p.K_elems == 32 * 25 * 25 + 64 * 25
    assert p.setup_pf_smem_bytes <= 232448 - 1024 and _lib.plan_for(100, 100, 0).setup_pf == 0      # (k_setup_fast is faster there)
    p = _lib.plan_for(200, 200, 16)        # does not fit any shared-memory variant: global-scratch kernels
    assert p.pf == 0 and p.solve_scratch_elems > 0
    p = _lib.plan_for(100, 100, 0)         # both product-form variants; the second one fits twice into an SM
    assert (p.pf, p.pf_global, p.pf2_ok) == (1, 0, 1) and 2 * (p.pf2_smem_bytes + 1024) <= 232448
    assert 3 * (p.pf3_smem_bytes + 1024) <= 233472 and p.pf3_ok == 1        # ... and the 192-thread build three times
    pt, pl = _lib.plan_for(100, 100, 0, two=True), _lib.plan_for(100, 100, 0, two=False)
    assert (pt.pf_three, pt.pf_two) == (1, 0) and (pl.pf_three, pl.pf_two) == (0, 0)
    assert _lib.plan_for(200, 200, 0).pf_threads == 512 and p.pf_threads == 256
    # kernel-family selection (include/qpth_b200.h): co-resident fast kernels at C2/C3, one warp per QP for tiny shapes
    p = _lib.plan_for(100, 100, 0)
    assert (p.fast, p.coop_ok, p.tiny, p.threads) == (1, 1, 0, 256) and 2 * (p.coop_smem_bytes + 1024) <= 232448
    p = _lib.plan_for(10, 5, 0)
    assert (p.tiny, p.threads, p.fast, p.smem_resident, p.coop) == (1, 32, 0, 1, 0) and 16 * p.solve_smem_bytes <= 232448
    p = _lib.plan_for(32, 24, 8)
    assert p.tiny == 1
    p = _lib.plan_for(33, 10, 0)
    assert p.tiny == 0
    p = _lib.plan_for(150, 20, 0)          # chol(Q) does not fit the S workspace it would have to visit
    assert (p.fast, p.setup_fast, p.coop_ok) == (1, 0, 0)
    bad = _lib.Plan()
    assert lib.qpb200_plan_init(5, 0, 0, ctypes.byref(bad)) == 2      # QPB200_ERR_NO_CONSTRAINTS
    assert lib.qpb200_plan_init(0, 3, 0, ctypes.byref(bad)) == 1


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from qpth_b200 import QPFunction
    from qpth_b200._lib import QpthB200Error
    Q = torch.eye(3, dtype=torch.float64)
    with pytest.raises(QpthB200Error, match="no CUDA device"):
        QPFunction()(Q, torch.zeros(3, dtype=torch.float64), torch.eye(3, dtype=torch.float64),
                     torch.ones(3, dtype=torch.float64), torch.Tensor(), torch.Tensor())


def test_util_mirrors_reference_broadcast_rules():
    import torch
    from qpth_b200.util import expandParam, extract_nBatch
    Q = torch.eye(3); p = torch.zeros(5, 3)
    assert extract_nBatch(Q, p, Q, p[0], torch.Tensor(), torch.Tensor()) == 5
    X, flag = expandParam(Q, 5, 3)
    assert flag and X.shape == (5, 3, 3) and X.stride(0) == 0
    X, flag = expandParam(torch.Tensor(), 5, 3)
    assert not flag
    with pytest.raises(RuntimeError, match="Unexpected number of dimensions."):
        expandParam(torch.zeros(2, 2, 2, 2), 5, 3)


def test_util_helpers_behave_like_qpth_util():
    """get_sizes / bger / bdiag / to_np (qpth/util.py:9-41), and against what the real module returns
    (tests/golden/util_ref.json, oracle/gen_golden_host.py)."""
    import json
    import numpy as np
    import torch
    from oracle.cases import util_results
    from qpth_b200 import util as U
    G, A = torch.zeros(4, 3, 5), torch.zeros(4, 2, 5)
    assert U.get_sizes(G, A) == (3, 5, 2, 4)
    assert U.get_sizes(G[0]) == (3, 5, None, 1)
    assert U.get_sizes(G, torch.Tensor()) == (3, 5, 0, 4)
    x, y = torch.arange(6.).view(2, 3), torch.arange(8.).view(2, 4)
    assert torch.equal(U.bger(x, y), torch.einsum("bi,bj->bij", x, y))
    D = U.bdiag(x)
    assert D.shape == (2, 3, 3) and torch.equal(torch.diagonal(D, dim1=1, dim2=2), x) and D.sum() == x.sum()
    assert U.to_np(None) is None and U.to_np(torch.Tensor()).size == 0 and np.array_equal(U.to_np(x), x.numpy())
    with open(os.path.join(ROOT, "tests", "golden", "util_ref.json")) as fh:
        assert util_results(U) == json.load(fh)


def test_shape_validation_raises_before_the_device_is_touched():
    """ADVICE r1: mismatched trailing dimensions / batch sizes must raise, not reach the kernels (CPU-only check:
    the validation runs before the library or a CUDA device is needed)."""
    import pytest
    import torch
    from qpth_b200 import QPFunction
    from qpth_b200.util import check_shapes
    B, n, m, e = 3, 5, 4, 2
    d = torch.float64
    Q, p = torch.eye(n, dtype=d).repeat(B, 1, 1), torch.zeros(B, n, dtype=d)
    G, h = torch.ones(B, m, n, dtype=d), torch.ones(B, m, dtype=d)
    A, b = torch.ones(B, e, n, dtype=d), torch.ones(B, e, dtype=d)
    E = torch.Tensor()
    assert check_shapes(Q, p, G, h, A, b) == (B, n, m, e)
    assert check_shapes(Q[0], p, G[0], h[0], E, E) == (B, n, m, 0)
    bad = [
        (Q, p[:, :-1], G, h, A, b),                 # p.size(-1) != nz
        (Q, p, G[:, :, :-1], h, A, b),              # G.size(-1) != nz
        (Q, p, G, h[:, :-1], A, b),                 # h.size(-1) != nineq
        (Q, p, G, h, A[:, :, :-1], b),              # A.size(-1) != nz
        (Q, p, G, h, A, b[:, :-1]),                 # b.size(-1) != neq
        (Q[:, :, :-1], p, G, h, A, b),              # Q not square
        (Q, p[:2], G, h, A, b),                     # batch sizes disagree
        (Q, p, G.new_ones(1, m, n), h, A, b),       # G batched over 1, Q over B
        (Q, p, G, h, E, b),                         # b without A
    ]
    for args in bad:
        with pytest.raises(RuntimeError, match="inconsistent shapes"):
            check_shapes(*args)
        with pytest.raises(RuntimeError, match="inconsistent shapes"):
            QPFunction(verbose=-1)(*args)
    with pytest.raises(RuntimeError, match="Unexpected number of dimensions."):
        QPFunction(verbose=-1)(Q[None], p, G, h, A, b)


def test_plan_invariants_over_a_shape_grid(lib):
    """Every shape the planner accepts must get a launchable configuration: the shared memory of the family it selects
    fits one CTA (227 KB opt-in limit), a promised co-residency (two / three QPs per SM) fits the SM's 228 KB including the
    1 KB the driver reserves per CTA, the tile bookkeeping of the product-form kernels stays inside its table, and a
    shape without a shared-memory variant has its global scratch sized. Shapes the kernels cannot take are refused by
    plan_init (QPB200_ERR_TOO_LARGE), never accepted with an impossible plan."""
    from qpth_b200 import _lib
    cta_max, sm_total = 232448, 233472
    seen = {"tiny": 0, "pf": 0, "pf3": 0, "pf2": 0, "global": 0, "refused": 0, "fast": 0}
    for nz in (1, 2, 7, 8, 9, 16, 31, 32, 33, 50, 64, 100, 104, 105, 128, 150, 200, 256, 400):
        for nineq in (0, 1, 5, 8, 24, 32, 50, 64, 100, 104, 105, 120, 128, 200, 256, 400):
            for neq in (0, 1, 8, 10, 40, 100):
                if nineq + neq == 0:
                    continue
                p = _lib.Plan()
                rc = lib.qpb200_plan_init(nz, nineq, neq, ctypes.byref(p))
                if rc != 0:
                    assert rc == 4, (nz, nineq, neq, rc)
                    seen["refused"] += 1
                    continue
                tag = (nz, nineq, neq)
                assert p.neq_pad % 8 == 0 and p.neq_pad >= neq and p.ms == p.neq_pad + nineq, tag
                assert p.ms_pad % 8 == 0 and 0 <= p.ms_pad - p.ms < 8, tag
                assert p.L_elems >= nz * (nz + 1) // 2 and p.W_elems >= p.ms * nz and p.K_elems > 0, tag
                assert p.threads in (32, 256) and p.pf_threads in (0, 256, 512), tag
                if p.tiny:
                    assert nz <= 32 and p.ms_pad <= 32 and p.threads == 32 and p.smem_resident == 1, tag
                    assert 4 * (p.solve_smem_bytes + 1024) <= sm_total, tag       # (up to 16 per SM for the smallest)
                    seen["tiny"] += 1
                if p.pf:
                    t = p.ms_pad // 8
                    assert p.K_elems == 32 * t * t + 64 * t, tag
                    assert p.pf_smem_bytes <= cta_max, tag
                    assert p.pf_global in (0, 1) and (p.pf_threads == 256 or (p.pf_global == 1 and p.ms_pad > 128)), tag
                    seen["pf"] += 1
                    if p.pf2_ok:
                        assert 2 * (p.pf2_smem_bytes + 1024) <= sm_total, tag
                        seen["pf2"] += 1
                    if p.pf3_ok:
                        assert 3 * (p.pf3_smem_bytes + 1024) <= sm_total, tag
                        seen["pf3"] += 1
                    if p.setup_pf:
                        assert p.setup_pf_smem_bytes <= cta_max, tag
                else:
                    assert (p.pf2_ok, p.pf3_ok, p.pf_two, p.pf_three) == (0, 0, 0, 0), tag
                if p.coop_ok:
                    assert 2 * (p.coop_smem_bytes + 1024) <= sm_total, tag
                if p.smem_resident:
                    assert p.solve_smem_bytes <= cta_max and p.solve_scratch_elems == 0, tag
                elif not p.pf:
                    assert p.solve_scratch_elems > 0 and p.setup_scratch_elems > 0, tag
                    seen["global"] += 1
                if not (p.pf and p.setup_pf) and p.smem_resident:
                    assert p.setup_smem_bytes <= cta_max, tag
                seen["fast"] += int(p.fast)
    assert min(seen[k] for k in ("tiny", "pf", "pf2", "pf3", "global", "fast")) > 0, seen     # the grid reaches every family
