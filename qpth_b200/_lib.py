"""ctypes binding of the C ABI in include/qpth_b200.h (libqpth_b200.so, built in-tree by build.py).

There is no CPU fallback: if the shared library is missing, or no CUDA device is
present when a solve is requested, the call fails loudly.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# QPB200_LIB: development override (A/B builds of the kernels); the product is the in-tree libqpth_b200.so
LIB_PATH = os.environ.get("QPB200_LIB") or os.path.join(_HERE, "libqpth_b200.so")

c_double_p = ctypes.c_void_p
c_int_p = ctypes.c_void_p


class Plan(ctypes.Structure):
    """Mirror of `qpb200_plan` (include/qpth_b200.h)."""
    _fields_ = [
        ("nz", ctypes.c_int), ("nineq", ctypes.c_int), ("neq", ctypes.c_int),
        ("neq_pad", ctypes.c_int), ("ms", ctypes.c_int), ("ms_pad", ctypes.c_int),
        ("ldw", ctypes.c_int), ("lds", ctypes.c_int), ("rows_s", ctypes.c_int), ("vl", ctypes.c_int),
        ("smem_resident", ctypes.c_int), ("threads", ctypes.c_int), ("fast", ctypes.c_int), ("setup_fast", ctypes.c_int),
        ("L_elems", ctypes.c_int64), ("W_elems", ctypes.c_int64), ("K_elems", ctypes.c_int64),
        ("setup_scratch_elems", ctypes.c_int64), ("solve_scratch_elems", ctypes.c_int64),
        ("setup_smem_bytes", ctypes.c_int64), ("solve_smem_bytes", ctypes.c_int64),
        ("coop_smem_bytes", ctypes.c_int64), ("coop_ok", ctypes.c_int), ("coop", ctypes.c_int), ("tiny", ctypes.c_int),
        ("pf", ctypes.c_int), ("pf_global", ctypes.c_int), ("pf_smem_bytes", ctypes.c_int64),
        ("pf2_ok", ctypes.c_int), ("pf_two", ctypes.c_int), ("pf2_smem_bytes", ctypes.c_int64),
        ("pf3_ok", ctypes.c_int), ("pf_three", ctypes.c_int), ("pf3_smem_bytes", ctypes.c_int64), ("pf_threads", ctypes.c_int),
        ("setup_pf", ctypes.c_int), ("setup_pf_smem_bytes", ctypes.c_int64),
    ]


# symbol -> (restype, argtypes); also the list tests use to check every declared export exists
_I, _L, _D, _P = ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p
SIGNATURES = {
    "qpb200_version": (_I, []),
    "qpb200_error_string": (ctypes.c_char_p, [_I]),
    "qpb200_last_cuda_error": (ctypes.c_char_p, []),
    "qpb200_plan_init": (_I, [_I, _I, _I, ctypes.POINTER(Plan)]),
    "qpb200_pre_factor_kkt": (_I, [ctypes.POINTER(Plan), _I, _P, _L, _P, _L, _P, _L, _P, _P, _P, _P, _P, _P]),
    "qpb200_forward": (_I, [ctypes.POINTER(Plan), _I, _P, _L, _P, _L, _P, _L, _P, _P, _P, _I,
                            _D, _D, _D, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "qpb200_backward": (_I, [ctypes.POINTER(Plan), _I, _P, _P, _P, _P, _P, _P, _P, _P, _I,
                             _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P]),
    "qpb200_solve_kkt": (_I, [ctypes.POINTER(Plan), _I, _P, _P, _P, _P, _P, _P, _P, _P, _I,
                              _P, _P, _P, _P, _P, _P]),
    "qpb200_pre_factor_kkt_reg": (_I, [ctypes.POINTER(Plan), _I, _P, _L, _P, _L, _P, _L, _D, _P, _P, _P, _P, _P, _P]),
    "qpb200_solve_kkt_reg": (_I, [ctypes.POINTER(Plan), _I, _P, _P, _P, _P, _P, _D, _P, _P, _P, _I,
                                  _P, _P, _P, _P, _P, _P]),
    "qpb200_optnet_construct": (_I, [_I, _I, _P, _P, _P, _P, _D, _P, _P, _P]),
    "qpb200_optnet_chain": (_I, [_I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "qpb200_dfma_probe": (_I, [_I, _I, _I, _P, _P]),
    "qpb200_copy_lower": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "qpb200_qp_host": (_I, [_I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _D, _I, _I,
                            _P, _P, _P, _P, _P, _P, _P, _P]),
}

_lib = None


class QpthB200Error(RuntimeError):
    pass


def load():
    """Load libqpth_b200.so (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise QpthB200Error(
            "qpth_b200: %s is missing — build it with `python -m qpth_b200.build` "
            "(there is no CPU fallback)." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        lib = load()
        msg = lib.qpb200_error_string(rc).decode()
        if rc == 3:
            msg += ": " + lib.qpb200_last_cuda_error().decode()
        raise QpthB200Error("qpth_b200: " + msg)


_plans = {}


def plan_for(nz, nineq, neq, two=None):
    """Plan for a shape (cached). `two`: None = the library default; True / False = select / deselect the
    several-QPs-per-SM variants of the product-form solve kernels when the shape has them (three per SM if
    plan.pf3_ok, else two if plan.pf2_ok). Every (shape, two) pair has its own Plan object, so concurrent callers
    never see each other's choice. QPB200_MAXQPS=2 (development knob) caps the choice at two per SM."""
    # QPB200_PF (development / A-B knob read by qpb200_plan_init: "0" never, "1" product-form kernels wherever they fit,
    # "2" = "1" + the two-QPs-per-SM variant by default). Every knob that changes the plan is part of the key.
    key = (nz, nineq, neq, os.environ.get("QPB200_PF"), os.environ.get("QPB200_MAXQPS"), os.environ.get("QPB200_NT512"),
           os.environ.get("QPB200_SETUP_PF"), os.environ.get("QPB200_COOP"),
           None if two is None else bool(two))
    if key not in _plans:
        p = Plan()
        rc = load().qpb200_plan_init(nz, nineq, neq, ctypes.byref(p))
        check(rc)
        if os.environ.get("QPB200_COOP") is not None and p.coop_ok:     # development knob: force a kernel family
            p.coop = 1 if os.environ["QPB200_COOP"] == "1" else 0
        if two is not None:        # throughput mode: as many QPs per SM as the shape has a kernel for
            p.pf_three = 1 if (two and p.pf3_ok and os.environ.get("QPB200_MAXQPS", "3") == "3") else 0
            p.pf_two = 1 if (two and p.pf2_ok and not p.pf_three) else 0
        _plans[key] = p
    return _plans[key]


_sm_count = {}


def sm_count(device_index):
    if device_index not in _sm_count:
        import torch
        _sm_count[device_index] = torch.cuda.get_device_properties(device_index).multi_processor_count
    return _sm_count[device_index]
