"""The argument checks of the C entry points, called through ctypes: return codes, and error texts that name the entry point.

Every call here either fails a check that comes before the n == 0 / npl == 0 return or runs at n == 0 / npl == 0, so no call
can reach a kernel launch whatever the order of the checks; all pointers are host buffers.  The no-device group passes
n > 0 and therefore runs only where no CUDA device exists: there every launcher must stop at its device check."""
import ctypes
import os
from ctypes import c_double, c_int, c_int64, c_size_t, c_uint32, c_void_p

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EK_OK, EK_ERR_ARG, EK_ERR_ENUM = 0, -1, -2
EK_TM_BISECT = 2
S_NSLOTS = 10


class Operand(ctypes.Structure):
    _fields_ = [("ptr", c_void_p), ("value", c_double)]


V, OP = c_void_p, Operand
ARGTYPES = {
    "suite_tqp": [OP, OP, OP, V, c_uint32, c_int, c_int64, V],
    "suite_ttdp": [OP, OP, OP, V, c_uint32, c_int, c_int64, V],
    "suite_tqp_batch": [c_int, V, V, V, V, V, V, c_uint32, c_int, c_int64, V],
    "suite_ttdp_batch": [c_int, V, V, V, V, V, V, c_uint32, c_int, c_int64, V],
    "suite_tq_hybrid": [V, V, V, V, V, c_int, c_int64, V, c_uint32, c_int, V, V],
    "suite_tq_hybrid_geo": [V, V, V, V, V, V, c_int, c_int64, V, c_uint32, c_int, V, c_int, c_double, V, V, V, c_int, V],
    "host_suite": [c_int, V, V, V, V, c_uint32, c_int, c_int64, V, c_size_t, c_int],
    "host_suite_tq_hybrid": [V, V, V, V, V, c_int, c_int64, V, c_uint32, c_int, V, c_size_t, c_int],
    "host_suite_tq_hybrid_geo": [V, V, V, V, V, V, c_int, c_int64, V, c_uint32, c_int, c_int, c_double, V, V, V, c_int, V, c_size_t, c_int],
    "pressure_on_hybrid_levels": [V, V, c_int, V, c_int64, V, c_int, V, c_int, c_int, c_int, c_double, V, V, V, V, c_int, V],
    "hybrid_top_is_toa": [V, c_int64, c_double, c_double, V, V],
    "geopotential_on_hybrid_levels": [V, V, c_int, c_int64, V, V, V, c_int, c_int, c_double, V, V, V, c_int, V, V],
    "potential_temperature": [OP, OP, V, c_int64, V],
    "ept_wet_bulb": [OP, OP, OP, c_int, c_int, c_int, c_int, V, V, c_int64, V],
}

_BUF = (c_double * 64)()
P = ctypes.addressof(_BUF)  # a host buffer: no case below may hand it to a kernel
_ROWS = (c_int * 1)(0)
ROWS = ctypes.addressof(_ROWS)
S = Operand(None, 1.0)  # a broadcast scalar
NLEV = 3


class Api:
    def __init__(self, lib, dtype):
        self.so = ctypes.CDLL(os.path.join(ROOT, "earthkit-meteo_b200", "ek_thermo", lib))
        self.so.ek_thermo_last_error.restype = ctypes.c_char_p
        self.lean = lib == "libek_thermo.so"
        self.dtype = dtype
        self._keep = []

    def ptr(self, obj):
        """The address of a ctypes object that must outlive the call (None stays NULL)."""
        if obj is None:
            return None
        self._keep.append(obj)
        return ctypes.addressof(obj)

    def call(self, name, *args):
        fn = getattr(self.so, f"ek_thermo_{name}_{self.dtype}")
        fn.argtypes, fn.restype = ARGTYPES[name], c_int
        return fn(*args)

    def error(self):
        return self.so.ek_thermo_last_error().decode()

    def expect(self, want, name, *args):
        rc = self.call(name, *args)
        assert rc == want, (name, rc, self.error() if rc else "")
        if rc:
            assert self.error().startswith(name + ":"), (name, self.error())


@pytest.fixture(params=[(lib, dt) for lib in ("libek_thermo.so", "libek_thermo_exact.so") for dt in ("f64", "f32")],
                ids=lambda p: f"{p[0].split('.')[0]}-{p[1]}")
def api(request):
    path = os.path.join(ROOT, "earthkit-meteo_b200", "ek_thermo", request.param[0])
    assert os.path.exists(path), "run __graft_entry__.build() first"
    return Api(*request.param)


def table(api, slots, entry=None):
    """An outs table with `entry` (default: the host buffer) at the given slots, NULL elsewhere; None for slots=None."""
    if slots is None:
        return None
    t = (V * S_NSLOTS)()
    for k in slots:
        t[k] = P if entry is None else entry
    return api.ptr(t)


def batch_table(api, slots):
    """The outs of a one-segment batch call: one host array of segment pointers per requested slot."""
    return table(api, slots, None if slots is None else api.ptr((V * 1)(P)))


# (case, outs slots given (None: outs is NULL), out_mask, ept_method, expected code); n = 0 throughout
TABLE_CASES = [
    ("outs_null", None, 0x1, 0, EK_ERR_ARG),
    ("mask_empty", (0,), 0x0, 0, EK_ERR_ARG),
    ("mask_beyond_slots", tuple(range(S_NSLOTS)), 1 << S_NSLOTS, 0, EK_ERR_ARG),
    ("requested_slot_null", (0,), 0x3, 0, EK_ERR_ARG),
    ("bad_ept_with_slot_8", (8,), 1 << 8, 7, EK_ERR_ENUM),
    ("bad_ept_without_slots_8_9", (0,), 0x1, 7, EK_OK),
]
TABLE_IDS = [c[0] for c in TABLE_CASES]


def device_suite_call(api, name, outs, mask, ept):
    if name in ("suite_tqp", "suite_ttdp"):
        return (name, S, S, S, outs, mask, ept, 0, None)
    if name.endswith("_batch"):
        return (name, 1, None, None, None, None, None, outs, mask, ept, 0, None)
    if name == "suite_tq_hybrid":
        return (name, P, P, P, P, P, NLEV, 0, outs, mask, ept, None, None)
    return (name, P, P, P, P, P, P, NLEV, 0, outs, mask, ept, None, 0, 0.69, None, None, None, 0, None)


@pytest.mark.parametrize("case", TABLE_CASES, ids=TABLE_IDS)
@pytest.mark.parametrize("name", ["suite_tqp", "suite_ttdp", "suite_tqp_batch", "suite_ttdp_batch", "suite_tq_hybrid", "suite_tq_hybrid_geo"])
def test_device_suite_output_table_and_ept_method(api, name, case):
    _, slots, mask, ept, want = case
    outs = batch_table(api, slots) if name.endswith("_batch") else table(api, slots)
    api.expect(want, *device_suite_call(api, name, outs, mask, ept))


@pytest.mark.parametrize("case", TABLE_CASES, ids=TABLE_IDS)
@pytest.mark.parametrize("name", ["host_suite", "host_suite_tq_hybrid", "host_suite_tq_hybrid_geo"])
def test_host_suite_output_table_and_ept_method(api, name, case):
    """The host pipelines check the table up front; the ept method only where a chunk is launched, so n = 0 accepts any."""
    cname, slots, mask, ept, want = case
    if cname == "bad_ept_with_slot_8":
        want = EK_OK
    if cname == "mask_empty" and name == "host_suite_tq_hybrid_geo":
        want = EK_OK  # the thickness column is an output
    outs = table(api, slots)
    if name == "host_suite":
        args = (0, P, P, P, outs, mask, ept, 0, P, 1 << 20, 3)
    elif name == "host_suite_tq_hybrid":
        args = (P, P, P, P, P, NLEV, 0, outs, mask, ept, P, 1 << 20, 3)
    else:
        args = (P, P, P, P, P, P, NLEV, 0, outs, mask, ept, 0, 0.69, P, None, None, 0, P, 1 << 20, 3)
    api.expect(want, name, *args)


def test_hybrid_suites_accept_an_empty_mask_with_another_output(api):
    api.expect(EK_ERR_ARG, "suite_tq_hybrid", P, P, P, P, P, NLEV, 0, table(api, ()), 0, 0, None, None)
    api.expect(EK_OK, "suite_tq_hybrid", P, P, P, P, P, NLEV, 0, table(api, ()), 0, 0, P, None)  # p_out
    for col in range(3):
        cols = [None, None, None]
        cols[col] = P
        api.expect(EK_OK, "suite_tq_hybrid_geo", P, P, P, P, P, P, NLEV, 0, table(api, ()), 0, 0, None, 0, 0.69, *cols, 0, None)


def test_hybrid_launcher_checks(api):
    geo = lambda zs, z_out, height_out, mode: ("suite_tq_hybrid_geo", P, P, P, zs, P, P, NLEV, 0, table(api, (0,)), 1, 0, None, 0, 0.69,
                                               None, z_out, height_out, mode, None)
    api.expect(EK_ERR_ENUM, *geo(P, None, P, 6))
    api.expect(EK_ERR_ARG, *geo(None, P, None, 0))
    api.expect(EK_ERR_ARG, "pressure_on_hybrid_levels", P, P, 4, P, 0, ROWS, 1, ROWS, 1, 0, 0, 0.69, None, None, None, None, 0, None)
    api.expect(EK_ERR_ARG, "geopotential_on_hybrid_levels", P, P, NLEV, 0, P, P, P, NLEV + 1, 0, 0.69, None, None, P, 6, P, None)
    api.expect(EK_ERR_ARG, "hybrid_top_is_toa", P, 0, 0.0, 0.0, None, None)


def _cuda_available():
    import torch

    return torch.cuda.is_available()


@pytest.mark.skipif(_cuda_available(), reason="passes n > 0 with host buffers: only meaningful where no CUDA device exists")
def test_every_launcher_family_reports_a_missing_device(api):
    n = 16
    calls = [
        ("suite_tqp", S, S, S, table(api, (0,)), 1, 0, n, None),
        ("suite_tqp_batch", 1, None, None, None, None, None, batch_table(api, (0,)), 1, 0, n, None),
        ("potential_temperature", S, S, P, n, None),
        ("pressure_on_hybrid_levels", P, P, NLEV + 1, P, n, ROWS, 1, None, 0, 0, 0, 0.69, P, None, None, None, 0, None),
        ("hybrid_top_is_toa", P, n, 0.0, 0.0, P, None),
        ("geopotential_on_hybrid_levels", P, P, NLEV, n, P, P, P, NLEV + 1, 0, 0.69, None, None, None, 0, P, None),
        ("suite_tq_hybrid", P, P, P, P, P, NLEV, n, table(api, (0,)), 1, 0, None, None),
        ("suite_tq_hybrid_geo", P, P, P, P, P, P, NLEV, n, table(api, (0,)), 1, 0, None, 0, 0.69, None, None, None, 0, None),
    ]
    for name, *args in calls:
        api.expect(EK_ERR_ARG, name, *args)
        assert "no CUDA device is current" in api.error(), (name, api.error())
    # the bisection solver fills its node table with a kernel of its own before any device check: a failed launch (lean)
    rc = api.call("ept_wet_bulb", S, S, S, 0, 0, EK_TM_BISECT, 1, P, P, n, None)
    assert rc > 0 if api.lean else rc == EK_ERR_ARG, (rc, api.error())
