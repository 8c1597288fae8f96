"""The (t, r, p) suite without a GPU: its composition of oracle functions (trp_parity.suite_trp), the g++ build of its functor
(mock device) against that composition through the package's host logic, the return codes of its C entry points, and the
out-of-line calls in its SASS."""
import ctypes
import os
import shutil
import subprocess
import sys
from ctypes import c_double, c_int, c_int64, c_uint32, c_void_p

import numpy as np
import pytest
import torch

import hostmath_backend
import test_launch_checks_cpu as lc
import thermo_oracle as oracle
from cases import T0, edge_inputs, random_inputs
from trp_parity import check_suite, suite_trp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "_hostmath", "hostmath_trp.cpp")
METHODS = ["ifs", "bolton35", "bolton39"]
# the compile-time output sets of suite() / suite_batch() in ek_ops_fused_impl.cuh (IFS only)
STATIC_MASKS = (0x1F, 0x05, 0x2C, 0x31F, 0x30D, 0x300)
STATIC_MASKS_BATCH = (0x1F, 0x05, 0x31F)


def _inputs(n, seed, dtype=np.float64):
    d = random_inputs(n, seed=seed)
    return [np.ascontiguousarray(d[k].astype(dtype)) for k in ("t", "r", "p")]


# ---- the oracle composition ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ept_method", METHODS)
def test_oracle_composition_is_the_reference_chain(ept_method):
    """Each output of the composition trp_parity.suite_trp is the named chain of pinned oracle functions, bit for bit, on random
    and edge inputs."""
    for t, r, p in (_inputs(2000, 3), [edge_inputs(n=2000, seed=4)[k] for k in ("t", "r", "p")]):
        with np.errstate(all="ignore"):
            got = suite_trp(t, r, p, ept_method=ept_method)
            q = oracle.specific_humidity_from_relative_humidity(t, r, p)
            want = {
                "theta": oracle.potential_temperature(t, p),
                "es": oracle.saturation_vapour_pressure(t),
                "td": oracle.dewpoint_from_relative_humidity(t, r),
                "q": q,
                "tv": oracle.virtual_temperature(t, q),
                "w": oracle.mixing_ratio_from_specific_humidity(q),
                "e": r * oracle.saturation_vapour_pressure(t) / 100.0,
                "thetav": oracle.virtual_potential_temperature(t, q, p),
                "ept": oracle.ept_from_specific_humidity(t, q, p, method=ept_method),
                "wbpt": oracle.wet_bulb_potential_temperature_from_specific_humidity(t, q, p, ept_method=ept_method, t_method="direct"),
            }
        assert list(got) == list(want)
        for name in want:
            assert np.array_equal(got[name], want[name], equal_nan=True), name
        assert np.array_equal(got["q"], oracle.specific_humidity_from_vapour_pressure(got["e"], p), equal_nan=True)  # e is T:662's


def test_parity_check_catches_the_rh_dewpoint_in_ept():
    """A suite that fed slot 2's dewpoint (over water, from r) into theta_e instead of the dewpoint of q (mixed phase) is wrong
    only on points below T0.  The parity check of the suite must reject it there and accept it above T0."""
    t, r, p = _inputs(20000, 8)
    with np.errstate(all="ignore"):
        want = suite_trp(t, r, p)
        td_r = oracle.dewpoint_from_relative_humidity(t, r)
        wrong = oracle._compute_ept("ifs", t=t, td=td_r, q=want["q"], p=p)
    cold, warm = t < T0 - 1.0, t > T0
    assert cold.sum() > 1000 and warm.sum() > 1000
    check_suite({"ept": want["ept"][warm]}, [x[warm] for x in (t, r, p)])
    check_suite({"ept": wrong[warm]}, [x[warm] for x in (t, r, p)])  # above T0 the two dewpoints agree
    with pytest.raises(AssertionError):
        check_suite({"ept": wrong[cold]}, [x[cold] for x in (t, r, p)])
    rel = np.abs(wrong[cold] - want["ept"][cold]) / want["ept"][cold]
    assert np.median(rel) > 1e-9


# ---- the functor on the mock device ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def trp_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostmath_trp") / "libek_hostmath_trp.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", SRC, "-o", so])
    lib = ctypes.CDLL(so)
    lib.hostmath_trp_run.argtypes = [c_int, ctypes.POINTER(c_void_p), ctypes.POINTER(c_double), ctypes.POINTER(c_void_p), c_int64, c_uint32, c_int,
                                     c_uint32]
    lib.hostmath_trp_run.restype = c_int
    return lib


def _val(x):
    return x.value if hasattr(x, "value") else x


@pytest.fixture()
def mock(monkeypatch, trp_lib):
    """The package's C calls go to the g++ build of the functors; suite_trp[_batch] to OpSuiteTRPm, picking the instantiation the
    library picks for the mask.  Returns the list of the compile-time mask (0: the run-time-mask instantiation) of every
    suite_trp "launch"."""
    from ek_thermo import _backend as b

    launches = []

    def run(dtype, operands, outs, n, mask, em, static_masks):
        static = mask if (em == 0 and mask in static_masks) else 0
        launches.append(static)
        ins = (c_void_p * 3)(*[o.ptr for o in operands])
        sc = (c_double * 3)(*[o.value for o in operands])
        o = (c_void_p * b.N_SUITE_SLOTS)(*outs)
        assert trp_lib.hostmath_trp_run(int(dtype == torch.float32), ins, sc, o, n, mask, em, static) == 0

    def fake_call(symbol, dtype, device, c_args):
        if symbol == "suite_trp":
            operands, (outs, mask, em, n) = c_args[:3], c_args[3:]
            mask = _val(mask)
            return run(dtype, operands, [outs[k] if (mask >> k) & 1 else None for k in range(b.N_SUITE_SLOTS)], _val(n), mask, _val(em), STATIC_MASKS)
        if symbol == "suite_trp_batch":
            n_seg, pa, pb, pc, scalars, level_scalars, out_tab, mask, em, n = c_args
            mask = _val(mask)
            for j in range(_val(n_seg)):
                ops = []
                for k, tab in enumerate((pa, pb, pc)):
                    tab = _val(tab)
                    if tab:
                        ops.append(b.ek_operand(ctypes.cast(tab, ctypes.POINTER(c_void_p))[j], 0.0))
                    else:
                        ops.append(b.ek_operand(None, level_scalars[j] if (k == 2 and level_scalars is not None) else scalars[k]))
                o = [ctypes.cast(out_tab[k], ctypes.POINTER(c_void_p))[j] if (mask >> k) & 1 else None for k in range(b.N_SUITE_SLOTS)]
                run(dtype, ops, o, _val(n), mask, _val(em), STATIC_MASKS_BATCH)
            return None
        return hostmath_backend.fake_call(symbol, dtype, device, c_args)

    monkeypatch.setattr(b, "_call", fake_call)
    monkeypatch.setattr(b, "_check_device", lambda tensors: tensors[0].device)
    return launches


def _mask(names):
    from ek_thermo import fused

    return sum(1 << fused.SUITE_TRP_OUTPUTS[k] for k in names)


def _output_sets(fused, ept_method):
    sets = [tuple(fused.SUITE_TRP_OUTPUTS), ("td",), ("q", "e"), ("es", "w", "thetav"), ("ept",), ("theta", "wbpt")]
    if ept_method == "ifs":  # every compile-time set
        names = list(fused.SUITE_TRP_OUTPUTS)
        sets += [tuple(n for n in names if (m >> fused.SUITE_TRP_OUTPUTS[n]) & 1) for m in STATIC_MASKS]
    return sets


@pytest.mark.parametrize("ept_method", METHODS)
@pytest.mark.parametrize("inputs", ["random", "edge"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_functor_matches_oracle(mock, dtype, inputs, ept_method):
    """Every output, the run-time-mask instantiation of each ept formulation and every compile-time set, against the oracle under
    the parity rule of tests/compare.py (NaN and inf positions identical in float64)."""
    from ek_thermo import fused

    with np.errstate(all="ignore"):
        src = random_inputs(3000, seed=17) if inputs == "random" else edge_inputs(n=1500, seed=29)
    args = [np.ascontiguousarray(src[k].astype(dtype)) for k in ("t", "r", "p")]
    targs = [torch.from_numpy(a.copy()) for a in args]
    seen = set()
    for outputs in _output_sets(fused, ept_method):
        del mock[:]
        got = fused.suite_trp(*targs, outputs=outputs, ept_method=ept_method)
        assert tuple(got) == outputs and len(mock) == 1
        seen.add(mock[0])
        check_suite({k: v.numpy() for k, v in got.items()}, args, ept_method, edge=(inputs == "edge"))
    assert seen == ({0, *STATIC_MASKS} if ept_method == "ifs" else {0})


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_functor_masks_and_instantiations_agree(mock, dtype):
    """A field's value does not depend on which other fields the call asks for, nor on which instantiation computes it."""
    from ek_thermo import fused

    args = [torch.from_numpy(a) for a in _inputs(2000, 31, dtype)]
    full = fused.suite_trp(*args, outputs=tuple(fused.SUITE_TRP_OUTPUTS))
    for outputs in _output_sets(fused, "ifs"):
        part = fused.suite_trp(*args, outputs=outputs)
        for name in outputs:
            assert torch.equal(torch.nan_to_num(part[name]), torch.nan_to_num(full[name])), (outputs, name)


def test_functor_scalar_pressure_and_batch(mock):
    """One pressure for the field (a pressure level), the batched form with per-field pressures or one scalar, and the errors of
    the Python side."""
    from ek_thermo import fused

    t, r, p = _inputs(4 * 500, 3)
    ts, rs, ps = ([torch.from_numpy(x[j * 500:(j + 1) * 500].copy()) for j in range(4)] for x in (t, r, p))
    got = fused.suite_trp(ts[0], rs[0], 85000.0, outputs=fused.SINGLE_PASS_TRP)
    check_suite({k: v.numpy() for k, v in got.items()}, [ts[0].numpy(), rs[0].numpy(), np.full(500, 85000.0)])
    levels = [100000.0, 85000.0, 50000, 3.0]
    for outputs, em in ((fused.DEFAULT_TRP, "ifs"), (fused.SINGLE_PASS_TRP, "ifs"), (("td", "ept", "wbpt"), "bolton39")):
        for pp in (ps, levels, 70000.0):
            del mock[:]
            got = fused.suite_trp_batch(ts, rs, pp, outputs=outputs, ept_method=em)
            assert len(got) == 4 and len(mock) == 4
            for j in range(4):
                pj = pp[j] if isinstance(pp, list) else pp
                pj = pj if isinstance(pj, torch.Tensor) else float(pj)
                want = fused.suite_trp(ts[j], rs[j], pj, outputs=outputs, ept_method=em)
                for name in outputs:
                    assert torch.equal(torch.nan_to_num(got[j][name]), torch.nan_to_num(want[name])), (j, name)
    pre = [{"q": torch.empty_like(ts[0])} for _ in range(4)]
    got = fused.suite_trp_batch(ts, rs, ps, outputs=("q", "td"), out=pre)
    assert all(got[j]["q"].data_ptr() == pre[j]["q"].data_ptr() for j in range(4))
    assert fused.suite_trp_batch([], [], []) == []
    with pytest.raises(ValueError):
        fused.suite_trp_batch(ts, rs, levels[:3])
    with pytest.raises(ValueError):
        fused.suite_trp(ts[0], rs[0], ps[0], outputs=("rh",))  # the (t, q, p) suite's name: not an output here
    with pytest.raises(KeyError):
        fused.suite_trp(ts[0], rs[0], ps[0], outputs=("ept",), ept_method="nope")
    with pytest.raises(KeyError):
        fused.suite_trp_batch(ts, rs, ps, outputs=("wbpt",), ept_method="nope")
    out = {"td": torch.empty(3, dtype=torch.float64)}
    with pytest.raises(ValueError):
        fused.suite_trp(ts[0], rs[0], ps[0], outputs=("td",), out=out)


def test_output_tables():
    from ek_thermo import fused

    assert fused.SUITE_TRP_OUTPUTS == {"theta": 0, "es": 1, "td": 2, "q": 3, "tv": 4, "w": 5, "e": 6, "thetav": 7, "ept": 8, "wbpt": 9}
    assert _mask(fused.DEFAULT_TRP) == 0x1F and _mask(fused.SINGLE_PASS_TRP) == 0x30D


# ---- the C entry points ----------------------------------------------------------------------------------------------------------
V, OP = c_void_p, lc.Operand
ARGTYPES = {
    "suite_trp": [OP, OP, OP, V, c_uint32, c_int, c_int64, V],
    "suite_trp_batch": [c_int, V, V, V, V, V, V, c_uint32, c_int, c_int64, V],
}


class TrpApi(lc.Api):
    def call(self, name, *args):
        fn = getattr(self.so, f"ek_thermo_{name}_{self.dtype}")
        fn.argtypes, fn.restype = ARGTYPES.get(name, lc.ARGTYPES.get(name)), c_int
        return fn(*args)


@pytest.fixture(params=[(lib, dt) for lib in ("libek_thermo.so", "libek_thermo_exact.so") for dt in ("f64", "f32")],
                ids=lambda p: f"{p[0].split('.')[0]}-{p[1]}")
def api(request):
    assert os.path.exists(os.path.join(ROOT, "earthkit-meteo_b200", "ek_thermo", request.param[0])), "run __graft_entry__.build() first"
    return TrpApi(*request.param)


@pytest.mark.parametrize("case", lc.TABLE_CASES, ids=lc.TABLE_IDS)
@pytest.mark.parametrize("name", ["suite_trp", "suite_trp_batch"])
def test_entry_point_output_table_and_ept_method(api, name, case):
    """Bad output tables, empty masks and a bad ept method with slot 8 / 9; n = 0 throughout, so nothing can launch."""
    _, slots, mask, ept, want = case
    if name == "suite_trp":
        api.expect(want, name, lc.S, lc.S, lc.S, lc.table(api, slots), mask, ept, 0, None)
    else:
        api.expect(want, name, 1, None, None, None, None, None, lc.batch_table(api, slots), mask, ept, 0, None)


def test_entry_point_bad_ept_with_slot_9(api):
    api.expect(lc.EK_ERR_ENUM, "suite_trp", lc.S, lc.S, lc.S, lc.table(api, (9,)), 1 << 9, -1, 0, None)
    api.expect(lc.EK_ERR_ENUM, "suite_trp_batch", 1, None, None, None, None, None, lc.batch_table(api, (9,)), 1 << 9, 3, 0, None)


@pytest.mark.parametrize("case", lc.TABLE_CASES, ids=lc.TABLE_IDS)
def test_host_suite_kind_2(api, case):
    """kind 2 is the (t, r, p) suite: the table is checked up front, the ept method only where a chunk is launched (n = 0 here)."""
    cname, slots, mask, ept, want = case
    if cname == "bad_ept_with_slot_8":
        want = lc.EK_OK
    api.expect(want, "host_suite", 2, lc.P, lc.P, lc.P, lc.table(api, slots), mask, ept, 0, lc.P, 1 << 20, 3)


@pytest.mark.parametrize("kind", [3, -1])
def test_host_suite_other_kinds_are_rejected(api, kind):
    api.expect(lc.EK_ERR_ENUM, "host_suite", kind, lc.P, lc.P, lc.P, lc.table(api, (0,)), 1, 0, 0, lc.P, 1 << 20, 3)


@pytest.mark.skipif(torch.cuda.is_available(), reason="passes n > 0 with host buffers: only meaningful where no CUDA device exists")
def test_entry_points_report_a_missing_device(api):
    api.expect(lc.EK_ERR_ARG, "suite_trp", lc.S, lc.S, lc.S, lc.table(api, (0, 2)), 0x5, 0, 16, None)
    assert "no CUDA device is current" in api.error()
    api.expect(lc.EK_ERR_ARG, "suite_trp_batch", 1, None, None, None, None, None, lc.batch_table(api, (3,)), 0x8, 0, 16, None)
    assert "no CUDA device is current" in api.error()


# ---- SASS ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("build", ["lean", "exact"])
def test_sass_call_sites(build):
    """No register that a kernel keeps live across an out-of-line call of ek_ops_fused_trp.o is written by the callee chain
    (tools/sass_call_check.py; DESIGN.md section 5).  Needs the object files of the in-tree build and cuobjdump."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_call_check

    path = os.path.join(ROOT, "earthkit-meteo_b200", "csrc", "build", build, "ek_ops_fused_trp.o")
    if not os.path.exists(path) or shutil.which("cuobjdump") is None:
        pytest.skip("no object files of the in-tree build (or no cuobjdump) here")
    calls, bad = sass_call_check.check(path, None)
    assert bad == 0
    if build == "lean":  # the exact-recompute calls of the float64 kernels
        assert calls > 50, calls
