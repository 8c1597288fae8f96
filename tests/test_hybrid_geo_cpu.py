"""suite_tq_hybrid with column outputs, without a GPU: argument errors raised before any launch, the new C symbols, and the
SASS of the new kernel's out-of-line exact-recompute calls."""
import os
import shutil
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def no_launch(monkeypatch):
    """CPU tensors pass the device check, and any attempt to enter the C ABI fails the test."""
    import ek_thermo

    monkeypatch.setattr(ek_thermo._backend, "_check_device", lambda tensors: tensors[0].device)

    def boom(*a, **k):
        raise AssertionError("a kernel was launched")

    monkeypatch.setattr(ek_thermo._backend, "_call", boom)


def _args(nlev=3, npl=5, dtype=torch.float64):
    t = torch.ones(nlev, npl, dtype=dtype)
    return t, t.clone(), torch.full((npl,), 1.0e5, dtype=dtype), list(np.linspace(0.0, 100.0, nlev + 1)), list(np.linspace(0.0, 1.0, nlev + 1))


def test_argument_errors_before_any_launch(no_launch):
    from ek_thermo import fused

    t, q, sp, a, b = _args()
    zs = torch.zeros(5, dtype=torch.float64)
    with pytest.raises(ValueError, match="zs"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"))  # z needs zs
    for ht, hr in (("geometric", "ground"), ("geometric", "sea"), ("geopotential", "sea")):
        with pytest.raises(ValueError, match="zs"):
            fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "height"), h_type=ht, h_reference=hr)
    with pytest.raises(ValueError, match="h_reference"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("height",), zs=zs, h_reference="moon")
    with pytest.raises(ValueError, match="unknown suite output"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "geopotential"), zs=zs)
    with pytest.raises(ValueError, match="Unknown method"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"), zs=zs, alpha_top="nope")
    with pytest.raises(ValueError):
        fused.suite_tq_hybrid(t, q, sp, a[:3], b[:3], outputs=("theta", "z"), zs=zs)  # A / B need nlev + 1 values
    with pytest.raises(ValueError):
        fused.suite_tq_hybrid(t, q[:2], sp, a, b, outputs=("theta", "z"), zs=zs)  # t / q shapes
    with pytest.raises(ValueError):
        fused.suite_tq_hybrid(t, q, sp[:4], a, b, outputs=("theta", "z"), zs=zs)  # sp shape
    with pytest.raises(ValueError, match="zs must be"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"), zs=zs[:4])  # zs shape
    with pytest.raises(ValueError, match="zs must be"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"), zs=zs.float())  # zs dtype
    with pytest.raises(TypeError):
        fused.suite_tq_hybrid(t, q.float(), sp, a, b, outputs=("theta", "z"), zs=zs)  # one dtype for t, q, sp
    with pytest.raises(TypeError):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"), zs="0")
    with pytest.raises(ValueError, match="preallocated"):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"), zs=zs, out={"z": torch.empty(3, 4, dtype=torch.float64)})
    with pytest.raises(KeyError):
        fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "z"), zs=zs, ept_method="nope")
    # thickness and geopotential height above ground need no zs: such calls reach the launch
    for outputs, kw in ((("theta", "thickness"), {}), (("height",), {"h_type": "geopotential"})):
        with pytest.raises(AssertionError, match="launched"):
            fused.suite_tq_hybrid(t, q, sp, a, b, outputs=outputs, **kw)


def test_host_suite_argument_errors(monkeypatch):
    import ek_thermo
    from ek_thermo import hostpipe

    monkeypatch.setattr(ek_thermo._backend, "host_suite_tq_hybrid_geo", lambda *a, **k: pytest.fail("the pipeline was entered"))
    hs = object.__new__(hostpipe.HostSuite)  # no device workspace needed for the checks
    t = np.ones((3, 5))
    sp = np.full(5, 1.0e5)
    a, b = np.linspace(0.0, 100.0, 4), np.linspace(0.0, 1.0, 4)
    with pytest.raises(ValueError, match="zs"):
        hs.suite_tq_hybrid(t, t, sp, a, b, outputs=("theta", "z"))
    with pytest.raises(ValueError, match="h_reference"):
        hs.suite_tq_hybrid(t, t, sp, a, b, outputs=("height",), zs=np.zeros(5), h_reference="moon")
    with pytest.raises(ValueError, match="Unknown method"):
        hs.suite_tq_hybrid(t, t, sp, a, b, outputs=("z",), zs=np.zeros(5), alpha_top="nope")
    with pytest.raises(TypeError, match="zs must be"):
        hs.suite_tq_hybrid(t, t, sp, a, b, outputs=("z",), zs=np.zeros(4))
    with pytest.raises(TypeError, match="zs must be"):
        hs.suite_tq_hybrid(t, t, sp, a, b, outputs=("z",), zs=np.zeros(5, dtype=np.float32))


def test_top_is_toa_on_host_arrays():
    """The field-wide top-of-atmosphere decision (V:678) for host arrays, as the host pipeline takes it."""
    from ek_thermo.vertical import _top_is_toa

    a, b = np.array([0.05, 50.0]), np.array([1.0e-6, 1.0])
    assert _top_is_toa(a, b, 0, np.array([6.0e4, 9.0e4]), None, None) == 0
    assert _top_is_toa(a, b, 0, np.array([6.0e4, 4.0e4]), None, None) == 1
    assert _top_is_toa(np.array([0.05, 1.0]), np.array([0.0, 1.0]), 0, np.array([6.0e4]), None, None) == 1
    assert _top_is_toa(np.array([5.0, 1.0]), np.array([0.0, 1.0]), 0, np.array([6.0e4]), None, None) == 0


def test_new_symbols_in_both_libraries():
    import ctypes

    from ek_thermo import _backend

    assert _backend.version() >= 112
    here = os.path.dirname(_backend.LIB_PATH)
    for lib in ("libek_thermo.so", "libek_thermo_exact.so"):
        path = os.path.join(here, lib)
        if not os.path.exists(path):
            pytest.skip(f"{lib} not built here")
        so = ctypes.CDLL(path)
        for name in ("suite_tq_hybrid_geo", "host_suite_tq_hybrid_geo"):
            for sfx in ("f64", "f32"):
                assert hasattr(so, f"ek_thermo_{name}_{sfx}"), (lib, name, sfx)


def test_no_live_register_is_clobbered_across_the_cold_calls_of_the_geo_kernel():
    """The fused walk calls three out-of-line exact paths (the suite point, delta / alpha, the height form) from one level loop,
    run-time-mask instantiations included: the shape ptxas once miscompiled (DESIGN.md section 5)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_call_check

    path = os.path.join(ROOT, "earthkit-meteo_b200", "csrc", "build", "lean", "ek_hybrid.o")
    if not os.path.exists(path) or shutil.which("cuobjdump") is None:
        pytest.skip("no object files of the in-tree build (or no cuobjdump) here")
    calls, bad = sass_call_check.check(path, r"suite_geo_kernel")
    assert calls >= 20, calls
    assert bad == 0


def test_call_routing(monkeypatch):
    """No column output: the suite launch exactly as before; only column outputs: the existing geopotential launch, one per
    output; a mixed call: the fused kernel -- or, below GEO_FUSED_MIN_COLUMNS, the suite launch and the geopotential launches."""
    import ek_thermo
    from ek_thermo import fused

    monkeypatch.setattr(ek_thermo._backend, "_check_device", lambda tensors: tensors[0].device)
    calls = []
    monkeypatch.setattr(ek_thermo._backend, "call_raw", lambda symbol, *a: calls.append(symbol))
    t, q, sp, a, b = _args()
    zs = torch.zeros(5, dtype=torch.float64)

    def route(outputs, **kw):
        calls.clear()
        res = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=outputs, zs=zs, **kw)
        assert list(res) == list(outputs) + (["p"] if kw.get("want_p") else [])
        return list(calls)

    monkeypatch.setitem(fused.GEO_FUSED_MIN_COLUMNS, "float64", 0)
    assert route(("theta", "rh")) == ["suite_tq_hybrid"]
    assert route(()) == ["suite_tq_hybrid"]  # selects nothing: the C entry point reports it, as before
    assert route(("z", "height")) == ["geopotential_on_hybrid_levels"] * 2
    assert route(("theta", "z", "thickness")) == ["suite_tq_hybrid_geo"]
    assert route(("z",), want_p=True) == ["suite_tq_hybrid_geo"]
    monkeypatch.setitem(fused.GEO_FUSED_MIN_COLUMNS, "float64", 6)
    assert route(("theta", "z", "thickness")) == ["suite_tq_hybrid", "geopotential_on_hybrid_levels", "geopotential_on_hybrid_levels"]
    monkeypatch.setitem(fused.GEO_FUSED_MIN_COLUMNS, "float64", 5)
    assert route(("theta", "z")) == ["suite_tq_hybrid_geo"]
