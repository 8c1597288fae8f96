"""Hybrid-level pressure (SURVEY.md 8(f)-1), CPU side: the oracle against the reference's golden vectors and the
live-reference fixtures; the per-point formulas the kernels use (g++ build) against the oracle; the wrapper's
argument errors."""
import ctypes
import os

import numpy as np
import pytest
import torch

import hostmath_backend
import vertical_oracle as voracle

LEVEL_SETS = {"all": None, "lower": list(range(90, 138)), "reversed": list(range(137, 90, -1)), "two": [2, 1], "top": [1]}
OUTS = ("full", "half", "delta", "alpha")


def test_oracle_matches_reference_golden_vectors(hyb):
    """tests/vertical/_hybrid_core_data.py, with the reference test's tolerances (atol 1e-8, rtol 1e-6; TT vertical :159-215)."""
    res = voracle.pressure_on_hybrid_levels(hyb["gold/A"], hyb["gold/B"], hyb["gold/p_surf"], output=list(OUTS))
    for name, r in zip(OUTS, res):
        np.testing.assert_allclose(r, hyb[f"gold/{name}"], rtol=1e-6, atol=1e-8, err_msg=name)


@pytest.mark.parametrize("dname", ["float64", "float32"])
def test_oracle_bit_identical_to_live_reference(hyb, dname):
    dt = np.dtype(dname).type
    a, b, sp = (hyb[k].astype(dt) for k in ("gold/A", "gold/B", "live/sp"))
    for lname, lv in LEVEL_SETS.items():
        for at in ("ifs", "arpege"):
            res = voracle.pressure_on_hybrid_levels(a, b, sp, levels=lv, alpha_top=at, output=list(OUTS))
            for name, r in zip(OUTS, res):
                want = hyb[f"live/{dname}/{lname}/{at}/{name}"]
                assert r.dtype == want.dtype and r.shape == want.shape
                np.testing.assert_allclose(r, want, rtol=8 * np.finfo(want.dtype).eps, atol=0, err_msg=f"{lname}/{at}/{name}")


def test_oracle_errors():
    a, b, sp = np.arange(4.0), np.arange(4.0), np.ones(3)
    for kw in (dict(output=[]), dict(output="x"), dict(alpha_top="x"), dict(levels=[4]), dict(levels=[0])):
        with pytest.raises(ValueError):
            voracle.pressure_on_hybrid_levels(a, b, sp, **kw)


def _host(op, ins, n_out, dtype, opt0=0, eps=0.0):
    lib = hostmath_backend.lib()
    n = ins[0].size
    arr = [np.ascontiguousarray(x.astype(dtype)) for x in ins]
    outs = [np.empty(n, dtype=dtype) for _ in range(n_out)]
    pin = (ctypes.c_void_p * len(arr))(*[x.ctypes.data for x in arr])
    sc = (ctypes.c_double * len(arr))()
    pout = (ctypes.c_void_p * n_out)(*[x.ctypes.data for x in outs])
    rc = lib.hostmath_run(op.encode(), int(dtype == np.float32), pin, sc, pout, n, opt0, 0, eps, 1, 0, 0)
    assert rc == 0
    return outs


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_per_point_formulas_match_oracle(hyb, dtype):
    """hyb_half / hyb_full / hyb_delta_alpha of ek_thermo_formulas.inc (what the kernels execute per point)."""
    a, b = hyb["gold/A"], hyb["gold/B"]
    sp = hyb["live/sp"]
    nlev = a.size - 1
    k = np.repeat(np.arange(nlev), sp.size)
    spp = np.tile(sp, nlev)
    full, half, delta, alpha = voracle.pressure_on_hybrid_levels(a.astype(dtype), b.astype(dtype), sp.astype(dtype), output=list(OUTS))
    rtol = 1e-13 if dtype == np.float64 else 2e-6
    got = _host("hyb_full", [a[k], b[k], a[k + 1], b[k + 1], spp], 1, dtype)[0]
    np.testing.assert_allclose(got, full.ravel(), rtol=rtol)
    ph0, ph1 = half[:-1].ravel(), half[1:].ravel()
    for top, at in ((0, 0.0), (1, np.log(2.0)), (1, 1.0)):
        d, al = _host("hyb_delta_alpha", [ph0, ph1], 2, dtype, opt0=top, eps=at)
        if top:
            np.testing.assert_allclose(d, np.log(ph1.astype(dtype) / dtype(0.1)), rtol=rtol * 10)
            np.testing.assert_allclose(al, at, rtol=rtol)
        else:
            sel = k >= 1  # the top layer of this coefficient set is the TOA special case in the oracle
            np.testing.assert_allclose(d[sel], delta.ravel()[sel], rtol=2e-5 if dtype == np.float32 else 1e-12)
            np.testing.assert_allclose(al[sel], alpha.ravel()[sel], rtol=2e-3 if dtype == np.float32 else 1e-9)


def test_wrapper_argument_errors(monkeypatch):
    import ek_thermo
    from ek_thermo import fused, vertical

    a = b = [0.0, 1.0, 2.0, 3.0]
    sp_cpu = torch.ones(5, dtype=torch.float64)
    with pytest.raises(ValueError):
        vertical.pressure_on_hybrid_levels(a, b, sp_cpu, output=[])
    with pytest.raises(ValueError):
        vertical.pressure_on_hybrid_levels(a, b, sp_cpu, output="nope")
    with pytest.raises(ValueError):
        vertical.pressure_on_hybrid_levels(a, b, sp_cpu, alpha_top="nope")
    with pytest.raises(TypeError):
        vertical.pressure_on_hybrid_levels(a, b, sp_cpu)  # CPU tensor: no CPU path
    with pytest.raises(TypeError):
        vertical.pressure_on_hybrid_levels(a, b, np.ones(5))
    monkeypatch.setattr(ek_thermo._backend, "_check_device", lambda tensors: tensors[0].device)
    with pytest.raises(ValueError):
        vertical.pressure_on_hybrid_levels(a, b, sp_cpu, levels=[4])
    with pytest.raises(ValueError):
        vertical.pressure_on_hybrid_levels(a, b, sp_cpu, levels=[0])
    t = torch.ones(3, 5, dtype=torch.float64)
    with pytest.raises(ValueError):
        fused.suite_tq_hybrid(t, t, sp_cpu, a[:3], b[:3])  # needs nlev + 1 coefficients
    with pytest.raises(ValueError):
        fused.suite_tq_hybrid(t, t, torch.ones(4, dtype=torch.float64), a, b)  # sp shape mismatch


# ---- SURVEY.md 8(f)-2: geopotential thickness / geopotential / height on hybrid levels --------------------------------
def test_geopotential_oracle_matches_reference_golden_vectors(hyb):
    """tests/vertical/test_array_vertical.py:385-520 (atol 1e-8, rtol 1e-6)."""
    a, b, sp, t, q, z = (hyb[f"gold/{k}"] for k in ("A", "B", "p_surf", "t", "q", "z"))
    np.testing.assert_allclose(voracle.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, hyb["gold/alpha"], hyb["gold/delta"]),
                               z, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(voracle.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp), z, rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(voracle.relative_geopotential_thickness_on_hybrid_levels(t[90:], q[90:], a, b, sp), z[90:], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(voracle.geopotential_on_hybrid_levels(t, q, np.zeros(2), a, b, sp), z, rtol=1e-6, atol=1e-8)
    a, b, sp, t, q, zs = (hyb[f"goldh/{k}"] for k in ("A", "B", "p_surf", "t", "q", "z_surf"))
    for ht in ("geometric", "geopotential"):
        for hr in ("sea", "ground"):
            got = voracle.height_on_hybrid_levels(t, q, zs, a, b, sp, h_type=ht, h_reference=hr)
            np.testing.assert_allclose(got, hyb[f"goldh/h_{ht}_{hr}"], rtol=1e-6, atol=1e-8, err_msg=f"{ht}/{hr}")
    with pytest.raises(ValueError):
        voracle.height_on_hybrid_levels(t, q, zs, a, b, sp, h_reference="moon")


GEO_NAMES = ("thickness", "geopotential", "h_geometric_sea", "h_geometric_ground", "h_geopotential_sea", "h_geopotential_ground")


def geo_call(mod, name, t, q, zs, a, b, sp, at):
    if name == "thickness":
        return mod.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp, alpha_top=at)
    if name == "geopotential":
        return mod.geopotential_on_hybrid_levels(t, q, zs, a, b, sp, alpha_top=at)
    _, ht, hr = name.split("_")
    return mod.height_on_hybrid_levels(t, q, zs, a, b, sp, alpha_top=at, h_type=ht, h_reference=hr)


@pytest.mark.parametrize("dname", ["float64", "float32"])
def test_geopotential_oracle_bit_identical_to_live_reference(hyb, dname):
    dt = np.dtype(dname).type
    a, b, sp, zs, t, q = (hyb[k].astype(dt) for k in ("gold/A", "gold/B", "geo/sp", "geo/zs", "geo/t", "geo/q"))
    for part, sl in (("all", slice(None)), ("lower", slice(90, None))):
        for at in ("ifs", "arpege"):
            for name in GEO_NAMES:
                got = geo_call(voracle, name, t[sl], q[sl], zs, a, b, sp, at)
                want = hyb[f"geo/{dname}/{part}/{at}/{name}"]
                assert got.dtype == want.dtype and got.shape == want.shape
                np.testing.assert_allclose(got, want, rtol=64 * np.finfo(want.dtype).eps, atol=0, err_msg=f"{part}/{at}/{name}")


def test_geopotential_wrapper_errors(monkeypatch):
    import ek_thermo
    from ek_thermo import vertical

    t = torch.ones(3, 5, dtype=torch.float64)
    a = b = [0.0, 1.0, 2.0, 3.0]
    with pytest.raises(ValueError):
        vertical.height_on_hybrid_levels(t, t, t[0], a, b, t[0], h_reference="moon")
    with pytest.raises(TypeError):
        vertical.relative_geopotential_thickness_on_hybrid_levels(t, t, a, b, t[0])  # CPU tensors: no CPU path
    monkeypatch.setattr(ek_thermo._backend, "_check_device", lambda tensors: tensors[0].device)
    with pytest.raises(ValueError):
        vertical.relative_geopotential_thickness_on_hybrid_levels(t, t, a[:3], b[:3], t[0])  # more data levels than A/B describe
    with pytest.raises(ValueError):
        vertical.relative_geopotential_thickness_on_hybrid_levels(t, t, a, b, t[0], alpha_top="nope")
    with pytest.raises(ValueError):
        vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, t, t[:2], t[:2])


def test_oracle_matches_reference_for_vertical_axis_not_zero():
    """The live-reference fixture of the vertical_axis != 0 behaviour (reference vertical.py:981-986; generated by
    tests/golden/make_golden.py --hybrid-axis): the oracle reproduces the reference's numbers bit for bit, raises where it
    raises, and PINNING.json records the comparison made at generation time."""
    import json

    here = os.path.dirname(os.path.abspath(__file__))
    with np.load(os.path.join(here, "golden", "ref_hybrid_axis.npz")) as z:
        fx = {k: z[k] for k in z.files}
    A, B, sp, zs = fx["A"], fx["B"], fx["sp"], fx["zs"]
    t1, q1 = np.ascontiguousarray(fx["t"].T), np.ascontiguousarray(fx["q"].T)
    for axis in (1, -1):
        np.testing.assert_array_equal(voracle.relative_geopotential_thickness_on_hybrid_levels(t1, q1, A, B, sp, vertical_axis=axis), fx[f"axis{axis}/thickness"])
        np.testing.assert_array_equal(voracle.geopotential_on_hybrid_levels(t1, q1, zs, A, B, sp, vertical_axis=axis), fx[f"axis{axis}/geopotential"])
        np.testing.assert_array_equal(voracle.height_on_hybrid_levels(t1, q1, zs, A, B, sp, vertical_axis=axis), fx[f"axis{axis}/h_geometric_ground"])
    with pytest.raises(ValueError):
        voracle.relative_geopotential_thickness_on_hybrid_levels(t1[:5], q1[:5], A, B, sp[:5], vertical_axis=1)
    with open(os.path.join(here, "golden", "PINNING.json")) as f:
        pin = json.load(f)["hybrid_axis"]
    assert pin["arrays_not_bit_identical_to_reference"] == 0 and pin["nonsquare_error"] == "ValueError"


def test_working_dtype_follows_numpy_promotion():
    """ek_thermo.vertical computes in the dtype numpy's promotion gives the reference (V:630-663): a float64 operand among
    float32 ones promotes, Python lists count as float64 arrays, Python numbers are weak, integers become float64."""
    from ek_thermo import vertical

    f32, f64 = torch.zeros(3, dtype=torch.float32), torch.zeros(3, dtype=torch.float64)
    wd = vertical._working_dtype
    assert wd(f32, f32) == torch.float32 and wd(f32, f64) == torch.float64 and wd(f64) == torch.float64
    assert wd(f32, np.zeros(3, dtype=np.float32)) == torch.float32 and wd(f32, np.zeros(3)) == torch.float64
    assert wd(f32, [0.0, 1.0]) == torch.float64  # xp.asarray([...]) is a float64 array
    assert wd(f32, 1.0, 2, None) == torch.float32  # Python scalars do not promote (numpy 2)
    assert wd(torch.zeros(3, dtype=torch.int32)) == torch.float64 and wd(torch.zeros(3, dtype=torch.float16)) == torch.float32
