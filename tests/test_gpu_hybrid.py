"""GPU parity of the hybrid-level kernels (SURVEY.md 8(f)-1) through the C ABI: against the oracle, the reference's
golden vectors, the live-reference fixtures, and -- for the fused kernel -- against suite_tqp fed with the
materialised pressure."""
import os

import numpy as np
import pytest
import torch

import thermo_oracle as oracle
import vertical_oracle as voracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OUTS = ("full", "half", "delta", "alpha")
LEVEL_SETS = {"all": None, "lower": list(range(90, 138)), "reversed": list(range(137, 90, -1)), "two": [2, 1], "top": [1]}


def _tol(name, f32):
    # delta/alpha difference quotients lose digits where ph1 - ph0 << ph0 (thin top layers); float32 as the reference's
    # own tolerance table (tests/vertical/test_array_vertical.py:196-203)
    if f32:
        return {"full": (2e-6, 0), "half": (2e-6, 0), "delta": (1e-4, 1e-6), "alpha": (2e-3, 1e-4)}[name]
    return {"full": (1e-14, 0), "half": (1e-14, 0), "delta": (1e-12, 0), "alpha": (1e-9, 1e-13)}[name]


def test_reference_golden_vectors(hyb):
    from ek_thermo import vertical

    sp = torch.from_numpy(hyb["gold/p_surf"]).to(DEV)
    res = vertical.pressure_on_hybrid_levels(hyb["gold/A"], hyb["gold/B"], sp, output=list(OUTS))
    for name, r in zip(OUTS, res):
        np.testing.assert_allclose(r.cpu().numpy(), hyb[f"gold/{name}"], rtol=1e-6, atol=1e-8, err_msg=name)  # the reference test's tolerance


@pytest.mark.parametrize("dname", ["float64", "float32"])
def test_live_reference_fixtures(hyb, dname):
    from ek_thermo import vertical

    dt = np.dtype(dname).type
    sp = torch.from_numpy(hyb["live/sp"].astype(dt)).to(DEV)
    for lname, lv in LEVEL_SETS.items():
        for at in ("ifs", "arpege"):
            res = vertical.pressure_on_hybrid_levels(hyb["gold/A"], hyb["gold/B"], sp, levels=lv, alpha_top=at, output=list(OUTS))
            for name, r in zip(OUTS, res):
                want = hyb[f"live/{dname}/{lname}/{at}/{name}"]
                rtol, atol = _tol(name, dname == "float32")
                np.testing.assert_allclose(r.cpu().numpy().astype(np.float64), want.astype(np.float64), rtol=rtol, atol=atol, err_msg=f"{lname}/{at}/{name}")


@pytest.mark.parametrize("shape", [(1001,), (37, 53), (6, 8, 16)])
def test_against_oracle_shapes_outputs_axis(hyb, shape):
    from ek_thermo import vertical

    rng = np.random.default_rng(5)
    sp = rng.uniform(4.8e4, 1.07e5, shape)
    d = torch.from_numpy(sp).to(DEV)
    a, b = hyb["gold/A"], hyb["gold/B"]
    for output in ("full", "half", ["delta", "alpha"], ["half", "full"], list(OUTS)):
        for va in (0, -1):
            got = vertical.pressure_on_hybrid_levels(a, b, d, output=output, vertical_axis=va)
            want = voracle.pressure_on_hybrid_levels(a, b, sp, output=output, vertical_axis=va)
            got = got if isinstance(got, tuple) else (got,)
            want = want if isinstance(want, tuple) else (want,)
            names = (output,) if isinstance(output, str) else output
            for name, g, w in zip(names, got, want):
                assert tuple(g.shape) == w.shape
                rtol, atol = _tol(name, False)
                np.testing.assert_allclose(g.cpu().numpy(), w, rtol=rtol, atol=atol, err_msg=f"{output}/{va}/{name}")
    # unaligned view of sp (scalar ld/st path) and an empty field
    got = vertical.pressure_on_hybrid_levels(a, b, d.reshape(-1)[1:], output="full")
    np.testing.assert_allclose(got.cpu().numpy(), voracle.pressure_on_hybrid_levels(a, b, sp.reshape(-1)[1:]), rtol=1e-14)
    assert vertical.pressure_on_hybrid_levels(a, b, d.reshape(-1)[:0]).shape == (137, 0)


def test_top_of_atmosphere_decision_is_field_wide():
    """V:678: if ANY point has p_half[top] <= 0.1 Pa, every point uses the TOA form for the top layer."""
    from ek_thermo import vertical

    a = np.array([0.05, 50.0, 500.0, 0.0])
    b = np.array([1.0e-6, 1.0e-3, 0.3, 1.0])  # top half-level pressure = 0.05 + 1e-6 * sp: <= 0.1 only for sp <= 5e4
    for sp in (np.array([6.0e4, 9.0e4, 1.0e5]), np.array([6.0e4, 4.0e4, 1.0e5])):
        for at in ("ifs", "arpege"):
            got = vertical.pressure_on_hybrid_levels(a, b, torch.from_numpy(sp).to(DEV), alpha_top=at, output=["delta", "alpha"])
            want = voracle.pressure_on_hybrid_levels(a, b, sp, alpha_top=at, output=["delta", "alpha"])
            for g, w in zip(got, want):
                np.testing.assert_allclose(g.cpu().numpy(), w, rtol=1e-12)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("npl", [4096 * 3, 10007])
def test_fused_suite_equals_materialised_pressure(hyb, dtype, npl):
    from ek_thermo import fused, vertical

    rng = np.random.default_rng(9)
    nlev = 137
    a, b = hyb["gold/A"], hyb["gold/B"]
    sp = rng.uniform(5.0e4, 1.05e5, npl).astype(dtype)
    p_ref = voracle.pressure_on_hybrid_levels(a.astype(dtype), b.astype(dtype), sp)
    t = np.clip(288.15 * (p_ref.astype(np.float64) / 101325.0) ** 0.19 + rng.uniform(-15, 15, (nlev, npl)), 180, 320).astype(dtype)
    q = rng.uniform(1e-6, 0.02, (nlev, npl)).astype(dtype)
    dt_, dq, dsp = (torch.from_numpy(x).to(DEV) for x in (t, q, sp))
    f32 = dtype == np.float32
    names = tuple(fused.SUITE_TQP_OUTPUTS)
    got = fused.suite_tq_hybrid(dt_, dq, dsp, a, b, outputs=names, want_p=True)
    p_dev = vertical.pressure_on_hybrid_levels(a.astype(dtype), b.astype(dtype), dsp)
    if f32:  # float64 coefficients next to a float32 sp promote the computation, as numpy does in the reference (V:630-663)
        assert vertical.pressure_on_hybrid_levels(a, b, dsp).dtype == torch.float64
        al = vertical.pressure_on_hybrid_levels(a.astype(dtype), b.astype(dtype), dsp, output="alpha")
        assert al.dtype == torch.float64  # alpha / delta are xp.zeros(...) arrays in the reference: always float64 (V:672,686)
    torch.testing.assert_close(got["p"], p_dev, rtol=0, atol=0)  # same formula, same kernel family: bit-identical
    np.testing.assert_allclose(got["p"].cpu().numpy(), p_ref, rtol=2e-6 if f32 else 1e-14)
    two_step = fused.suite_tqp(dt_, dq, p_dev, outputs=names)
    with np.errstate(all="ignore"):
        want = oracle.suite_tqp(t, q, p_ref)
    for name in names:
        torch.testing.assert_close(got[name], two_step[name], rtol=1e-5 if f32 else 1e-14, atol=0, equal_nan=True, msg=name)
        g = got[name].cpu().numpy().astype(np.float64)
        w = np.asarray(want[name]).astype(np.float64)
        bad = np.abs(g - w) > (2e-5 if f32 else 1e-12) * np.abs(w)
        assert bad.mean() <= (0.01 if f32 else 0.0), (name, np.abs(g - w).max())
    # default five outputs (compile-time mask) and preallocated buffers
    out = {"theta": torch.empty_like(dt_)}
    five = fused.suite_tq_hybrid(dt_, dq, dsp, a, b, out=out)
    assert five["theta"].data_ptr() == out["theta"].data_ptr() and set(five) == set(fused.DEFAULT_TQP)
    for name in fused.DEFAULT_TQP:
        torch.testing.assert_close(five[name], got[name], rtol=1e-5 if f32 else 1e-14, atol=0, equal_nan=True, msg=name)


# ---- SURVEY.md 8(f)-2: geopotential thickness / geopotential / height on hybrid levels --------------------------------
from test_hybrid_cpu import GEO_NAMES, geo_call  # noqa: E402


def test_geopotential_reference_golden_vectors(hyb):
    """The reference's own vectors and tolerances (tests/vertical/test_array_vertical.py:385-520)."""
    from ek_thermo import vertical

    d = lambda k: torch.from_numpy(hyb[k]).to(DEV)  # noqa: E731
    a, b = hyb["gold/A"], hyb["gold/B"]
    t, q, sp, z = d("gold/t"), d("gold/q"), d("gold/p_surf"), hyb["gold/z"]
    close = lambda got, want: np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-6, atol=1e-8)  # noqa: E731
    close(vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, d("gold/alpha"), d("gold/delta")), z)
    close(vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp), z)
    close(vertical.relative_geopotential_thickness_on_hybrid_levels(t[90:], q[90:], a, b, sp), z[90:])
    close(vertical.geopotential_on_hybrid_levels(t, q, torch.zeros(2, device=DEV, dtype=torch.float64), a, b, sp), z)
    a, b = hyb["goldh/A"], hyb["goldh/B"]
    t, q, sp, zs = d("goldh/t"), d("goldh/q"), d("goldh/p_surf"), d("goldh/z_surf")
    for ht in ("geometric", "geopotential"):
        for hr in ("sea", "ground"):
            close(vertical.height_on_hybrid_levels(t, q, zs, a, b, sp, h_type=ht, h_reference=hr), hyb[f"goldh/h_{ht}_{hr}"])


@pytest.mark.parametrize("dname", ["float64", "float32"])
def test_geopotential_live_reference_fixtures(hyb, dname):
    from ek_thermo import vertical

    dt = np.dtype(dname).type
    f32 = dname == "float32"
    a, b = hyb["gold/A"], hyb["gold/B"]
    sp, zs, t, q = (torch.from_numpy(hyb[k].astype(dt)).to(DEV) for k in ("geo/sp", "geo/zs", "geo/t", "geo/q"))
    for part, sl in (("all", slice(None)), ("lower", slice(90, None))):
        for at in ("ifs", "arpege"):
            for name in GEO_NAMES:
                got = geo_call(vertical, name, t[sl], q[sl], zs, a, b, sp, at).cpu().numpy().astype(np.float64)
                want = hyb[f"geo/{dname}/{part}/{at}/{name}"].astype(np.float64)
                # float32: the reference itself keeps alpha/delta in float64 there; its own test allows atol 10 (m2/s2)
                np.testing.assert_allclose(got, want, rtol=2e-5 if f32 else 1e-12, atol=10.0 if f32 else 1e-7, err_msg=f"{part}/{at}/{name}")
    al, de = vertical.pressure_on_hybrid_levels(a, b, sp, output=("alpha", "delta"))
    got = vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, al, de)
    np.testing.assert_allclose(got.cpu().numpy().astype(np.float64), hyb[f"geo/{dname}/from_alpha_delta"].astype(np.float64),
                               rtol=2e-5 if f32 else 1e-12, atol=10.0 if f32 else 1e-7)


@pytest.mark.parametrize("shape", [(3001,), (17, 20)])
def test_geopotential_against_oracle(hyb, shape):
    """Columns of any shape, odd sizes (scalar ld/st path), vertical_axis, and the thickness identities."""
    from ek_thermo import vertical

    rng = np.random.default_rng(31)
    a, b = hyb["gold/A"], hyb["gold/B"]
    sp = rng.uniform(5.0e4, 1.06e5, shape)
    zs = rng.uniform(-400.0, 4.0e4, shape)
    pf = voracle.pressure_on_hybrid_levels(a, b, sp)
    t = np.clip(288.15 * (pf / 101325.0) ** 0.19 + rng.uniform(-12, 12, pf.shape), 180.0, 320.0)
    q = rng.uniform(1e-6, 0.02, pf.shape)
    dsp, dzs, dt_, dq = (torch.from_numpy(x).to(DEV) for x in (sp, zs, t, q))
    for name in GEO_NAMES:
        got = geo_call(vertical, name, dt_, dq, dzs, a, b, dsp, "ifs")
        want = geo_call(voracle, name, t, q, zs, a, b, sp, "ifs")
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-12, atol=1e-7, err_msg=name)
    # identities: geopotential = thickness + zs; thickness decreases towards the surface and is positive
    thick = vertical.relative_geopotential_thickness_on_hybrid_levels(dt_, dq, a, b, dsp)
    geo = vertical.geopotential_on_hybrid_levels(dt_, dq, dzs, a, b, dsp)
    torch.testing.assert_close(geo, thick + dzs, rtol=1e-15, atol=1e-9)
    assert bool((thick[:-1] > thick[1:]).all()) and bool((thick[-1] > 0).all())


def test_vertical_axis_behaves_as_the_reference():
    """vertical_axis != 0 (SURVEY.md 7.3-H5, "replicate, don't fix"): the reference moves the alpha / delta it computed level-
    axis-first a second time (V:981-986), so only square fields pass numpy's broadcast check -- with scrambled alpha / delta --
    and every other shape raises ValueError.  The wrapper returns the reference's own numbers for the square field of the live
    fixture (tests/golden/ref_hybrid_axis.npz, generated from the unmodified reference), which are NOT the axis-0 answer, and
    raises ValueError otherwise; vertical axis 0 stays the consistent kernel path.  Also the two stand-alone height conversions."""
    import os

    from ek_thermo import vertical

    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_hybrid_axis.npz")) as z:
        fx = {k: z[k] for k in z.files}
    A, B = fx["A"], fx["B"]
    d = {k: torch.from_numpy(fx[k]).to(DEV) for k in ("sp", "zs", "t", "q")}
    t1, q1 = d["t"].T.contiguous(), d["q"].T.contiguous()  # [column, level]
    for axis in (1, -1):
        got = {"thickness": vertical.relative_geopotential_thickness_on_hybrid_levels(t1, q1, A, B, d["sp"], vertical_axis=axis),
               "geopotential": vertical.geopotential_on_hybrid_levels(t1, q1, d["zs"], A, B, d["sp"], vertical_axis=axis)}
        for ht in ("geometric", "geopotential"):
            for hr in ("sea", "ground"):
                got[f"h_{ht}_{hr}"] = vertical.height_on_hybrid_levels(t1, q1, d["zs"], A, B, d["sp"], h_type=ht, h_reference=hr, vertical_axis=axis)
        for name, g in got.items():
            np.testing.assert_allclose(g.cpu().numpy(), fx[f"axis{axis}/{name}"], rtol=1e-12, atol=1e-7, err_msg=f"axis {axis} {name}")
    consistent = vertical.relative_geopotential_thickness_on_hybrid_levels(d["t"], d["q"], A, B, d["sp"])
    np.testing.assert_allclose(consistent.cpu().numpy(), fx["axis0/thickness"], rtol=1e-12, atol=1e-7)
    assert not np.allclose(fx["axis1/thickness"].T, fx["axis0/thickness"], rtol=1e-3)  # the reference's axis-1 result is not the axis-0 one
    assert str(fx["nonsquare_error"]) == "ValueError"
    with pytest.raises(ValueError):
        vertical.relative_geopotential_thickness_on_hybrid_levels(t1[:5], q1[:5], A, B, d["sp"][:5], vertical_axis=1)
    with pytest.raises(ValueError):
        vertical.height_on_hybrid_levels(t1[:5], q1[:5], d["zs"][:5], A, B, d["sp"][:5], vertical_axis=-1)
    zz = torch.from_numpy(fx["conv/z"]).to(DEV)
    np.testing.assert_allclose(vertical.geopotential_height_from_geopotential(zz).cpu().numpy(), fx["conv/geopotential_height"], rtol=1e-15, equal_nan=True)
    np.testing.assert_allclose(vertical.geometric_height_from_geopotential(zz).cpu().numpy(), fx["conv/geometric_height"], rtol=1e-12, equal_nan=True)
