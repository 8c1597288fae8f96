"""GPU parity of suite_tq_hybrid with column outputs (the suite and the geopotential of the same levels in one walk of the
columns): every output against the separate launches it replaces -- fused.suite_tq_hybrid without column outputs, and
vertical.pressure_on_hybrid_levels / relative_geopotential_thickness_on_hybrid_levels / geopotential_on_hybrid_levels /
height_on_hybrid_levels with A / B given as tensors of the field dtype -- and against the oracle."""
import numpy as np
import pytest
import torch

import vertical_oracle as voracle
from test_hybrid_cpu import geo_call

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SUITE5 = ("theta", "es", "rh", "td", "tv")
# GEO_NAMES form -> (column output, h_type, h_reference)
FORMS = {"thickness": ("thickness", "geometric", "ground"), "geopotential": ("z", "geometric", "ground"),
         "h_geometric_sea": ("height", "geometric", "sea"), "h_geometric_ground": ("height", "geometric", "ground"),
         "h_geopotential_sea": ("height", "geopotential", "sea"), "h_geopotential_ground": ("height", "geopotential", "ground")}


@pytest.fixture(autouse=True)
def fused_kernel_at_every_size(monkeypatch):
    """The test fields are small: run mixed calls through the fused kernel whatever their size (the small-field test sets its own
    threshold)."""
    from ek_thermo import fused

    for key in ("float64", "float32"):
        monkeypatch.setitem(fused.GEO_FUSED_MIN_COLUMNS, key, 0)


def _field(npl, dtype, seed=3, a=None, b=None, nlev=137, hyb=None):
    rng = np.random.default_rng(seed)
    if a is None:
        a, b = hyb["gold/A"][-nlev - 1:], hyb["gold/B"][-nlev - 1:]
    sp = rng.uniform(5.0e4, 1.05e5, npl)
    pf = voracle.pressure_on_hybrid_levels(a, b, sp)
    t = np.clip(288.15 * (pf / 101325.0) ** 0.19 + rng.uniform(-15, 15, pf.shape), 180, 320)
    q = rng.uniform(1e-6, 0.02, pf.shape)
    zs = rng.uniform(-400.0, 4.0e4, npl)
    d = {k: torch.from_numpy(v.astype(dtype)).to(DEV) for k, v in (("t", t), ("q", q), ("sp", sp), ("zs", zs))}
    d["A"], d["B"] = torch.tensor(a, dtype=d["t"].dtype, device=DEV), torch.tensor(b, dtype=d["t"].dtype, device=DEV)
    return d, {"t": t, "q": q, "sp": sp, "zs": zs, "A": a, "B": b}


def _suite_equal(got, want, f32):
    """The tolerances of test_fused_suite_equals_materialised_pressure, NaN positions identical."""
    torch.testing.assert_close(got, want, rtol=1e-5 if f32 else 1e-14, atol=0, equal_nan=True)


def _bits_equal(got, want, name):
    g, w = got.cpu().numpy(), want.cpu().numpy()
    assert np.array_equal(np.isnan(g), np.isnan(w)), name
    assert np.array_equal(g[~np.isnan(g)], w[~np.isnan(w)]), (name, np.nanmax(np.abs(g - w)))


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("npl", [4096 * 3, 10007])
def test_mixed_call_equals_separate_launches(hyb, dtype, npl):
    """Suite outputs equal the call without column outputs, p is bit-identical to pressure_on_hybrid_levels, and each of the
    six column forms x alpha_top is bit-identical to the vertical.* launch on the same tensors (same formulas, same order of
    the running sum)."""
    from ek_thermo import fused, vertical

    f32 = dtype == np.float32
    d, h = _field(npl, dtype, hyb=hyb)
    t, q, sp, zs, a, b = (d[k] for k in ("t", "q", "sp", "zs", "A", "B"))
    base = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=SUITE5)
    p = vertical.pressure_on_hybrid_levels(a, b, sp)
    for at in ("ifs", "arpege"):
        for form, (col, ht, hr) in FORMS.items():
            got = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=SUITE5 + (col,), want_p=True, zs=zs, alpha_top=at, h_type=ht, h_reference=hr)
            assert list(got) == list(SUITE5) + [col, "p"]
            for name in SUITE5:
                _suite_equal(got[name], base[name], f32)
            _bits_equal(got["p"], p, "p")
            _bits_equal(got[col], geo_call(vertical, form, t, q, zs, a, b, sp, at), f"{at}/{form}")
            # and the oracle, at the tolerances of the existing geopotential tests (float32: the float32 live-fixture bar)
            want = geo_call(voracle, form, h["t"], h["q"], h["zs"], h["A"], h["B"], h["sp"], at)
            np.testing.assert_allclose(got[col].cpu().numpy().astype(np.float64), want, rtol=2e-5 if f32 else 1e-12,
                                       atol=10.0 if f32 else 1e-7, err_msg=f"{at}/{form}")


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_every_ept_method_and_mask_with_z(hyb, dtype):
    """Slots 8 / 9 with z under every ept method; the static masks 0x1F and 0x31F and a run-time mask; all three column outputs."""
    from ek_thermo import fused, vertical

    f32 = dtype == np.float32
    d, _ = _field(8192, dtype, seed=4, hyb=hyb)
    t, q, sp, zs, a, b = (d[k] for k in ("t", "q", "sp", "zs", "A", "B"))
    z = vertical.geopotential_on_hybrid_levels(t, q, zs, a, b, sp)
    thick = vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp)
    height = vertical.height_on_hybrid_levels(t, q, zs, a, b, sp)
    sets = {"0x1F": SUITE5, "0x31F": SUITE5 + ("ept", "wbpt"), "run-time": ("rh", "w", "e", "thetav"), "ept": ("ept", "wbpt"),
            "all": tuple(fused.SUITE_TQP_OUTPUTS)}
    for em in ("ifs", "bolton35", "bolton39"):
        for label, names in sets.items():
            got = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=names + ("thickness", "z", "height"), zs=zs, ept_method=em)
            base = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=names, ept_method=em)
            for name in names:
                _suite_equal(got[name], base[name], f32)
            _bits_equal(got["z"], z, f"{em}/{label}/z")
            _bits_equal(got["thickness"], thick, f"{em}/{label}/thickness")
            _bits_equal(got["height"], height, f"{em}/{label}/height")


def test_scalar_path_edges_and_buffers(hyb):
    """npl not a multiple of the vector width and an unaligned view (scalar path), npl = 0, nlev = 1, zs as a Python number,
    preallocated outputs and want_p; the column-only call (existing geopotential launch)."""
    from ek_thermo import fused, vertical

    d, _ = _field(4097, np.float64, seed=6, hyb=hyb)
    t, q, sp, zs, a, b = (d[k] for k in ("t", "q", "sp", "zs", "A", "B"))

    def shifted(x):  # the same values in a view that starts one element (8 bytes) into its allocation
        buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=DEV)
        return buf[1:].view(x.shape).copy_(x)

    # npl = 4097 (not a multiple of the vector width), then 4096 columns in unaligned views: both the scalar path
    for tv, qv, spv, zsv in ((t, q, sp, zs), tuple(shifted(x) for x in (t[:, :4096], q[:, :4096], sp[:4096], zs[:4096]))):
        got = fused.suite_tq_hybrid(tv, qv, spv, a, b, outputs=("theta", "td", "z", "height"), zs=zsv, want_p=True, h_type="geopotential")
        _bits_equal(got["z"], vertical.geopotential_on_hybrid_levels(tv, qv, zsv, a, b, spv), "z")
        _bits_equal(got["height"], vertical.height_on_hybrid_levels(tv, qv, zsv, a, b, spv, h_type="geopotential"), "height")
        _bits_equal(got["p"], vertical.pressure_on_hybrid_levels(a, b, spv), "p")
        base = fused.suite_tq_hybrid(tv, qv, spv, a, b, outputs=("theta", "td"))
        for name in ("theta", "td"):
            _suite_equal(got[name], base[name], False)
    # zs as a Python number
    got = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("tv", "z", "height"), zs=250.0, h_reference="sea")
    _bits_equal(got["z"], vertical.geopotential_on_hybrid_levels(t, q, torch.full_like(sp, 250.0), a, b, sp), "z scalar zs")
    _bits_equal(got["height"], vertical.height_on_hybrid_levels(t, q, torch.full_like(sp, 250.0), a, b, sp, h_reference="sea"), "h scalar zs")
    # preallocated outputs, want_p, and column outputs that need no zs
    out = {"theta": torch.empty_like(t), "thickness": torch.empty_like(t), "p": torch.empty_like(t)}
    got = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "thickness", "height"), out=out, want_p=True, h_type="geopotential")
    assert all(got[k].data_ptr() == out[k].data_ptr() for k in out)
    _bits_equal(got["thickness"], vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp), "thickness")
    _bits_equal(got["height"], vertical.height_on_hybrid_levels(t, q, None, a, b, sp, h_type="geopotential"), "gh ground")
    # column outputs only: the existing geopotential launch, also into a preallocated buffer
    zo = torch.empty_like(t)
    got = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("z",), zs=zs, out={"z": zo})
    assert list(got) == ["z"] and got["z"].data_ptr() == zo.data_ptr()
    _bits_equal(got["z"], vertical.geopotential_on_hybrid_levels(t, q, zs, a, b, sp), "z only")
    # npl = 0 and nlev = 1
    e = fused.suite_tq_hybrid(t[:, :0], q[:, :0], sp[:0], a, b, outputs=("theta", "z"), zs=zs[:0])
    assert e["z"].shape == (137, 0) and e["theta"].shape == (137, 0)
    a1, b1 = torch.tensor([500.0, 0.0], dtype=torch.float64, device=DEV), torch.tensor([0.2, 1.0], dtype=torch.float64, device=DEV)
    got = fused.suite_tq_hybrid(t[-1:], q[-1:], sp, a1, b1, outputs=("es", "z", "height"), zs=zs, want_p=True)
    _bits_equal(got["z"], vertical.geopotential_on_hybrid_levels(t[-1:], q[-1:], zs, a1, b1, sp), "z nlev 1")
    _bits_equal(got["height"], vertical.height_on_hybrid_levels(t[-1:], q[-1:], zs, a1, b1, sp), "h nlev 1")
    _bits_equal(got["p"], vertical.pressure_on_hybrid_levels(a1, b1, sp), "p nlev 1")


def test_top_of_atmosphere_decision_is_field_wide():
    """B[0] != 0: whether the top layer takes the TOA form is decided by the data, for the whole field (V:678)."""
    from ek_thermo import fused, vertical

    a = torch.tensor([0.05, 50.0, 500.0, 0.0], dtype=torch.float64, device=DEV)
    b = torch.tensor([1.0e-6, 1.0e-3, 0.3, 1.0], dtype=torch.float64, device=DEV)  # top half level <= 0.1 Pa only for sp <= 5e4
    for spv in ([6.0e4, 9.0e4, 1.0e5, 8.0e4], [6.0e4, 4.0e4, 1.0e5, 8.0e4]):
        sp = torch.tensor(spv, dtype=torch.float64, device=DEV)
        t = torch.full((3, 4), 250.0, dtype=torch.float64, device=DEV)
        q = torch.full((3, 4), 1e-3, dtype=torch.float64, device=DEV)
        for at in ("ifs", "arpege"):
            got = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "thickness"), alpha_top=at)
            _bits_equal(got["thickness"], vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp, alpha_top=at), f"{spv}/{at}")
            want = voracle.relative_geopotential_thickness_on_hybrid_levels(t.cpu().numpy(), q.cpu().numpy(), a.cpu().numpy(), b.cpu().numpy(),
                                                                            sp.cpu().numpy(), alpha_top=at)
            np.testing.assert_allclose(got["thickness"].cpu().numpy(), want, rtol=1e-12)


def test_small_field_path_equals_fused(hyb, monkeypatch):
    """Below GEO_FUSED_MIN_COLUMNS a mixed call runs the two existing launches: the same numbers either way."""
    import ek_thermo
    from ek_thermo import fused

    d, _ = _field(2048, np.float64, seed=8, hyb=hyb)
    t, q, sp, zs, a, b = (d[k] for k in ("t", "q", "sp", "zs", "A", "B"))
    names = SUITE5 + ("z", "height")
    res = {}
    for thr, launches in ((0, 1), (1 << 40, 3)):  # the fused kernel; the suite and one geopotential launch per column output
        monkeypatch.setitem(fused.GEO_FUSED_MIN_COLUMNS, "float64", thr)
        before = ek_thermo.launch_count()
        res[thr] = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=names, zs=zs, want_p=True)
        assert ek_thermo.launch_count() - before == launches
    for name in names + ("p",):
        _bits_equal(res[0][name], res[1 << 40][name], name)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_host_suite_with_column_outputs_equals_device(hyb, dtype):
    """HostSuite.suite_tq_hybrid with z / height on numpy arrays is bit for bit the device call, also when a small workspace
    forces several column chunks; and thickness / geopotential height above ground without zs."""
    from ek_thermo import fused
    from ek_thermo.hostpipe import HostSuite

    d, h = _field(5000, dtype, seed=12, hyb=hyb)
    t, q, sp, zs, a, b = (h[k].astype(dtype) for k in ("t", "q", "sp", "zs", "A", "B"))
    names = ("theta", "rh", "ept", "z", "height")
    want = fused.suite_tq_hybrid(d["t"], d["q"], d["sp"], d["A"], d["B"], outputs=names, zs=d["zs"], h_reference="sea")
    esz = np.dtype(dtype).itemsize
    for ws in (1 << 26, 2 * 1024 * esz * (8 * 137 + 2) + 4096):  # one chunk; 1024-column chunks (5 of them) over 2 slots
        hs = HostSuite(DEV, workspace_bytes=ws, n_slots=2)
        got = hs.suite_tq_hybrid(t, q, sp, a, b, outputs=names, zs=zs, h_reference="sea")
        assert list(got) == list(names)
        for name in names:
            _bits_equal(torch.from_numpy(got[name]), want[name].cpu(), f"{ws}/{name}")
        got = hs.suite_tq_hybrid(t, q, sp, a, b, outputs=("thickness", "height"), h_type="geopotential")
        want2 = fused.suite_tq_hybrid(d["t"], d["q"], d["sp"], d["A"], d["B"], outputs=("thickness", "height"), h_type="geopotential")
        for name in ("thickness", "height"):
            _bits_equal(torch.from_numpy(got[name]), want2[name].cpu(), f"{ws}/{name} no zs")
