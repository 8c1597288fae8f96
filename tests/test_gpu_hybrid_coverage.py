"""The hybrid-level kernels at the launch shapes, level counts, dtypes and special values they meet in production, against the
long-double reference and per-point error bound of tests/test_hybrid_coverage_cpu.py:

- every column output and the pressure outputs on L137, a band of it and synthetic grids, both dtypes, aligned / odd / unaligned;
- bit-for-bit invariance under the level chunking of the suite and pressure kernels and under several column tiles per CTA;
- level counts whose coefficient copy needs more than 48 KiB of shared memory after a 137-level call, and the 200 KiB limit;
- NaN / inf / zero / negative inputs on model levels;
- the output dtype of every combination of argument dtypes.
"""
import gc
import os

import numpy as np
import pytest
import torch

import thermo_oracle as oracle
import vertical_oracle as voracle
from test_hybrid_coverage_cpu import (GEO_NAMES, LD, G, R_EARTH, column_reference, kernel_top_toa, l137, ld_pressure, ld_thickness,
                                      needs_ld, npl_for_rows_per_item, physical_columns, pressure_bounds, synthetic_ab, thickness_bound,
                                      tile_of, u_of, assert_within)
from test_hybrid_cpu import geo_call

pytestmark = [pytest.mark.gpu, needs_ld]
DEV = "cuda:0"
OUTS = ("full", "half", "delta", "alpha")
SUITE_ALL = ("theta", "es", "rh", "td", "tv", "w", "e", "thetav", "ept", "wbpt")
DEFAULT_CTAS_PER_SM = 16  # g_ctas_per_sm (csrc/ek_api.cu)


@pytest.fixture(autouse=True)
def restore_and_free():
    """Every test leaves the launch configuration and the fused-call threshold as the library defines them, and its device memory
    freed."""
    import ek_thermo
    from ek_thermo import fused

    saved = dict(fused.GEO_FUSED_MIN_COLUMNS)
    try:
        yield
    finally:
        ek_thermo.set_launch_config(0, DEFAULT_CTAS_PER_SM)
        fused.GEO_FUSED_MIN_COLUMNS.clear()
        fused.GEO_FUSED_MIN_COLUMNS.update(saved)
        gc.collect()
        torch.cuda.empty_cache()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(x, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(x if dtype is None else np.asarray(x).astype(dtype))).to(DEV)


def _shifted(x):
    """The same values in a contiguous view that starts one element into its allocation (not 16-byte aligned: scalar path)."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    return buf[1:].view(x.shape).copy_(x)


def _bits_equal(got, want, what):
    assert got.dtype == want.dtype and got.shape == want.shape, what
    assert torch.equal(torch.nan_to_num(got), torch.nan_to_num(want)), (what, float((got - want).abs().nan_to_num().max()))


GRIDS = {"L137": (l137, None), "L137-lower": (l137, 48), "L19-toa": (lambda: synthetic_ab(19, toa=True), None),
         "L60-top": (lambda: synthetic_ab(60, toa=False), None), "L91-toa": (lambda: synthetic_ab(91, toa=True), None)}


# ---- a. against the high-precision reference --------------------------------------------------------------------------------
@pytest.mark.parametrize("dname", ["float64", "float32"])
@pytest.mark.parametrize("grid", list(GRIDS))
def test_column_and_pressure_outputs_within_the_bound(grid, dname):
    """Six forms x both alpha_top, from_alpha_delta, and the four pressure outputs, within the per-point bound of the kernel dtype.
    float32: A / B given as float32 arrays (a float32 computation), the reference fed the same float32 values."""
    from ek_thermo import vertical

    dt = np.dtype(dname)
    make, nband = GRIDS[grid]
    A, B = (x.astype(dt) for x in make())
    u = u_of(dt)
    for npl, view in ((1024, False), (1001, False), (1024, True)):
        rng = np.random.default_rng(npl)
        sp = rng.uniform(5.0e4, 1.06e5, npl).astype(dt)
        zs = rng.uniform(-400.0, 4.0e4, npl).astype(dt)
        t, q = (x.astype(dt) for x in physical_columns(A.astype(np.float64), B.astype(np.float64), sp.astype(np.float64), seed=npl))
        if nband:
            t, q = t[-nband:], q[-nband:]
        d = {k: _dev(v) for k, v in (("t", t), ("q", q), ("sp", sp), ("zs", zs))}
        if view:
            d = {k: _shifted(v) for k, v in d.items()}
        what = f"{grid}/{dname}/{npl}{'/view' if view else ''}"
        for at in ("ifs", "arpege"):
            ref = column_reference(t, q, A, B, sp, zs, dt, at)
            for name in GEO_NAMES:
                got = geo_call(vertical, name, d["t"], d["q"], d["zs"], A, B, d["sp"], at)
                assert got.dtype == d["t"].dtype, (what, name)
                assert_within(got.cpu().numpy(), *ref[name], f"{what}/{at}/{name}")
        levels = None if not nband else list(range(len(A) - nband, len(A)))
        for at in ("ifs", "arpege"):
            P = ld_pressure(A, B, sp, at, top_toa=kernel_top_toa(A, B, sp, dt, len(A) - 1 - (nband or len(A) - 1)))
            pb = pressure_bounds(P, u)
            got = vertical.pressure_on_hybrid_levels(A, B, d["sp"], levels=levels, alpha_top=at, output=list(OUTS))
            for name, g in zip(OUTS, got):
                rows = slice(None) if not nband else slice(-nband, None)  # half rows of `levels` are the half levels of those numbers
                if nband and name in ("delta", "alpha"):  # the band's own top-of-atmosphere decision and top layer
                    Pb = ld_pressure(A, B, sp, at, len(A) - 1 - nband, kernel_top_toa(A, B, sp, dt, len(A) - 1 - nband))
                    assert_within(g.cpu().numpy(), Pb[name], pressure_bounds(Pb, u)[name], f"{what}/{at}/{name}")
                else:
                    assert_within(g.cpu().numpy(), P[name][rows], pb[name][rows], f"{what}/{at}/{name}")
            al, de = vertical.pressure_on_hybrid_levels(A, B, d["sp"], levels=levels, alpha_top=at, output=("alpha", "delta"))
            got = vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(d["t"], d["q"], al, de)
            assert got.dtype == d["t"].dtype  # float64 alpha / delta: computed in float64, rounded once to the field dtype
            given = {"alpha": al.cpu().numpy().astype(LD), "delta": de.cpu().numpy().astype(LD)}
            want = ld_thickness(t, q, given["alpha"], given["delta"])
            assert_within(got.cpu().numpy(), want, thickness_bound(t, q, given, u_of(np.float64)), f"{what}/{at}/from_alpha_delta", u_out=u)


# ---- b. launch-shape invariance -----------------------------------------------------------------------------------------------
def _tq_field(a, b, npl, seed):
    """t, q, sp of a plausible atmosphere on the levels of the device coefficients a / b, generated on the device (the largest
    fields have ~5 M columns)."""
    dtype = a.dtype
    g = torch.Generator(device=DEV).manual_seed(seed)
    sp = 5.0e4 + 5.6e4 * torch.rand((npl,), generator=g, device=DEV, dtype=dtype)
    pf = 0.5 * (a[:-1] + a[1:])[:, None] + 0.5 * (b[:-1] + b[1:])[:, None] * sp[None, :]
    noise = torch.rand(pf.shape, generator=g, device=DEV, dtype=dtype)
    t = (288.15 * (pf.clamp_min(1.0) / 101325.0) ** 0.19 + 30.0 * noise - 15.0).clamp(180.0, 320.0)
    del pf
    q = 1e-6 + 0.02 * torch.rand(t.shape, generator=g, device=DEV, dtype=dtype)
    return t, q, sp


def _slices(total, sizes):
    """Consecutive column slices of sizes `sizes` (cycled) covering [0, total)."""
    out, lo, k = [], 0, 0
    while lo < total:
        hi = min(total, lo + sizes[k % len(sizes)])
        out.append((lo, hi))
        lo, k = hi, k + 1
    return out


def _invariant(run, total, sizes, what):
    whole = run(0, total)
    for lo, hi in _slices(total, sizes):
        part = run(lo, hi)
        for name, v in part.items():
            _bits_equal(v, whole[name][..., lo:hi].contiguous(), f"{what}/{name}/[{lo}:{hi}]")
        del part
    return whole


@pytest.mark.parametrize("dname", ["float64", "float32"])
@pytest.mark.parametrize("nlev", [10, 11, 15])
def test_suite_and_pressure_are_invariant_under_level_chunking(nlev, dname):
    """suite_hybrid_kernel and hybrid_pressure_kernel split each tile's levels into work items of rows_per_item levels: 2, 4, 6, 8
    or the whole column by field size.  Groups of kHybLevels = 3 then leave remainders of 1 and 2 and start at levels that are not
    multiples of 3.  The whole field at the largest chunking is bit for bit the concatenation of column slices at the others."""
    from ek_thermo import fused, vertical

    dtype = getattr(torch, dname)
    ndt = np.dtype(dname)
    sms = _sms()
    A, B = synthetic_ab(nlev, toa=True)
    a, b = torch.tensor(A, dtype=dtype, device=DEV), torch.tensor(B, dtype=dtype, device=DEV)
    rpis = {10: (10, 2, 4, 6), 11: (12, 2, 4, 6), 15: (8, 2, 4, 6)}[nlev]
    if nlev == 15 and dname == "float32":
        pytest.skip("rows per item 8 is reached in float64")
    npls = {r: npl_for_rows_per_item(r, nlev, ndt, sms) for r in rpis}
    total = npls[rpis[0]]
    t, q, sp = _tq_field(a, b, total, seed=nlev)
    sizes = [npls[r] for r in rpis[1:]] + [tile_of(ndt) + 1]  # and an odd slice: scalar path

    def run_suite(lo, hi):
        tv, qv = t[:, lo:hi], q[:, lo:hi]
        return fused.suite_tq_hybrid(tv, qv, sp[lo:hi], a, b, outputs=SUITE_ALL, want_p=True)

    whole = _invariant(run_suite, total, sizes, f"suite/{nlev}/{dname}")
    cols = np.linspace(0, total - 1, 64).astype(np.int64)
    tc, qc, spc = (x[..., cols].cpu().numpy().astype(np.float64) for x in (t, q, sp))
    p_ref = voracle.pressure_on_hybrid_levels(A.astype(ndt), B.astype(ndt), spc.astype(ndt))
    np.testing.assert_allclose(whole["p"][:, cols].cpu().numpy(), p_ref, rtol=2e-6 if ndt == np.float32 else 1e-14)
    with np.errstate(all="ignore"):
        want = oracle.suite_tqp(tc.astype(ndt), qc.astype(ndt), p_ref)
    for name in SUITE_ALL:
        g = whole[name][:, cols].cpu().numpy().astype(np.float64)
        w = np.asarray(want[name]).astype(np.float64)
        bad = ~(np.abs(g - w) <= (2e-5 if ndt == np.float32 else 1e-12) * np.abs(w)) & ~(np.isnan(g) & np.isnan(w))
        assert bad.mean() <= (0.01 if ndt == np.float32 else 0.0), (name, np.nanmax(np.abs(g - w)))
    del whole
    gc.collect()
    torch.cuda.empty_cache()
    level_sets = {"all": None, "lower": list(range(nlev - 6, nlev + 1)), "reversed": list(range(nlev, 1, -1)), "one": [nlev // 2]}
    for lname, lv in level_sets.items():
        n_rows = nlev if lv is None else len(lv)
        big = max(range(2, n_rows + 3, 2), key=lambda r: npl_for_rows_per_item(r, n_rows, ndt, sms) or 0)
        tot = npl_for_rows_per_item(big, n_rows, ndt, sms)
        small = [npl_for_rows_per_item(r, n_rows, ndt, sms) for r in (2, 4, 6) if r < big]
        small = [s for s in small if s] + [tile_of(ndt) + 1]

        def run_p(lo, hi):
            res = vertical.pressure_on_hybrid_levels(a, b, sp[lo:hi], levels=lv, output=list(OUTS))
            return dict(zip(OUTS, res))

        whole = _invariant(run_p, min(tot, total), small, f"pressure/{nlev}/{dname}/{lname}")
        del whole
    del t, q, sp


@pytest.mark.parametrize("dname", ["float64", "float32"])
def test_column_and_geo_kernels_walk_several_tiles_per_cta(dname):
    """column_geopotential_kernel and suite_geo_kernel take column tiles in a grid-stride loop: with one CTA per SM each CTA walks
    several tiles, and every per-tile state (running sum, half-level pressure, zs, geom(zs)) must restart.  Bit for bit the default
    launch, where each CTA takes one tile."""
    import ek_thermo
    from ek_thermo import fused, vertical

    fused.GEO_FUSED_MIN_COLUMNS.update({"float64": 0, "float32": 0})
    dtype = getattr(torch, dname)
    A, B = l137()
    a, b = torch.tensor(A, dtype=dtype, device=DEV), torch.tensor(B, dtype=dtype, device=DEV)
    for npl in (400_001, 401_408):
        assert -(-npl // tile_of(np.dtype(dname))) > 2 * _sms()
        t, q, sp = _tq_field(a, b, npl, seed=npl)
        zs = (torch.rand(npl, device=DEV, dtype=dtype) - 0.01) * 4.0e4
        al, de = vertical.pressure_on_hybrid_levels(a, b, sp, output=("alpha", "delta"))
        res = {}
        for ctas in (DEFAULT_CTAS_PER_SM, 1):
            ek_thermo.set_launch_config(0, ctas)
            r = {name: geo_call(vertical, name, t, q, zs, a, b, sp, "ifs") for name in GEO_NAMES}
            r["from_alpha_delta"] = vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, al, de)
            for ht, hr in (("geometric", "ground"), ("geopotential", "sea")):
                f = fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "td", "thickness", "z", "height"), zs=zs, h_type=ht, h_reference=hr,
                                          want_p=True)
                r.update({f"fused/{ht}/{hr}/{k}": v for k, v in f.items()})
            res[ctas] = r
        for name, v in res[1].items():
            _bits_equal(v, res[DEFAULT_CTAS_PER_SM][name], f"{dname}/{npl}/{name}")
        del res, t, q, sp, zs, al, de


# ---- c. level counts beyond 48 KiB of shared memory ----------------------------------------------------------------------------
def _max_levels(dtype):
    """The largest level count whose coefficient copy fits the 200 KiB the launchers accept: behind the float64 lean-math tables
    (32 KiB) in the product library, alone in the exact twin and in float32."""
    from ek_thermo import _backend

    tables = 32768 if np.dtype(dtype) == np.float64 and "exact" not in os.path.basename(_backend.LIB_PATH) else 0
    return (200 * 1024 - tables) // (2 * np.dtype(dtype).itemsize) - 1


@pytest.mark.parametrize("dname,nlev", [("float64", 1100), ("float32", 6200)])
def test_large_level_counts_after_a_137_level_call(dname, nlev):
    """Each kernel instantiation is configured for its dynamic shared memory the first time it runs.  After a 137-level call (35 KiB
    of coefficients in float64), a call whose copy needs more than 48 KiB must raise the limit again, for every hybrid entry point:
    the column kernel under every MODE on the vector and the scalar path, suite_tq_hybrid with and without column outputs, and the
    host-array suite."""
    from ek_thermo import fused, vertical
    from ek_thermo.hostpipe import HostSuite

    fused.GEO_FUSED_MIN_COLUMNS.update({"float64": 0, "float32": 0})
    ndt = np.dtype(dname)
    dtype = getattr(torch, dname)
    u = u_of(ndt)
    hs = HostSuite(DEV, workspace_bytes=1 << 29, n_slots=2)
    for levels in (137, nlev):
        A, B = (x.astype(ndt) for x in synthetic_ab(levels, toa=True))
        a, b = _dev(A), _dev(B)
        for npl in (1024, 1001):  # the vector and the scalar path
            rng = np.random.default_rng(npl + levels)
            sp = rng.uniform(5.0e4, 1.06e5, npl).astype(ndt)
            zs = rng.uniform(-400.0, 4.0e4, npl).astype(ndt)
            t, q = (x.astype(ndt) for x in physical_columns(A.astype(np.float64), B.astype(np.float64), sp.astype(np.float64), seed=levels))
            d = {k: _dev(v) for k, v in (("t", t), ("q", q), ("sp", sp), ("zs", zs))}
            ref = column_reference(t, q, A, B, sp, zs, ndt) if levels == nlev else None
            what = f"{dname}/{levels}/{npl}"
            for name in GEO_NAMES:
                got = geo_call(vertical, name, d["t"], d["q"], d["zs"], a, b, d["sp"], "ifs")
                if ref:
                    assert_within(got.cpu().numpy(), *ref[name], f"{what}/{name}")
            suite = fused.suite_tq_hybrid(d["t"], d["q"], d["sp"], a, b, outputs=("theta", "rh"), want_p=True)
            mixed = fused.suite_tq_hybrid(d["t"], d["q"], d["sp"], a, b, outputs=("theta", "rh", "thickness", "z", "height"), zs=d["zs"], want_p=True)
            host = hs.suite_tq_hybrid(t, q, sp, A, B, outputs=("theta", "rh"))
            host_mixed = hs.suite_tq_hybrid(t, q, sp, A, B, outputs=("theta", "rh", "z"), zs=zs)
            if ref:
                p = vertical.pressure_on_hybrid_levels(a, b, d["sp"])
                two_step = fused.suite_tqp(d["t"], d["q"], p, outputs=("theta", "rh"))
                _bits_equal(suite["p"], p, f"{what}/p")
                _bits_equal(mixed["p"], p, f"{what}/mixed p")
                for name in ("theta", "rh"):
                    for label, r in (("suite", suite), ("mixed", mixed)):
                        torch.testing.assert_close(r[name], two_step[name], rtol=1e-5 if u > 1e-10 else 1e-14, atol=0, equal_nan=True,
                                                   msg=f"{what}/{label}/{name}")
                    _bits_equal(torch.from_numpy(host[name]), suite[name].cpu(), f"{what}/host/{name}")
                    _bits_equal(torch.from_numpy(host_mixed[name]), mixed[name].cpu(), f"{what}/host mixed/{name}")
                for col, name in (("thickness", "thickness"), ("z", "geopotential"), ("height", "h_geometric_ground")):
                    assert_within(mixed[col].cpu().numpy(), *ref[name], f"{what}/mixed/{col}")
                _bits_equal(torch.from_numpy(host_mixed["z"]), mixed["z"].cpu(), f"{what}/host mixed/z")
            del d, suite, mixed


@pytest.mark.parametrize("dname", ["float64", "float32"])
def test_level_count_limit_of_the_coefficient_copy(dname):
    """The largest level count whose coefficient copy fits 200 KiB runs; one level more raises ValueError before any kernel is
    launched (on a grid with B[0] = 0 the top-of-atmosphere decision needs no reduction kernel)."""
    import ek_thermo
    from ek_thermo import fused, vertical

    fused.GEO_FUSED_MIN_COLUMNS.update({"float64": 0, "float32": 0})
    ndt = np.dtype(dname)
    dtype = getattr(torch, dname)
    top = _max_levels(ndt)
    npl = 64
    for nlev, ok in ((top, True), (top + 1, False)):
        A, B = synthetic_ab(nlev, toa=True)
        a, b = torch.tensor(A, dtype=dtype, device=DEV), torch.tensor(B, dtype=dtype, device=DEV)
        t, q, sp = _tq_field(a, b, npl, seed=nlev)
        calls = {"thickness": lambda: vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp),
                 "suite": lambda: fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta",)),
                 "mixed": lambda: fused.suite_tq_hybrid(t, q, sp, a, b, outputs=("theta", "thickness"))}
        for label, call in calls.items():
            before = ek_thermo.launch_count()
            if ok:
                out = call()
                torch.cuda.synchronize()
                assert ek_thermo.launch_count() == before + 1, label
                th = out if isinstance(out, torch.Tensor) else out.get("thickness", out["theta"])
                assert bool(torch.isfinite(th).all()), label
            else:
                with pytest.raises(ValueError, match="too large"):
                    call()
                assert ek_thermo.launch_count() == before, label
        if ok:
            thick = vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp)
            tn, qn, spn = (x.cpu().numpy() for x in (t, q, sp))
            assert_within(thick.cpu().numpy(), *column_reference(tn, qn, A.astype(ndt), B.astype(ndt), spn, 0.0, ndt)["thickness"], f"{dname}/{nlev}")
        del t, q, sp


# ---- d. special values on model levels ---------------------------------------------------------------------------------------
def _special_field(partial_toa):
    """A 19-level grid whose top half level is 0.05 + 1e-6 sp (<= 0.1 Pa only for sp <= 5e4) and columns of special values."""
    A, B = synthetic_ab(19, toa=False)
    A[0], B[0] = 0.05, 1.0e-6
    npl = 2051
    rng = np.random.default_rng(77)
    sp = rng.uniform(5.5e4, 1.06e5, npl)
    zs = rng.uniform(-400.0, 4.0e4, npl)
    t, q = physical_columns(A, B, sp, seed=77)
    sp[:2] = [np.nan, np.inf]
    if partial_toa:  # the top half level <= 0.1 Pa at these points only
        sp[2:11] = [-np.inf, 0.0, -5.0e4, 1.0e-300, 4.0e4, 3.0e4, 5.0e4, 5.0e4 - 1e-6, -0.0]
    t[7, 10], q[3, 11], t[0, 12], q[18, 13] = np.nan, np.nan, np.nan, np.nan  # one level of some columns
    t[:, 14], q[:, 15] = np.nan, np.nan  # whole masked columns
    q[:, 16], q[:, 17], q[:, 18], t[:, 19], t[4, 20] = 0.0, 1.0, -0.01, 0.0, 0.0
    t[5, 21], q[9, 22] = np.inf, -np.inf
    zs[23:26] = [np.nan, np.inf, -np.inf]
    gr = float(G * R_EARTH)
    zs[26:40] = gr + np.linspace(-3.0e5, 3.0e5, 14)  # R - z / g passes near 0 within these columns
    return A, B, sp, zs, t, q


@pytest.mark.parametrize("partial_toa", [False, True])
def test_special_values_on_model_levels(partial_toa):
    """NaN / inf positions of every column output are the oracle's; finite values within the bound, or within 1e-12 of the oracle
    where the long-double reference and the float64 one part ways (overflow range).  Suite outputs equal suite_tqp on the
    materialised pressure under the special-value rule of the flat suites; the fused walk is bit for bit the separate launches."""
    from ek_thermo import fused, vertical

    A, B, sp, zs, t, q = _special_field(partial_toa)
    assert kernel_top_toa(A, B, sp, np.float64) == partial_toa
    d = {k: _dev(v) for k, v in (("t", t), ("q", q), ("sp", sp), ("zs", zs))}
    a, b = _dev(A), _dev(B)
    for at in ("ifs", "arpege"):
        ref = column_reference(t, q, A, B, sp, zs, np.float64, at)
        for name in GEO_NAMES:
            got = geo_call(vertical, name, d["t"], d["q"], d["zs"], a, b, d["sp"], at).cpu().numpy()
            with np.errstate(all="ignore"):
                want = geo_call(voracle, name, t, q, zs, A, B, sp, at)
            assert np.array_equal(np.isnan(got), np.isnan(want)), (at, name)
            assert np.array_equal(got[np.isinf(want)], want[np.isinf(want)]) and np.array_equal(np.isinf(got), np.isinf(want)), (at, name)
            fin = np.isfinite(want)
            with np.errstate(all="ignore"):
                near = np.abs(got - want) <= 1e-12 * np.abs(want)
            v, bd = ref[name]
            with np.errstate(all="ignore"):
                ok = np.abs(got.astype(LD) - v) <= bd
            assert bool((near | ok | ~fin).all()), (at, name, int((fin & ~near & ~ok).sum()))
    p = vertical.pressure_on_hybrid_levels(a, b, d["sp"])
    single = fused.suite_tqp(d["t"], d["q"], p, outputs=SUITE_ALL)
    fused.GEO_FUSED_MIN_COLUMNS.update({"float64": 0})
    for at in ("ifs", "arpege"):
        for ht, hr in (("geometric", "ground"), ("geometric", "sea"), ("geopotential", "sea"), ("geopotential", "ground")):
            got = fused.suite_tq_hybrid(d["t"], d["q"], d["sp"], a, b, outputs=SUITE_ALL + ("thickness", "z", "height"), zs=d["zs"], want_p=True,
                                        alpha_top=at, h_type=ht, h_reference=hr)
            _bits_equal(got["p"], p, "p")
            _bits_equal(got["thickness"], vertical.relative_geopotential_thickness_on_hybrid_levels(d["t"], d["q"], a, b, d["sp"], alpha_top=at), "thickness")
            _bits_equal(got["z"], vertical.geopotential_on_hybrid_levels(d["t"], d["q"], d["zs"], a, b, d["sp"], alpha_top=at), "z")
            _bits_equal(got["height"], vertical.height_on_hybrid_levels(d["t"], d["q"], d["zs"], a, b, d["sp"], alpha_top=at, h_type=ht, h_reference=hr),
                        f"height/{ht}/{hr}")
            plain = fused.suite_tq_hybrid(d["t"], d["q"], d["sp"], a, b, outputs=SUITE_ALL)
            for name in SUITE_ALL:
                for label, g in (("walk", got[name]), ("suite", plain[name])):
                    w = single[name]
                    assert torch.equal(torch.isnan(g), torch.isnan(w)), (label, name)
                    inf = torch.isinf(g) | torch.isinf(w)
                    assert torch.equal(g[inf], w[inf]), (label, name)
                    fin = torch.isfinite(g) & torch.isfinite(w)
                    tiny = (g[fin] - w[fin]).abs() <= 1e-300
                    rel = (g[fin] - w[fin]).abs() / w[fin].abs().clamp_min(1e-300)
                    assert bool(((rel <= 1e-10) | tiny).all()), (label, name, float(rel.max()))


# ---- e. output dtype ---------------------------------------------------------------------------------------------------------
def _np_dtype(x):
    return np.float64 if isinstance(x, (list, float)) else x.dtype


@pytest.mark.parametrize("ab", ["f32", "f64", "list"])
def test_output_dtype_equals_the_reference(ab):
    """Every combination of t / q / sp / zs dtypes (zs also a Python number) and A / B as float32, float64 or lists: the column
    functions (vertical_axis 0 and 1 on a square field) and pressure_on_hybrid_levels return the oracle's dtype, with values
    within the bound of the working dtype plus one rounding to the output dtype."""
    from ek_thermo import vertical

    nlev = 19
    A64, B64 = synthetic_ab(nlev, toa=True)
    A = {"f32": A64.astype(np.float32), "f64": A64, "list": A64.tolist()}[ab]
    B = {"f32": B64.astype(np.float32), "f64": B64, "list": B64.tolist()}[ab]
    rng = np.random.default_rng(5)
    sp0 = rng.uniform(5.0e4, 1.06e5, nlev)
    zs0 = rng.uniform(-400.0, 4.0e4, nlev)
    t0, q0 = physical_columns(A64, B64, sp0, seed=5)
    f = {"f32": np.float32, "f64": np.float64}
    for tk in f:
        for qk in f:
            for sk in f:
                for zk in ("f32", "f64", "number"):
                    t, q, sp = t0.astype(f[tk]), q0.astype(f[qk]), sp0.astype(f[sk])
                    zs = 250.0 if zk == "number" else zs0.astype(f[zk])
                    dz = zs if zk == "number" else _dev(zs)
                    dt_, dq, dsp = _dev(t), _dev(q), _dev(sp)
                    what = f"t{tk}/q{qk}/sp{sk}/zs{zk}/AB{ab}"
                    refs = {}
                    for name in GEO_NAMES:
                        # the working dtype of the call: zs is an argument of every function but the thickness; a number is weak
                        work = np.result_type(t, q, sp, _np_dtype(A), *(() if zk == "number" or name == "thickness" else (zs,)))
                        if work not in refs:
                            refs[work] = column_reference(t.astype(work), q.astype(work), np.asarray(A).astype(work), np.asarray(B).astype(work),
                                                          sp.astype(work), np.asarray(zs).astype(work), work)
                        ref = refs[work]
                        with np.errstate(all="ignore"):
                            want = geo_call(voracle, name, t, q, zs, A, B, sp, "ifs")
                        got = geo_call(vertical, name, dt_, dq, dz, A, B, dsp, "ifs")
                        assert str(got.dtype).split(".")[-1] == str(want.dtype), (what, name, got.dtype, want.dtype)
                        uo = u_of(want.dtype) if np.dtype(want.dtype).itemsize < np.dtype(work).itemsize else 0.0
                        assert_within(got.cpu().numpy(), *ref[name], f"{what}/{name}", u_out=uo)
                        # vertical_axis 1 on the square field: the reference's own (scrambled) numbers, in its dtype
                        g1 = geo_call_axis(vertical, name, dt_.T.contiguous(), dq.T.contiguous(), dz, A, B, dsp)
                        with np.errstate(all="ignore"):
                            w1 = geo_call_axis(voracle, name, np.ascontiguousarray(t.T), np.ascontiguousarray(q.T), zs, A, B, sp)
                        assert str(g1.dtype).split(".")[-1] == str(w1.dtype), (what, "axis1", name, g1.dtype, w1.dtype)
                        f32 = any(np.dtype(_np_dtype(x)) == np.float32 for x in (t, q, sp, A, zs))  # the oracle rounds to float32 somewhere
                        np.testing.assert_allclose(g1.cpu().numpy().astype(np.float64), w1.astype(np.float64), rtol=2e-5 if f32 else 1e-12,
                                                   atol=10.0 if f32 else 1e-7, err_msg=f"{what}/axis1/{name}")
                    al, de = voracle.pressure_on_hybrid_levels(A, B, sp, output=("alpha", "delta"))
                    for ak in f:
                        got = vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(dt_, dq, _dev(al, f[ak]), _dev(de, f[ak]))
                        want = voracle.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, al.astype(f[ak]), de.astype(f[ak]))
                        assert str(got.dtype).split(".")[-1] == str(want.dtype), (what, "from_alpha_delta", ak)
            got = vertical.pressure_on_hybrid_levels(A, B, _dev(sp0.astype(f[sk])), output=list(OUTS))
            want = voracle.pressure_on_hybrid_levels(A, B, sp0.astype(f[sk]), output=list(OUTS))
            for name, g, w in zip(OUTS, got, want):
                assert str(g.dtype).split(".")[-1] == str(w.dtype), (ab, sk, name)


def geo_call_axis(mod, name, t, q, zs, a, b, sp):
    if name == "thickness":
        return mod.relative_geopotential_thickness_on_hybrid_levels(t, q, a, b, sp, vertical_axis=1)
    if name == "geopotential":
        return mod.geopotential_on_hybrid_levels(t, q, zs, a, b, sp, vertical_axis=1)
    _, ht, hr = name.split("_")
    return mod.height_on_hybrid_levels(t, q, zs, a, b, sp, h_type=ht, h_reference=hr, vertical_axis=1)
