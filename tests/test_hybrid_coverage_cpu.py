"""A high-precision reference of the hybrid-level computations and the per-point error bar the GPU kernels are held to.

``np.longdouble`` (64-bit significand on x86-64) restatement of ``oracle/vertical_oracle.py`` in its operation order: half-level
pressure, full-level pressure, delta / alpha (both ``alpha_top`` values and the field-wide top-of-atmosphere rule), the geopotential
thickness and its six output forms.  The oracle itself cannot serve as this reference: it allocates alpha / delta with
``np.zeros(...)``, which truncates every intermediate to float64.

The tests here check the bar itself on the CPU: the float64 oracle lies within it, and plausible bugs do not.  They also hold the
synthetic A / B generator and the Python mirror of the hybrid kernels' launch arithmetic used by tests/test_gpu_hybrid_coverage.py.
"""
import numpy as np
import pytest

import vertical_oracle as voracle

LD = np.longdouble
LD_OK = np.finfo(LD).nmant >= 63
needs_ld = pytest.mark.skipif(not LD_OK, reason="np.longdouble has no 64-bit significand on this platform")

RD, RV = LD("287.0597"), LD("461.51")  # constants.py:22,26
G, R_EARTH = LD("9.80665"), LD(6371229)  # constants.py:53,57
PRESSURE_TOA = LD("0.1")  # V:667
GEO_NAMES = ("thickness", "geopotential", "h_geometric_sea", "h_geometric_ground", "h_geopotential_sea", "h_geopotential_ground")
U = {np.dtype(np.float64): 2.0 ** -53, np.dtype(np.float32): 2.0 ** -24}  # unit roundoff

# Constant of the error bound.  The bound terms below are first-order error propagations through the operation order of the
# kernels, each with the number of roundings it contains: the two half-level pressures carry <= 2u each and their difference
# turns that into <= (4r + 3)u relative on dp (r = p_top / dp); the ratio and the logarithm give delta an absolute error of
# ~5u, of which r * delta amplifies the (r-proportional) part, so alpha = 1 - r * delta is off by <= ~(9r + 8)u; R(q) * t
# carries ~4u including the rounded gas constants; each of the (nlev - k) additions of the running sum adds u of the partial sum.
# The largest coefficient is ~10.  The lean float64 logarithm is within a few ulp, the float32 intrinsics within ~2 ulp, which at
# most doubles the delta and alpha coefficients; 32 leaves the remaining factor for the second-order terms.
C_BOUND = 32.0


def u_of(dtype):
    return U[np.dtype(dtype)]


# ---- the reference --------------------------------------------------------------------------------------------------------
def _col(x, ndim):
    return x.reshape((-1,) + (1,) * ndim)


def kernel_top_toa(A, B, sp, dtype, band0=0):
    """V:678, the field-wide top-of-atmosphere decision, taken as the library takes it: in the working dtype."""
    dt = np.dtype(dtype).type
    a, b = dt(np.asarray(A, dtype=np.float64)[band0]), dt(np.asarray(B, dtype=np.float64)[band0])
    with np.errstate(all="ignore"):
        return bool(np.any(a + b * np.asarray(sp).astype(dt) <= dt(0.1)))


def ld_pressure(A, B, sp, alpha_top="ifs", band0=0, top_toa=None):
    """Half-level pressure of half levels ``band0..``, full-level pressure, delta and alpha of the full levels below (V:663-708),
    in long double.  ``top_toa``: the field-wide decision (``kernel_top_toa``), or None to take it here."""
    A, B = np.asarray(A, dtype=LD)[band0:], np.asarray(B, dtype=LD)[band0:]
    sp = np.asarray(sp, dtype=LD)
    with np.errstate(all="ignore"):
        ph = _col(A, sp.ndim) + _col(B, sp.ndim) * sp[np.newaxis]  # V:663
        full = ph[:-1] + LD("0.5") * (ph[1:] - ph[:-1])  # V:708
        delta = np.log(ph[1:] / ph[:-1])  # V:675
        alpha = LD(1) - ph[:-1] / (ph[1:] - ph[:-1]) * delta  # V:687-689
        if top_toa is None:
            top_toa = bool(np.any(ph[0] <= PRESSURE_TOA))
        if top_toa:
            delta[0] = np.log(ph[1] / PRESSURE_TOA)  # V:679
            alpha[0] = np.log(LD(2)) if alpha_top == "ifs" else LD(1)  # V:693
    return {"half": ph, "full": full, "delta": delta, "alpha": alpha, "top_toa": top_toa}


def ld_gas_t(t, q):
    """d = R(q) t (V:799-801, T:1706)."""
    t, q = np.asarray(t, dtype=LD), np.asarray(q, dtype=LD)
    with np.errstate(all="ignore"):
        return (RD + (RV - RD) * q) * t


def _below(x):
    """sum over j > k of x[j], for every level k (the running sum of the bottom-up walk)."""
    s = np.zeros_like(x)
    if x.shape[0] > 1:
        s[:-1] = np.flip(np.cumsum(np.flip(x[1:], axis=0), axis=0), axis=0)
    return s


def ld_thickness(t, q, alpha, delta):
    """V:804-809: dphi_k = sum_{j>k} d_j delta_j + d_k alpha_k."""
    d = ld_gas_t(t, q)
    with np.errstate(all="ignore"):
        return _below(d * delta) + d * alpha


def ld_geom(z):
    with np.errstate(all="ignore"):
        h = z / G
        return R_EARTH * h / (R_EARTH - h)  # V:500-501


def ld_form(name, dphi, zs):
    """The six output forms of a thickness (V:1064-1069, V:1163-1188)."""
    zs = np.asarray(zs, dtype=LD)
    with np.errstate(all="ignore"):
        if name == "thickness":
            return dphi
        if name == "geopotential":
            return dphi + zs
        if name == "h_geopotential_sea":
            return (dphi + zs) / G
        if name == "h_geopotential_ground":
            return dphi / G
        if name == "h_geometric_sea":
            return ld_geom(dphi + zs)
        return ld_geom(dphi + zs) - ld_geom(zs)


# ---- the per-point error bound ----------------------------------------------------------------------------------------------
def pressure_bounds(P, u, c=C_BOUND):
    """Per-point bounds of half / full / delta / alpha computed with unit roundoff u."""
    ph0, ph1 = P["half"][:-1], P["half"][1:]
    with np.errstate(all="ignore"):
        r = np.abs(ph0) / np.abs(ph1 - ph0)  # the layer's conditioning p_top / dp
        return {"half": c * u * np.abs(P["half"]), "full": c * u * (np.abs(ph0) + np.abs(ph1)),
                "delta": c * u * (1 + np.abs(P["delta"])), "alpha": c * u * (r + 1 + np.abs(P["alpha"]))}


def thickness_bound(t, q, P, u, c=C_BOUND):
    """Bound of the thickness: c u [ |d_k| (r_k + 1) + sum_{j>k} |d_j| (1 + |delta_j|) + (nlev - k) S_k ], S_k the sum of the
    magnitudes of the terms the running sum has added at level k (|dphi_k| when every term is positive).  Without "half" in P,
    alpha / delta are given inputs: only the products and the running sum round."""
    d = np.abs(ld_gas_t(t, q))
    with np.errstate(all="ignore"):
        a, de = np.abs(P["alpha"]), np.abs(P["delta"])
        if "half" in P:
            ph0, ph1 = P["half"][:-1], P["half"][1:]
            r = np.abs(ph0) / np.abs(ph1 - ph0)
            ad = d * (r + 1 + a) + _below(d * (1 + de))
        else:
            ad = d * a
        nlev = d.shape[0]
        steps = _col(np.arange(nlev, 0, -1).astype(LD), d.ndim - 1)  # additions up to level k: nlev - k
        s = _below(d * de) + d * a
        return c * u * (ad + steps * s)


def form_bound(name, dphi, zs, e_thick, u, c=C_BOUND):
    """Propagate the thickness bound through an output form, plus the roundings of the form itself."""
    zs = np.asarray(zs, dtype=LD)
    with np.errstate(all="ignore"):
        if name == "thickness":
            return e_thick
        z = dphi + zs if name != "h_geopotential_ground" else dphi
        e_z = e_thick + c * u * np.abs(z)
        if name == "geopotential":
            return e_z
        h = z / G
        e_h = e_z / G + c * u * np.abs(h)
        if name.startswith("h_geopotential"):
            return e_h
        cond = R_EARTH / np.abs(R_EARTH - h)  # d geom / dh = (R / (R - h))^2
        e_g = cond * cond * e_h + c * u * np.abs(ld_geom(z)) * (1 + cond)
        if name == "h_geometric_sea":
            return e_g
        hs = zs / G
        cs = R_EARTH / np.abs(R_EARTH - hs)
        return e_g + c * u * np.abs(ld_geom(zs)) * (1 + cs)


def column_reference(t, q, A, B, sp, zs, dtype, alpha_top="ifs", u=None):
    """{form: (long-double value, bound)} of the six forms for t / q on the bottom-most t.shape[0] levels of A / B, computed in
    `dtype` (u = its unit roundoff unless given).  The top-of-atmosphere decision is the library's, in `dtype`."""
    nlev = np.asarray(t).shape[0]
    band0 = len(A) - 1 - nlev
    u = u_of(dtype) if u is None else u
    P = ld_pressure(A, B, sp, alpha_top, band0, kernel_top_toa(A, B, sp, dtype, band0))
    dphi = ld_thickness(t, q, P["alpha"], P["delta"])
    e = thickness_bound(t, q, P, u)
    return {name: (ld_form(name, dphi, zs), form_bound(name, dphi, zs, e, u)) for name in GEO_NAMES}


def violations(got, want, bound, u_out=0.0):
    """Points where `got` is off `want` by more than `bound` (+ the rounding of the output to a coarser dtype): NaN / +-inf
    positions must agree exactly; returns the number of offending points."""
    g = np.asarray(got).astype(LD)
    w = np.asarray(want, dtype=LD)
    bad = np.isnan(g) != np.isnan(w)
    inf = np.isinf(g) | np.isinf(w)
    bad |= inf & ~(np.isnan(g) | np.isnan(w)) & (g != w)
    fin = np.isfinite(g) & np.isfinite(w)
    with np.errstate(all="ignore"):
        err = np.abs(g - w)
        lim = np.asarray(bound, dtype=LD) + LD(u_out) * np.abs(w)
        bad |= fin & ~(err <= lim)  # a NaN bound (NaN input) passes no finite point
    return int(np.count_nonzero(bad))


def assert_within(got, want, bound, what, u_out=0.0):
    n = violations(got, want, bound, u_out)
    if n:
        g, w = np.asarray(got).astype(LD), np.asarray(want, dtype=LD)
        with np.errstate(all="ignore"):
            ratio = np.abs(g - w) / (np.asarray(bound, dtype=LD) + LD(u_out) * np.abs(w))
        ratio = np.where(np.isfinite(g) & np.isfinite(w), ratio, 0)
        k = np.unravel_index(int(np.nanargmax(ratio)), ratio.shape)
        raise AssertionError(f"{what}: {n} points outside the bound; worst at {k}: got {g[k]!r} want {w[k]!r} error/bound {ratio[k]:.3g}")


# ---- synthetic grids ---------------------------------------------------------------------------------------------------
def synthetic_ab(nlev, toa=True, p0=1.0e5, p_top=20.0):
    """Monotone hybrid coefficients for any nlev: reference half-level pressure p_top + (p0 - p_top) eta^2, B = eta^3 (pure
    pressure at the top, sigma at the surface: A[-1] = 0, B[-1] = 1, as the IFS grids).  ``toa``: A[0] = B[0] = 0, the top
    half level is the top of the atmosphere; otherwise A[0] = p_top > 0.1 Pa.  Layers thin as 1 / nlev^2 at the top."""
    eta = np.arange(nlev + 1, dtype=np.float64) / nlev
    top = 0.0 if toa else float(p_top)
    b = eta ** 3
    a = top + (p0 - top) * eta ** 2 - b * p0
    a[-1], b[-1] = 0.0, 1.0
    return a, b


def l137():
    with np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "ifs_l137_ab.npz")) as z:
        return z["A"].astype(np.float64), z["B"].astype(np.float64)


def physical_columns(A, B, sp, nlev=None, seed=0):
    """t, q of a plausible atmosphere on the bottom-most `nlev` levels of A / B."""
    rng = np.random.default_rng(seed)
    nlev = len(A) - 1 if nlev is None else nlev
    pf = voracle.pressure_on_hybrid_levels(A, B, sp)[len(A) - 1 - nlev:]
    t = np.clip(288.15 * (np.maximum(pf, 1.0) / 101325.0) ** 0.19 + rng.uniform(-12, 12, pf.shape), 180.0, 320.0)
    q = rng.uniform(1e-6, 0.02, pf.shape)
    return t, q


# ---- mirror of the hybrid kernels' launch arithmetic (csrc/ek_hybrid.cu) -------------------------------------------------------
THREADS = 256  # kThreads (ek_thermo_kernels.cuh)
HYB_LEVELS = 3  # kHybLevels (ek_hybrid.cu): levels in flight per thread of suite_hybrid_kernel


def vec_of(dtype):
    return 16 // np.dtype(dtype).itemsize  # Vec16<T>::N


def tile_of(dtype):
    return THREADS * vec_of(dtype)  # points per work item of every hybrid kernel


def rows_per_item_for(ptiles, n_rows, sms):
    """Must follow rows_per_item_for() in csrc/ek_hybrid.cu: levels (output rows) per work item of suite_hybrid_kernel and
    hybrid_pressure_kernel.  Used only to choose field sizes that reach a given chunking."""
    want_items = (sms if sms > 0 else 148) * 64
    chunks = max(1, -(-want_items // ptiles))
    rpi = max(2, -(-n_rows // chunks))
    return rpi + (rpi & 1)


def npl_for_rows_per_item(rpi, n_rows, dtype, sms):
    """The smallest whole number of tiles whose field gets `rpi` rows per item, or None."""
    tile = tile_of(dtype)
    for chunks in range(1, n_rows + 1):
        if rows_per_item_for(-(-sms * 64 // chunks), n_rows, sms) == rpi:
            ptiles = -(-sms * 64 // chunks)
            while ptiles > 1 and rows_per_item_for(ptiles - 1, n_rows, sms) == rpi:
                ptiles -= 1
            return ptiles * tile
    return None


# ---- checks of the bar on the CPU ----------------------------------------------------------------------------------------
def _case(grid, npl=257, seed=1):
    A, B = grid
    rng = np.random.default_rng(seed)
    sp = rng.uniform(5.0e4, 1.06e5, npl)
    zs = rng.uniform(-400.0, 4.0e4, npl)
    t, q = physical_columns(A, B, sp, seed=seed)
    return A, B, sp, zs, t, q


GRIDS = {"L137": l137, "L19": lambda: synthetic_ab(19, toa=True), "L60": lambda: synthetic_ab(60, toa=False),
         "L91": lambda: synthetic_ab(91, toa=True)}


@pytest.mark.parametrize("nlev", [1, 2, 10, 11, 15, 19, 60, 91, 137, 1100, 6200, 10751, 10752, 25599, 25600])
@pytest.mark.parametrize("toa", [True, False])
def test_synthetic_grid_is_monotone(nlev, toa):
    a, b = synthetic_ab(nlev, toa=toa)
    assert a.shape == b.shape == (nlev + 1,) and a[-1] == 0.0 and b[-1] == 1.0 and b[0] == 0.0
    assert (a[0] == 0.0) if toa else (a[0] > 0.1)
    sp = np.linspace(5.0e4, 1.06e5, 57)
    for dt in (np.float64, np.float32):
        ph = a.astype(dt)[:, None] + b.astype(dt)[:, None] * sp.astype(dt)[None, :]
        assert np.all(np.diff(ph, axis=0) > 0), dt


@needs_ld
@pytest.mark.parametrize("grid", list(GRIDS))
@pytest.mark.parametrize("alpha_top", ["ifs", "arpege"])
def test_float64_oracle_is_within_the_bound(grid, alpha_top):
    A, B, sp, zs, t, q = _case(GRIDS[grid]())
    u = u_of(np.float64)
    ref = column_reference(t, q, A, B, sp, zs, np.float64, alpha_top)
    for name in GEO_NAMES:
        want, bound = ref[name]
        from test_hybrid_cpu import geo_call

        assert_within(geo_call(voracle, name, t, q, zs, A, B, sp, alpha_top), want, bound, f"{grid}/{alpha_top}/{name}")
    P = ld_pressure(A, B, sp, alpha_top)
    pb = pressure_bounds(P, u)
    got = voracle.pressure_on_hybrid_levels(A, B, sp, alpha_top=alpha_top, output=["full", "half", "delta", "alpha"])
    for name, g in zip(("full", "half", "delta", "alpha"), got):
        assert_within(g, P[name], pb[name], f"{grid}/{alpha_top}/{name}")
    # a lower band of the grid
    k = len(A) // 3
    ref = column_reference(t[k:], q[k:], A, B, sp, zs, np.float64, alpha_top)
    assert_within(voracle.relative_geopotential_thickness_on_hybrid_levels(t[k:], q[k:], A, B, sp, alpha_top=alpha_top), *ref["thickness"],
                  f"{grid}/band")


@needs_ld
def test_the_bound_explains_the_float32_and_float64_tolerances():
    """L137 bottom levels: the float32 bar is of the order of the 10 m2/s2 the reference's own float32 test allows, the float64 bar
    ~1e-9 relative (thin bottom layers: r = p / dp is large where alpha is small)."""
    A, B, sp, zs, t, q = _case(GRIDS["L137"]())
    for dt, lo, hi in ((np.float32, 1.0, 100.0), (np.float64, 1e-13, 1e-6)):
        want, bound = column_reference(t, q, A, B, sp, zs, dt)["thickness"]
        bottom = bound[-10:]
        if dt == np.float32:
            assert lo <= float(bottom.max()) <= hi, float(bottom.max())
        else:
            rel = float((bottom / np.abs(want[-10:])).max())
            assert lo <= rel <= hi, rel


def _thick_from_alpha(t, q, alpha, delta):
    return voracle.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, alpha, delta)


@needs_ld
@pytest.mark.parametrize("mutation", ["off_by_one", "arpege_for_ifs", "full_is_half_below", "float32_coefficients", "alpha_scaled"])
def test_plausible_bugs_violate_the_bound(mutation):
    A, B, sp, zs, t, q = _case(GRIDS["L137"]())  # A[0] = B[0] = 0: the top layer takes the alpha_top constant
    ref = column_reference(t, q, A, B, sp, zs, np.float64)
    P = ld_pressure(A, B, sp)
    pb = pressure_bounds(P, u_of(np.float64))
    al, de = voracle.pressure_on_hybrid_levels(A, B, sp, output=("alpha", "delta"))
    d = (voracle.RD + (voracle.RV - voracle.RD) * q) * t
    if mutation == "off_by_one":  # the running sum includes the current level's d * delta
        got, (want, bound) = _thick_from_alpha(t, q, al, de) + d * de, ref["thickness"]
    elif mutation == "arpege_for_ifs":
        got, (want, bound) = voracle.relative_geopotential_thickness_on_hybrid_levels(t, q, A, B, sp, alpha_top="arpege"), ref["thickness"]
    elif mutation == "full_is_half_below":
        got, want, bound = voracle.pressure_on_hybrid_levels(A, B, sp, output="half")[1:], P["full"], pb["full"]
    elif mutation == "float32_coefficients":
        a32, b32 = A.astype(np.float32).astype(np.float64), B.astype(np.float32).astype(np.float64)
        got, (want, bound) = voracle.relative_geopotential_thickness_on_hybrid_levels(t, q, a32, b32, sp), ref["thickness"]
    else:  # one level's alpha scaled by 1 + 1e-6
        al = al.copy()
        al[100] *= 1.0 + 1e-6
        got, (want, bound) = _thick_from_alpha(t, q, al, de), ref["thickness"]
    assert violations(got, want, bound) >= 1, mutation
    assert violations(_thick_from_alpha(t, q, *voracle.pressure_on_hybrid_levels(A, B, sp, output=("alpha", "delta"))), *ref["thickness"]) == 0


@needs_ld
def test_special_values_keep_their_positions_in_the_reference():
    """NaN / inf in the inputs give the oracle's NaN / inf positions in the long-double reference too."""
    A, B = synthetic_ab(19)
    sp = np.array([1.0e5, np.nan, np.inf, 0.0, -5.0e4, 7.0e4])
    zs = np.array([0.0, 10.0, np.nan, np.inf, -np.inf, 3.0e7])
    t, q = physical_columns(A, B, np.full(sp.shape, 1.0e5))
    t[5, 0] = np.nan
    with np.errstate(all="ignore"):
        for name in GEO_NAMES:
            from test_hybrid_cpu import geo_call

            w = geo_call(voracle, name, t, q, zs, A, B, sp, "ifs")
            want, bound = column_reference(t, q, A, B, sp, zs, np.float64)[name]
            assert violations(w, want, bound) == 0, name


def test_rows_per_item_mirror():
    """The mirror reaches every chunking the GPU tests ask for, on 148 SMs."""
    sms = 148
    assert rows_per_item_for(1, 137, sms) == 2 and rows_per_item_for(sms * 64, 11, sms) == 12
    for n_rows, rpis in ((10, (2, 4, 6, 10)), (11, (2, 4, 6, 12)), (15, (8,))):
        for rpi in rpis:
            npl = npl_for_rows_per_item(rpi, n_rows, np.float64, sms)
            assert npl is not None and npl % tile_of(np.float64) == 0
            assert rows_per_item_for(npl // tile_of(np.float64), n_rows, sms) == rpi, (n_rows, rpi)
    assert npl_for_rows_per_item(8, 10, np.float64, sms) is None
