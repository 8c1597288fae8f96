"""Generate the committed golden fixtures from the LIVE reference (build container only).

Run:  python tests/golden/make_golden.py

Needs /root/reference (read-only) and the numpy stand-in for earthkit-utils under
oracle/refshim.  Produces, next to this file:

* ref_csv.npz    -- the reference's own golden CSVs (reference tests/data/*.csv, consumed by
                    reference tests/thermo/test_thermo.py:171-186,206-331,346-356,706-849),
                    re-packed column by column as float64 (keys "<file stem>/<column>").
* ref_live.npz   -- inputs and outputs of the unmodified reference functions for every Case of
                    tests/cases.py on four input sets (seeded random, edge values, the reference's
                    t_hum_p_data.csv grid, the moist-adiabat grid), float64 and float32.  The outputs on the
                    seeded random set are in ref_live_rand_float64.npz and ref_live_rand_float32.npz.
* ref_hybrid.npz -- hybrid-level pressure: the reference's golden vectors (tests/vertical/_hybrid_core_data.py) and live
                    outputs of earthkit.meteo.vertical.pressure_on_hybrid_levels (SURVEY.md 8(f)-1); the live
                    geopotential outputs (SURVEY.md 8(f)-2) are in ref_hybrid_geo.npz.
  A set split over several files is merged back by tests/conftest.py; the split keeps every file under 1 MB.
* ref_wind.npz   -- live outputs of the reference's elementwise wind functions (SURVEY.md 8(f)-3).
* ifs_l137_ab.npz -- the IFS L137 A/B half-level coefficients from the reference's conf JSON (bench input layout).
* PINNING.json   -- oracle-vs-reference comparison made at generation time (max relative
                    difference and NaN-position mismatches per case).

Nothing in the GPU tests, smoke() or bench.py reads /root/reference; they read these files.
"""
from __future__ import annotations

import json
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"

sys.path.insert(0, os.path.join(ROOT, "oracle", "refshim"))
sys.path.insert(0, os.path.join(REF, "src"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from earthkit.meteo import thermo as ref_thermo  # noqa: E402  (the live reference)

import thermo_oracle as oracle  # noqa: E402
from cases import CASES, edge_inputs, random_inputs  # noqa: E402

warnings.simplefilter("ignore")


def load_csv(name):
    d = np.genfromtxt(os.path.join(REF, "tests", "data", name), delimiter=",", names=True)
    return {k: np.asarray(d[k], dtype=np.float64) for k in d.dtype.names}


def pack_csvs():
    out = {}
    for name in sorted(os.listdir(os.path.join(REF, "tests", "data"))):
        if name.endswith(".csv"):
            for k, v in load_csv(name).items():
                out[f"{name[:-4]}/{k}"] = v
    return out


def input_sets():
    csv = load_csv("t_hum_p_data.csv")
    ma = load_csv("t_on_most_adiabat.csv")
    n = csv["t"].size
    rng = np.random.default_rng(3)
    # the reference grid only carries t, td, r, q, p -- fill the other fields deterministically
    grid = dict(t=csv["t"], td=csv["td"], r=csv["r"], q=csv["q"], p=csv["p"])
    grid["tc"] = grid["t"] - 273.16
    grid["w"] = grid["q"] / (1 - grid["q"])
    grid["e"] = grid["p"] * grid["q"] / (0.621981 + 0.378019 * grid["q"])
    grid["es"] = grid["e"] * 100.0 / grid["r"]
    grid["ept"] = grid["t"] * (1e5 / grid["p"]) ** 0.285691 * np.exp(2488.88 * grid["q"] / grid["td"])
    grid["th"] = grid["t"] * (1e5 / grid["p"]) ** 0.285691
    grid["t_def"] = rng.uniform(250.0, 310.0, n)
    grid["p_def"] = rng.uniform(7e4, 1.05e5, n)
    madict = random_inputs(ma["ept"].size, seed=11)
    madict["ept"] = ma["ept"]
    madict["p"] = ma["p"]
    return {"rand": random_inputs(1024, seed=0), "edge": edge_inputs(), "grid": grid, "ma": madict}


def call(mod, case, inputs, dtype):
    args = [np.ascontiguousarray(inputs[a].astype(dtype)) for a in case.args]
    with np.errstate(all="ignore"):
        res = getattr(mod, case.fn)(*args, **case.kwargs)
    if not isinstance(res, tuple):
        res = (res,)
    return [np.asarray(r) for r in res]


def pack_ifs_levels():
    """IFS L137 hybrid A/B half-level coefficients (reference src/earthkit/meteo/conf/ifs_levels_conf.json),
    used by bench.py to lay out the synthetic O1280 x 137 pressure field (SURVEY.md 8(d))."""
    with open(os.path.join(REF, "src", "earthkit", "meteo", "conf", "ifs_levels_conf.json")) as f:
        d = json.load(f)["137"]
    return {"A": np.asarray(d["A"], dtype=np.float64), "B": np.asarray(d["B"], dtype=np.float64)}


HYBRID_LEVEL_SETS = {"all": None, "lower": list(range(90, 138)), "reversed": list(range(137, 90, -1)), "two": [2, 1], "top": [1]}


def pack_hybrid():
    """Hybrid-level pressure (SURVEY.md 8(f)-1): the reference's golden vectors (tests/vertical/_hybrid_core_data.py,
    consumed at tests/vertical/test_array_vertical.py:159-370) and live outputs of the unmodified
    earthkit.meteo.vertical.pressure_on_hybrid_levels on seeded surface pressures, float64 and float32.
    Returns (blob, worst oracle-vs-reference difference)."""
    sys.path.insert(0, os.path.join(REF, "tests", "vertical"))
    import _hybrid_core_data as D
    import vertical_oracle as voracle
    from earthkit.meteo import vertical as ref_vertical

    blob = {"gold/A": np.asarray(D.A, dtype=np.float64), "gold/B": np.asarray(D.B, dtype=np.float64),
            "gold/p_surf": np.asarray(D.p_surf, dtype=np.float64), "gold/full": np.asarray(D.p_full, dtype=np.float64),
            "gold/half": np.asarray(D.p_half, dtype=np.float64), "gold/delta": np.asarray(D.delta, dtype=np.float64),
            "gold/alpha": np.asarray(D.alpha, dtype=np.float64)}
    rng = np.random.default_rng(17)
    sp = rng.uniform(4.5e4, 1.06e5, 40)
    blob["live/sp"] = sp
    mism = 0
    for dt in (np.float64, np.float32):
        a, b, s = (np.asarray(x, dtype=dt) for x in (D.A, D.B, sp))
        for lname, lv in HYBRID_LEVEL_SETS.items():
            for at in ("ifs", "arpege"):
                r = ref_vertical.pressure_on_hybrid_levels(a, b, s, levels=lv, alpha_top=at, output=["full", "half", "delta", "alpha"])
                o = voracle.pressure_on_hybrid_levels(a, b, s, levels=lv, alpha_top=at, output=["full", "half", "delta", "alpha"])
                for name, rv, ov in zip(("full", "half", "delta", "alpha"), r, o):
                    blob[f"live/{np.dtype(dt).name}/{lname}/{at}/{name}"] = rv
                    mism += int(not (rv.shape == ov.shape and rv.dtype == ov.dtype and np.array_equal(rv, ov, equal_nan=True)))
    # --- SURVEY.md 8(f)-2: geopotential thickness / geopotential / height on hybrid levels ------------------------
    import _hybrid_height_data as H

    blob.update({"gold/t": np.asarray(D.t, dtype=np.float64), "gold/q": np.asarray(D.q, dtype=np.float64),
                 "gold/z": np.asarray(D.z, dtype=np.float64)})
    for k in ("A", "B", "t", "q", "z_surf", "p_surf", "h_geopotential_sea", "h_geopotential_ground", "h_geometric_sea", "h_geometric_ground"):
        blob[f"goldh/{k}"] = np.asarray(getattr(H, k), dtype=np.float64)
    npt = 24
    sp2 = rng.uniform(5.0e4, 1.05e5, npt)
    zs2 = rng.uniform(-500.0, 3.0e4, npt)
    pf = ref_vertical.pressure_on_hybrid_levels(np.asarray(D.A), np.asarray(D.B), sp2)
    t2 = np.clip(288.15 * (pf / 101325.0) ** 0.19 + rng.uniform(-10, 10, pf.shape), 180.0, 320.0)
    q2 = rng.uniform(1e-6, 0.02, pf.shape)
    blob.update({"geo/sp": sp2, "geo/zs": zs2, "geo/t": t2, "geo/q": q2})
    for dt in (np.float64, np.float32):
        dn = np.dtype(dt).name
        a, b, s_, z_, tt, qq = (np.asarray(x, dtype=dt) for x in (D.A, D.B, sp2, zs2, t2, q2))
        for part, sl in (("all", slice(None)), ("lower", slice(90, None))):
            for at in ("ifs", "arpege"):
                calls = {
                    "thickness": lambda m: m.relative_geopotential_thickness_on_hybrid_levels(tt[sl], qq[sl], a, b, s_, alpha_top=at),
                    "geopotential": lambda m: m.geopotential_on_hybrid_levels(tt[sl], qq[sl], z_, a, b, s_, alpha_top=at),
                }
                for ht in ("geometric", "geopotential"):
                    for hr in ("sea", "ground"):
                        calls[f"h_{ht}_{hr}"] = (lambda m, ht=ht, hr=hr: m.height_on_hybrid_levels(tt[sl], qq[sl], z_, a, b, s_, alpha_top=at, h_type=ht, h_reference=hr))
                for name, fn in calls.items():
                    rv, ov = fn(ref_vertical), fn(voracle)
                    blob[f"geo/{dn}/{part}/{at}/{name}"] = rv
                    mism += int(not (rv.shape == ov.shape and rv.dtype == ov.dtype and np.array_equal(rv, ov, equal_nan=True)))
        al, de = ref_vertical.pressure_on_hybrid_levels(a, b, s_, output=("alpha", "delta"))
        rv = ref_vertical.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(tt, qq, al, de)
        ov = voracle.relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(tt, qq, al, de)
        blob[f"geo/{dn}/from_alpha_delta"] = rv
        mism += int(not np.array_equal(rv, ov, equal_nan=True))
    return blob, mism


def pack_hybrid_axis():
    """vertical_axis != 0 in the geopotential functions (reference vertical.py:981-986): the reference moves the alpha / delta
    it just computed with their level axis FIRST a second time, which is only shape-consistent for square fields (as many columns
    as levels) and scrambles alpha / delta there; every other shape raises numpy's broadcast ValueError.  SURVEY 7.3-H5 is
    "replicate, don't fix": these are the reference's own outputs for a square field, and the exception it raises otherwise.
    Also the stand-alone height conversions (vertical.py:330-502) that the replicated path post-processes with."""
    sys.path.insert(0, os.path.join(REF, "tests", "vertical"))
    import _hybrid_core_data as D
    import vertical_oracle as voracle
    from earthkit.meteo import vertical as ref_vertical

    rng = np.random.default_rng(29)
    A, B = np.asarray(D.A, dtype=np.float64), np.asarray(D.B, dtype=np.float64)
    n = 12  # 12 bottom-most levels x 12 columns
    sp = rng.uniform(6.0e4, 1.05e5, n)
    zs = rng.uniform(-300.0, 2.0e4, n)
    pf = ref_vertical.pressure_on_hybrid_levels(A, B, sp, levels=list(range(A.size - n, A.size)))
    t = np.clip(288.15 * (pf / 101325.0) ** 0.19 + rng.uniform(-8, 8, pf.shape), 180.0, 320.0)  # [level, column]
    q = rng.uniform(1e-6, 0.02, pf.shape)
    blob = {"A": A, "B": B, "sp": sp, "zs": zs, "t": t, "q": q}
    mism = 0
    t1, q1 = np.ascontiguousarray(t.T), np.ascontiguousarray(q.T)  # [column, level]: vertical axis 1
    for axis in (1, -1):
        calls = {"thickness": lambda m: m.relative_geopotential_thickness_on_hybrid_levels(t1, q1, A, B, sp, vertical_axis=axis),
                 "geopotential": lambda m: m.geopotential_on_hybrid_levels(t1, q1, zs, A, B, sp, vertical_axis=axis)}
        for ht in ("geometric", "geopotential"):
            for hr in ("sea", "ground"):
                calls[f"h_{ht}_{hr}"] = (lambda m, ht=ht, hr=hr: m.height_on_hybrid_levels(t1, q1, zs, A, B, sp, h_type=ht, h_reference=hr, vertical_axis=axis))
        for name, fn in calls.items():
            rv, ov = fn(ref_vertical), fn(voracle)
            blob[f"axis{axis}/{name}"] = rv
            mism += int(not (rv.shape == ov.shape and np.array_equal(rv, ov, equal_nan=True)))
    # the consistent answer (vertical axis first), to show that the reference's axis != 0 result is NOT it
    blob["axis0/thickness"] = ref_vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, A, B, sp)
    try:  # any non-square field
        ref_vertical.relative_geopotential_thickness_on_hybrid_levels(t1[:5], q1[:5], A, B, sp[:5], vertical_axis=1)
        blob["nonsquare_error"] = np.asarray("none")
    except Exception as e:  # noqa: BLE001
        blob["nonsquare_error"] = np.asarray(type(e).__name__)
    z = np.concatenate([rng.uniform(-5.0e3, 6.0e5, 200), [0.0, np.nan, np.inf, -np.inf, 6371229.0 * 9.80665]])
    blob["conv/z"] = z
    with np.errstate(all="ignore"):
        blob["conv/geopotential_height"] = ref_vertical.geopotential_height_from_geopotential(z)
        blob["conv/geometric_height"] = ref_vertical.geometric_height_from_geopotential(z)
        mism += int(not np.array_equal(blob["conv/geopotential_height"], voracle.geopotential_height_from_geopotential(z), equal_nan=True))
        mism += int(not np.array_equal(blob["conv/geometric_height"], voracle.geometric_height_from_geopotential(z), equal_nan=True))
    return blob, mism


def main_hybrid_axis():
    blob, mism = pack_hybrid_axis()
    np.savez_compressed(os.path.join(HERE, "ref_hybrid_axis.npz"), **blob)
    path = os.path.join(HERE, "PINNING.json")
    with open(path) as f:
        pin = json.load(f)
    pin["hybrid_axis"] = {"arrays_not_bit_identical_to_reference": mism, "n_arrays": sum(k.startswith(("axis", "conv/g")) for k in blob),
                          "nonsquare_error": str(blob["nonsquare_error"])}
    with open(path, "w") as f:
        json.dump(pin, f, indent=1, sort_keys=True)
    print(json.dumps(pin["hybrid_axis"]))


WIND_CASES = [  # (function, argument names, kwargs)
    ("speed", ("u", "v"), {}),
    ("direction", ("u", "v"), {"convention": "meteo"}),
    ("direction", ("u", "v"), {"convention": "polar"}),
    ("direction", ("u", "v"), {"convention": "polar", "to_positive": False}),
    ("xy_to_polar", ("u", "v"), {"convention": "meteo"}),
    ("xy_to_polar", ("u", "v"), {"convention": "polar"}),
    ("polar_to_xy", ("mag", "dir"), {"convention": "meteo"}),
    ("polar_to_xy", ("mag", "dir"), {"convention": "polar"}),
    ("w_from_omega", ("omega", "t", "p"), {}),
    ("coriolis", ("lat",), {}),
]


def wind_case_id(fn, kwargs):
    return fn + "".join(f";{k}={v}" for k, v in sorted(kwargs.items()))


def wind_inputs(n=600, seed=23):
    rng = np.random.default_rng(seed)
    special = np.array([0.0, -0.0, 1.0, -1.0, np.nan, np.inf, -np.inf, 1e-300, 1e300, 25.0, -12.5])
    u = np.concatenate([rng.normal(0, 12, n), special[rng.integers(0, special.size, 60)], [0, 1, 1, 1, 0, -1, -1, -1, 0, np.nan, 1, np.nan]])
    v = np.concatenate([rng.normal(0, 12, n), special[rng.integers(0, special.size, 60)], [1, 1, 0, -1, -1, -1, 0, 1, 0, 1, np.nan, np.nan]])
    m = u.size
    return dict(u=u, v=v, mag=np.abs(rng.normal(8, 6, m)), dir=rng.uniform(-90, 450, m), omega=rng.normal(0, 2, m),
                t=rng.uniform(200, 320, m), p=rng.uniform(1e3, 1.05e5, m), lat=rng.uniform(-90, 90, m))


def pack_wind():
    """SURVEY.md 8(f)-3: live outputs of the unmodified earthkit.meteo.wind elementwise functions (float64 and float32)."""
    import wind_oracle as woracle
    from earthkit.meteo import wind as ref_wind

    inp = wind_inputs()
    blob = {f"in/{k}": v for k, v in inp.items()}
    mism = 0
    for dt in (np.float64, np.float32):
        for fn, args, kw in WIND_CASES:
            a = [inp[x].astype(dt) for x in args]
            with np.errstate(all="ignore"):
                r, o = getattr(ref_wind, fn)(*a, **kw), getattr(woracle, fn)(*a, **kw)
            r = r if isinstance(r, tuple) else (r,)
            o = o if isinstance(o, tuple) else (o,)
            for k, (rv, ov) in enumerate(zip(r, o)):
                rv = np.asarray(rv)
                blob[f"out/{np.dtype(dt).name}/{wind_case_id(fn, kw)}/{k}"] = rv
                mism += int(not (rv.shape == np.shape(ov) and rv.dtype == np.asarray(ov).dtype and np.array_equal(rv, ov, equal_nan=True)))
    return blob, mism


def save_split(stem, blob, parts):
    """`blob` as <stem>_<suffix>.npz for every (suffix, key prefix) of `parts` and <stem>.npz for the other keys."""
    prefixes = tuple(pre for _, pre in parts)
    np.savez_compressed(os.path.join(HERE, f"{stem}.npz"), **{k: v for k, v in blob.items() if not k.startswith(prefixes)})
    for suffix, pre in parts:
        np.savez_compressed(os.path.join(HERE, f"{stem}_{suffix}.npz"), **{k: v for k, v in blob.items() if k.startswith(pre)})


def main():
    np.savez_compressed(os.path.join(HERE, "ref_csv.npz"), **pack_csvs())
    wind_blob, wind_mismatch = pack_wind()
    np.savez_compressed(os.path.join(HERE, "ref_wind.npz"), **wind_blob)
    hyb, hyb_mismatch = pack_hybrid()
    save_split("ref_hybrid", hyb, [("geo", "geo/")])
    np.savez_compressed(os.path.join(HERE, "ifs_l137_ab.npz"), **pack_ifs_levels())

    sets = input_sets()
    blob = {}
    pin = {"numpy": np.__version__, "cases": {}, "summary": {}}
    worst = 0.0
    nan_mismatch = 0
    n_entries = 0
    for sname, inputs in sets.items():
        for k, v in inputs.items():
            blob[f"in/{sname}/{k}"] = v
        for dtype in (np.float64, np.float32):
            if dtype is np.float32 and sname in ("grid", "ma"):
                continue
            dname = np.dtype(dtype).name
            for case in CASES:
                if sname == "ma" and case.fn != "temperature_on_moist_adiabat":
                    continue
                r = call(ref_thermo, case, inputs, dtype)
                o = call(oracle, case, inputs, dtype)
                for k, (rv, ov) in enumerate(zip(r, o)):
                    blob[f"out/{sname}/{dname}/{case.id}/{k}"] = rv
                    assert rv.shape == ov.shape, (case.id, rv.shape, ov.shape)
                    assert rv.dtype == ov.dtype, (case.id, rv.dtype, ov.dtype)
                    nm = int(np.sum(np.isnan(rv) != np.isnan(ov)))
                    fin = np.isfinite(rv) & np.isfinite(ov)
                    infs = int(np.sum((~fin) & ~np.isnan(rv) & (rv != ov)))
                    with np.errstate(all="ignore"):
                        rel = np.abs(rv[fin] - ov[fin]) / np.maximum(np.abs(rv[fin]), 1e-300)
                    m = float(rel.max()) if rel.size else 0.0
                    worst = max(worst, m)
                    nan_mismatch += nm + infs
                    n_entries += 1
                    if m > 0.0 or nm or infs:  # only deviations are listed; an empty dict = bit-identical
                        pin["cases"][f"{sname}/{dname}/{case.id}/{k}"] = {"max_rel": m, "nan_mismatch": nm, "inf_mismatch": infs}
    pin["summary"] = {"worst_max_rel": worst, "nan_or_inf_mismatches": nan_mismatch, "n_entries": n_entries}
    pin["wind"] = {"arrays_not_bit_identical_to_reference": wind_mismatch, "n_arrays": sum(k.startswith("out/") for k in wind_blob)}
    pin["hybrid"] = {"arrays_not_bit_identical_to_reference": hyb_mismatch, "n_arrays": sum(k.startswith("live/float") or k.startswith("geo/float") for k in hyb)}
    save_split("ref_live", blob, [("rand_float64", "out/rand/float64/"), ("rand_float32", "out/rand/float32/")])
    with open(os.path.join(HERE, "PINNING.json"), "w") as f:
        json.dump(pin, f, indent=1, sort_keys=True)
    print(json.dumps(pin["summary"]))


if __name__ == "__main__":
    if "--hybrid-axis" in sys.argv:  # only the vertical_axis != 0 fixtures (added in round 2; the other files stay as generated)
        main_hybrid_axis()
    else:
        main()
        main_hybrid_axis()
