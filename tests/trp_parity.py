"""What the (t, r, p) suite must equal, and the parity rule of tests/compare.py applied to it output by output.

``suite_trp`` states the suite as a composition of the pinned functions of oracle/thermo_oracle.py (no new reference semantics),
next to the oracle's own ``suite_tqp`` / ``suite_ttdp``.  Shared by tests/test_suite_trp_cpu.py (mock device) and
tests/test_gpu_suite_trp.py.  The conditioning and float32 noise that ``compare`` accepts are those of compare.conditioning /
compare.reference_f32_noise, computed here for every output of the suite from one composition call per perturbation."""
from types import SimpleNamespace

import numpy as np

import thermo_oracle as oracle
from compare import _step_ulps, compare


def suite_trp(t, r, p, ept_method="ifs"):
    """What the fused (t,r,p) kernel must equal, output by output (r in %).  "ept" / "wbpt" follow q, so their dewpoint is
    dewpoint_from_specific_humidity(q, p) (T:1036-1037), not the "td" output's dewpoint_from_relative_humidity(t, r)."""
    q = oracle.specific_humidity_from_relative_humidity(t, r, p)
    with np.errstate(all="ignore"):
        e = r * oracle.saturation_vapour_pressure(t) / 100.0  # T:662
    return {
        "theta": oracle.potential_temperature(t, p),
        "es": oracle.saturation_vapour_pressure(t),
        "td": oracle.dewpoint_from_relative_humidity(t, r),
        "q": q,
        "tv": oracle.virtual_temperature(t, q),
        "w": oracle.mixing_ratio_from_specific_humidity(q),
        "e": e,
        "thetav": oracle.virtual_potential_temperature(t, q, p),
        "ept": oracle.ept_from_specific_humidity(t, q, p, method=ept_method),
        "wbpt": oracle.wet_bulb_potential_temperature_from_specific_humidity(t, q, p, ept_method=ept_method, t_method="direct"),
    }


def _asf64(d):
    return {k: np.asarray(v).astype(np.float64) for k, v in d.items()}


def suite_conditioning(args, ept_method="ifs"):
    """{name: relative change of the oracle output per ulp of input perturbation}, as compare.conditioning."""
    with np.errstate(all="ignore"):
        base = _asf64(suite_trp(*args, ept_method=ept_method))
        cond = {k: np.zeros(v.shape) for k, v in base.items()}
        for i, a in enumerate(args):
            for k in (1, -1, 16, -16):
                pert = list(args)
                pert[i] = _step_ulps(a, k)
                res = _asf64(suite_trp(*pert, ept_method=ept_method))
                for name, b in base.items():
                    d = np.abs(res[name] - b) / np.maximum(np.abs(b), 1e-300) / abs(k)
                    cond[name] = np.fmax(cond[name], np.where(np.isfinite(d), d, 0.0))
    return cond


def suite_f32_noise(args, ept_method="ifs"):
    """{name: the oracle in float32 against the oracle in float64 on the same inputs}, as compare.reference_f32_noise."""
    with np.errstate(all="ignore"):
        w32 = _asf64(suite_trp(*args, ept_method=ept_method))
        w64 = _asf64(suite_trp(*[np.asarray(a).astype(np.float64) for a in args], ept_method=ept_method))
        return {k: np.where(np.isfinite(n), n, 0.0) for k in w32 for n in [np.abs(w32[k] - w64[k]) / np.maximum(np.abs(w64[k]), 1e-300)]}


def check_suite(got, args, ept_method="ifs", edge=False):
    """Assert every output in `got` ({name: numpy array}) equals suite_trp(*args) under compare()'s rule; args are the
    numpy (t, r, p) of the dtype the suite ran in.  NaN and inf positions must be identical in float64."""
    dtype = np.asarray(args[0]).dtype.type
    with np.errstate(all="ignore"):
        want = suite_trp(*args, ept_method=ept_method)
    cond = suite_conditioning(args, ept_method)
    noise = suite_f32_noise(args, ept_method) if dtype == np.float32 else {}
    for name, g in got.items():
        case = SimpleNamespace(id=f"suite_trp[{name}, ept_method={ept_method}]", iterative="")
        compare(case, g, want[name], dtype, edge=edge, cond=cond[name], noise=noise.get(name))
