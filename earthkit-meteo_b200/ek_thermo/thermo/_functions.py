"""Drop-in for ``earthkit.meteo.thermo.array`` on torch CUDA tensors.

Same 39 names, positional order, keyword names, defaults and exceptions as the reference
(src/earthkit/meteo/thermo/array/thermo.py = "T", es_comp.py = "E"; SURVEY.md §8(b)).  Each function
validates its options the way the reference does and then launches ONE sm_100a kernel through the
C ABI (include/ek_thermo.h).  Inputs: torch CUDA tensors (float64 or float32) and/or Python numbers
(broadcast by value).  Output: a new tensor of the broadcast shape on the same device.

Extensions over the reference (supersets, never changes of behaviour for valid 1-D calls):
N-D inputs are accepted by the bisect/newton solvers (the reference raises a broadcast error for
N-D, SURVEY.md §7.3-H6).
"""
from __future__ import annotations

from .. import _backend as _b
from .._backend import _EPT

_PHASE = {"mixed": 0, "water": 1, "ice": 2}  # E:22
_LCL = {"davies": 0, "bolton": 1}  # T:960-968
_TM = {"direct": 1, "bisect": 2, "newton": 3}

__all__ = [
    "celsius_to_kelvin",
    "kelvin_to_celsius",
    "specific_humidity_from_mixing_ratio",
    "mixing_ratio_from_specific_humidity",
    "vapour_pressure_from_specific_humidity",
    "vapour_pressure_from_mixing_ratio",
    "specific_humidity_from_vapour_pressure",
    "mixing_ratio_from_vapour_pressure",
    "saturation_vapour_pressure",
    "saturation_mixing_ratio",
    "saturation_specific_humidity",
    "saturation_vapour_pressure_slope",
    "saturation_mixing_ratio_slope",
    "saturation_specific_humidity_slope",
    "temperature_from_saturation_vapour_pressure",
    "relative_humidity_from_dewpoint",
    "relative_humidity_from_specific_humidity",
    "specific_humidity_from_dewpoint",
    "mixing_ratio_from_dewpoint",
    "specific_humidity_from_relative_humidity",
    "dewpoint_from_relative_humidity",
    "dewpoint_from_specific_humidity",
    "virtual_temperature",
    "virtual_potential_temperature",
    "potential_temperature",
    "temperature_from_potential_temperature",
    "pressure_on_dry_adiabat",
    "temperature_on_dry_adiabat",
    "lcl_temperature",
    "lcl",
    "ept_from_dewpoint",
    "ept_from_specific_humidity",
    "saturation_ept",
    "temperature_on_moist_adiabat",
    "wet_bulb_temperature_from_dewpoint",
    "wet_bulb_temperature_from_specific_humidity",
    "wet_bulb_potential_temperature_from_dewpoint",
    "wet_bulb_potential_temperature_from_specific_humidity",
    "specific_gas_constant",
]


def _ept_id(method):
    # the reference looks the method up in a dict: an unknown name is a KeyError (T:1024-1026)
    return _EPT[method]


def celsius_to_kelvin(t):
    """t [degC] -> K.  Reference T:21-35."""
    return _b.execute("celsius_to_kelvin", (t,))


def kelvin_to_celsius(t):
    """t [K] -> degC.  Reference T:38-52."""
    return _b.execute("kelvin_to_celsius", (t,))


def specific_humidity_from_mixing_ratio(w):
    """q = w/(1+w).  Reference T:55-77."""
    return _b.execute("specific_humidity_from_mixing_ratio", (w,))


def mixing_ratio_from_specific_humidity(q):
    """w = q/(1-q).  Reference T:80-102."""
    return _b.execute("mixing_ratio_from_specific_humidity", (q,))


def vapour_pressure_from_specific_humidity(q, p):
    """e = p q / (eps + (1-eps) q).  Reference T:105-131."""
    return _b.execute("vapour_pressure_from_specific_humidity", (q, p))


def vapour_pressure_from_mixing_ratio(w, p):
    """e = p w / (eps + w).  Reference T:134-159."""
    return _b.execute("vapour_pressure_from_mixing_ratio", (w, p))


def specific_humidity_from_vapour_pressure(e, p, eps=1e-4):
    """q from vapour pressure; NaN where p - e < eps; eps <= 0 raises ValueError.  Reference T:162-196."""
    if eps <= 0:
        raise ValueError(f"specific_humidity_from_vapour_pressure(): eps={eps} must be > 0")
    return _b.execute("specific_humidity_from_vapour_pressure", (e, p), (float(eps),))


def mixing_ratio_from_vapour_pressure(e, p, eps=1e-4):
    """w from vapour pressure; NaN where p - e < eps; eps <= 0 raises ValueError.  Reference T:199-232."""
    if eps <= 0:
        raise ValueError(f"mixing_ratio_from_vapour_pressure(): eps={eps} must be > 0")
    return _b.execute("mixing_ratio_from_vapour_pressure", (e, p), (float(eps),))


def saturation_vapour_pressure(t, phase="mixed"):
    """es(t) over water / ice / mixed phase.  Reference T:235-279, E:31-79.

    As in the reference, an unknown ``phase`` silently returns None (E:74-79; check_phase is never called).
    """
    if phase not in _PHASE:
        return None
    return _b.execute("saturation_vapour_pressure", (t,), (_PHASE[phase],))


def saturation_mixing_ratio(t, p, phase="mixed"):
    """ws(t, p).  Reference T:282-310."""
    if phase not in _PHASE:
        # reference: es is None -> TypeError inside mixing_ratio_from_vapour_pressure (p - None)
        raise TypeError("unsupported operand type(s) for -: 'Tensor' and 'NoneType'")
    return _b.execute("saturation_mixing_ratio", (t, p), (_PHASE[phase],))


def saturation_specific_humidity(t, p, phase="mixed"):
    """qs(t, p).  Reference T:313-341."""
    if phase not in _PHASE:
        raise TypeError("unsupported operand type(s) for *: 'float' and 'NoneType'")
    return _b.execute("saturation_specific_humidity", (t, p), (_PHASE[phase],))


def saturation_vapour_pressure_slope(t, phase="mixed"):
    """d es / dt.  Reference T:344-364, E:82-106.  Unknown phase -> None, as in the reference."""
    if phase not in _PHASE:
        return None
    return _b.execute("saturation_vapour_pressure_slope", (t,), (_PHASE[phase],))


def _slope(symbol, t, p, es, es_slope, phase, eps):
    if eps <= 0:
        raise ValueError(f"{symbol}(): eps={eps} must be > 0")
    if phase not in _PHASE and (es is None or es_slope is None):
        raise TypeError("unsupported operand type(s) for -: 'Tensor' and 'NoneType'")
    ph = _PHASE.get(phase, 0)
    return _b.execute(symbol, (t, p, es, es_slope), (int(es is not None), int(es_slope is not None), ph, float(eps)))


def saturation_mixing_ratio_slope(t, p, es=None, es_slope=None, phase="mixed", eps=1e-4):
    """d ws / dt; es and es_slope may be passed in precomputed.  Reference T:367-415."""
    return _slope("saturation_mixing_ratio_slope", t, p, es, es_slope, phase, eps)


def saturation_specific_humidity_slope(t, p, es=None, es_slope=None, phase="mixed", eps=1e-4):
    """d qs / dt; es and es_slope may be passed in precomputed.  Reference T:418-467."""
    return _slope("saturation_specific_humidity_slope", t, p, es, es_slope, phase, eps)


def temperature_from_saturation_vapour_pressure(es):
    """Inverse of the water-phase es formula; es = 0 gives NaN.  Reference T:470-491, E:109-130."""
    return _b.execute("temperature_from_saturation_vapour_pressure", (es,))


def relative_humidity_from_dewpoint(t, td):
    """r [%] = 100 es_w(td)/es_w(t).  Reference T:494-521."""
    return _b.execute("relative_humidity_from_dewpoint", (t, td))


def relative_humidity_from_specific_humidity(t, q, p):
    """r [%] = 100 e(q,p)/es_mixed(t).  Reference T:524-556."""
    return _b.execute("relative_humidity_from_specific_humidity", (t, q, p))


def specific_humidity_from_dewpoint(td, p):
    """Reference T:559-591."""
    return _b.execute("specific_humidity_from_dewpoint", (td, p))


def mixing_ratio_from_dewpoint(td, p):
    """Reference T:594-626."""
    return _b.execute("mixing_ratio_from_dewpoint", (td, p))


def specific_humidity_from_relative_humidity(t, r, p):
    """Reference T:629-663."""
    return _b.execute("specific_humidity_from_relative_humidity", (t, r, p))


def dewpoint_from_relative_humidity(t, r):
    """Reference T:666-699 (r = 0 gives NaN)."""
    return _b.execute("dewpoint_from_relative_humidity", (t, r))


def dewpoint_from_specific_humidity(q, p):
    """Reference T:702-735 (q = 0 gives NaN)."""
    return _b.execute("dewpoint_from_specific_humidity", (q, p))


def virtual_temperature(t, q):
    """Reference T:738-764."""
    return _b.execute("virtual_temperature", (t, q))


def virtual_potential_temperature(t, q, p):
    """Reference T:767-798."""
    return _b.execute("virtual_potential_temperature", (t, q, p))


def potential_temperature(t, p):
    """theta = t (p0/p)^kappa.  Reference T:801-829."""
    return _b.execute("potential_temperature", (t, p))


def temperature_from_potential_temperature(th, p):
    """Reference T:832-858."""
    return _b.execute("temperature_from_potential_temperature", (th, p))


def pressure_on_dry_adiabat(t, t_def, p_def):
    """Reference T:861-889."""
    return _b.execute("pressure_on_dry_adiabat", (t, t_def, p_def))


def temperature_on_dry_adiabat(p, t_def, p_def):
    """Reference T:892-920."""
    return _b.execute("temperature_on_dry_adiabat", (p, t_def, p_def))


def lcl_temperature(t, td, method="davies"):
    """Closed-form LCL temperature (Davies-Jones or Bolton).  Reference T:923-968."""
    if method not in _LCL:
        raise ValueError(f"lcl_temperature: invalid method={method} specified!")
    return _b.execute("lcl_temperature", (t, td), (_LCL[method],))


def lcl(t, td, p, method="davies"):
    """(t_lcl, p_lcl) in one kernel.  Reference T:971-1000."""
    if method not in _LCL:
        raise ValueError(f"lcl_temperature: invalid method={method} specified!")
    return _b.execute("lcl", (t, td, p), (_LCL[method],))


def ept_from_dewpoint(t, td, p, method="ifs"):
    """Equivalent potential temperature from dewpoint.  Reference T:1326-1387."""
    return _b.execute("ept_from_dewpoint", (t, td, p), (_ept_id(method),))


def ept_from_specific_humidity(t, q, p, method="ifs"):
    """Equivalent potential temperature from specific humidity.  Reference T:1390-1415."""
    return _b.execute("ept_from_specific_humidity", (t, q, p), (_ept_id(method),))


def saturation_ept(t, p, method="ifs"):
    """Saturation equivalent potential temperature.  Reference T:1418-1469."""
    return _b.execute("saturation_ept", (t, p), (_ept_id(method),))


def temperature_on_moist_adiabat(ept, p, ept_method="ifs", t_method="bisect"):
    """Temperature at p on the moist adiabat of ept ("bisect": 12 halvings; "newton": 1 step).  Reference T:1472-1509."""
    m = _ept_id(ept_method)
    if t_method not in ("bisect", "newton"):
        raise ValueError(f"temperature_on_moist_adiabat: invalid t_method={t_method} specified!")
    return _b.execute("temperature_on_moist_adiabat", (ept, p), (m, _TM[t_method]))


def _wet_bulb(symbol, t, h, p, ept_method, t_method, allow_direct):
    m = _ept_id(ept_method)
    ok = ("direct", "bisect", "newton") if allow_direct else ("bisect", "newton")
    if t_method not in ok:
        raise ValueError(f"temperature_on_moist_adiabat: invalid t_method={t_method} specified!")
    return _b.execute(symbol, (t, h, p), (m, _TM[t_method]))


def wet_bulb_temperature_from_dewpoint(t, td, p, ept_method="ifs", t_method="bisect"):
    """Reference T:1512-1549."""
    return _wet_bulb("wet_bulb_temperature_from_dewpoint", t, td, p, ept_method, t_method, False)


def wet_bulb_temperature_from_specific_humidity(t, q, p, ept_method="ifs", t_method="bisect"):
    """Reference T:1552-1590."""
    return _wet_bulb("wet_bulb_temperature_from_specific_humidity", t, q, p, ept_method, t_method, False)


def wet_bulb_potential_temperature_from_dewpoint(t, td, p, ept_method="ifs", t_method="direct"):
    """Reference T:1593-1634."""
    return _wet_bulb("wet_bulb_potential_temperature_from_dewpoint", t, td, p, ept_method, t_method, True)


def wet_bulb_potential_temperature_from_specific_humidity(t, q, p, ept_method="ifs", t_method="direct"):
    """Reference T:1637-1675."""
    return _wet_bulb("wet_bulb_potential_temperature_from_specific_humidity", t, q, p, ept_method, t_method, True)


def specific_gas_constant(q):
    """R = Rd + (Rv - Rd) q.  Reference T:1678-1707."""
    return _b.execute("specific_gas_constant", (q,))
