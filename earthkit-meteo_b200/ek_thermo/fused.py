"""Fused multi-output kernels: read the state of each grid point once, write every requested field.

These have no counterpart function in the reference; every output equals the reference function
named in ``SUITE_TQP_OUTPUTS`` / ``SUITE_TTDP_OUTPUTS`` / ``SUITE_TRP_OUTPUTS`` applied to the same inputs (the
oracle's ``suite_tqp`` / ``suite_ttdp`` and the tests' ``trp_parity.suite_trp`` state that composition).  HBM traffic per point is
``8 * (3 + len(outputs))`` bytes in float64, instead of one full read+write pass per function.
"""
from __future__ import annotations

from ctypes import c_void_p

import torch

from . import _backend as _b
from ._backend import _EPT
from .vertical import COLUMN_OUTPUTS  # noqa: F401  (part of this module's API: the column outputs of suite_tq_hybrid)
from .vertical import _alpha_top_value, _column_kernel, _split_suite_outputs, _top_is_toa

# output name -> slot (include/ek_thermo.h EK_S_*), with the reference function each one equals
SUITE_TQP_OUTPUTS = {
    "theta": 0,  # potential_temperature(t, p)                          T:801-829
    "es": 1,  # saturation_vapour_pressure(t)                            T:235-279
    "rh": 2,  # relative_humidity_from_specific_humidity(t, q, p)        T:524-556
    "td": 3,  # dewpoint_from_specific_humidity(q, p)                    T:702-735
    "tv": 4,  # virtual_temperature(t, q)                                T:738-764
    "w": 5,  # mixing_ratio_from_specific_humidity(q)                    T:80-102
    "e": 6,  # vapour_pressure_from_specific_humidity(q, p)              T:105-131
    "thetav": 7,  # virtual_potential_temperature(t, q, p)               T:767-798
    "ept": 8,  # ept_from_specific_humidity(t, q, p, method=ept_method)  T:1390-1415
    "wbpt": 9,  # wet_bulb_potential_temperature_from_specific_humidity(t, q, p, ept_method, t_method="direct")  T:1637-1675
}
SUITE_TTDP_OUTPUTS = {
    "theta": 0,  # potential_temperature(t, p)
    "es": 1,  # saturation_vapour_pressure(t)
    "rh": 2,  # relative_humidity_from_dewpoint(t, td)                   T:494-521
    "q": 3,  # specific_humidity_from_dewpoint(td, p)                    T:559-591
    "tv": 4,  # virtual_temperature(t, q(td, p))
    "w": 5,  # mixing_ratio_from_dewpoint(td, p)                         T:594-626
    "e": 6,  # saturation_vapour_pressure(td, phase="water")
    "thetav": 7,  # virtual_potential_temperature(t, q(td, p), p)
    "ept": 8,  # ept_from_dewpoint(t, td, p, method=ept_method)          T:1326-1387
    "wbpt": 9,  # wet_bulb_potential_temperature_from_dewpoint(t, td, p, ept_method, t_method="direct")  T:1593-1634
}
# q = specific_humidity_from_relative_humidity(t, r, p) (T:629-663), r in %; "ept" / "wbpt" follow q, so their dewpoint is
# dewpoint_from_specific_humidity(q, p) (T:1036-1037), not the "td" slot's, which is over water and differs below T0
SUITE_TRP_OUTPUTS = {
    "theta": 0,  # potential_temperature(t, p)
    "es": 1,  # saturation_vapour_pressure(t)
    "td": 2,  # dewpoint_from_relative_humidity(t, r)                    T:666-699
    "q": 3,  # specific_humidity_from_relative_humidity(t, r, p)         T:629-663
    "tv": 4,  # virtual_temperature(t, q)
    "w": 5,  # mixing_ratio_from_specific_humidity(q)
    "e": 6,  # r * saturation_vapour_pressure(t) / 100.0                 T:662
    "thetav": 7,  # virtual_potential_temperature(t, q, p)
    "ept": 8,  # ept_from_specific_humidity(t, q, p, method=ept_method)
    "wbpt": 9,  # wet_bulb_potential_temperature_from_specific_humidity(t, q, p, ept_method, t_method="direct")
}
# the single pass BASELINE.json names: "read t/q/p (or t/td/p) once and write theta, rh, td, theta_e and wbpt"
SINGLE_PASS_TQP = ("theta", "rh", "td", "ept", "wbpt")
SINGLE_PASS_TTDP = ("theta", "rh", "q", "ept", "wbpt")
# ... and with the two remaining fields of the default suite: 10 arrays = 80 bytes per point in float64
ALL7_TQP = ("theta", "es", "rh", "td", "tv", "ept", "wbpt")
ALL7_TTDP = ("theta", "es", "rh", "q", "tv", "ept", "wbpt")
DEFAULT_TQP = ("theta", "es", "rh", "td", "tv")
DEFAULT_TTDP = ("theta", "es", "rh", "q", "tv")
DEFAULT_TRP = ("theta", "es", "td", "q", "tv")
SINGLE_PASS_TRP = ("theta", "td", "q", "ept", "wbpt")

_TM = {None: 0, "none": 0, "direct": 1, "bisect": 2, "newton": 3}


def _slots(table, outputs):
    try:
        return [table[o] for o in outputs]
    except KeyError as e:
        raise ValueError(f"unknown suite output {e.args[0]!r}; choose from {sorted(table)}") from None


def _ept_id(ept_method):
    return _EPT[ept_method]


def suite_tqp(t, q, p, outputs=DEFAULT_TQP, out=None, ept_method="ifs"):
    """One pass over (t, q, p) producing the requested fields; returns ``{name: tensor}``.

    ``ept_method`` ("ifs", "bolton35", "bolton39") is the formulation of the ``"ept"`` / ``"wbpt"`` outputs."""
    outputs = tuple(outputs)
    return _b.execute_suite("suite_tqp", (t, q, p), outputs, _slots(SUITE_TQP_OUTPUTS, outputs), out, _ept_id(ept_method))


def suite_ttdp(t, td, p, outputs=DEFAULT_TTDP, out=None, ept_method="ifs"):
    """One pass over (t, td, p) producing the requested fields; returns ``{name: tensor}``."""
    outputs = tuple(outputs)
    return _b.execute_suite("suite_ttdp", (t, td, p), outputs, _slots(SUITE_TTDP_OUTPUTS, outputs), out, _ept_id(ept_method))


def suite_trp(t, r, p, outputs=DEFAULT_TRP, out=None, ept_method="ifs"):
    """One pass over (t, r, p), ``r`` the relative humidity in %, producing the requested fields; returns ``{name: tensor}``.

    Each output is the reference chain named in ``SUITE_TRP_OUTPUTS``.  ``r = 0`` gives ``td = NaN``, as in the reference."""
    outputs = tuple(outputs)
    return _b.execute_suite("suite_trp", (t, r, p), outputs, _slots(SUITE_TRP_OUTPUTS, outputs), out, _ept_id(ept_method))


def suite_tqp_batch(ts, qs, ps, outputs=DEFAULT_TQP, out=None, ept_method="ifs"):
    """``suite_tqp`` over a LIST of separate fields (one tensor per level / member, each its own allocation) in one launch.

    ``ts`` / ``qs`` / ``ps`` are lists of same-shape contiguous CUDA tensors, or a Python number for a broadcast operand; ``ps``
    may also be a list of Python numbers, ONE PRESSURE PER FIELD -- pressure-level data, the reference user's loop
    ``for lev: potential_temperature(t[lev], p_lev)`` in one launch.  Returns ``[{name: tensor}, ...]``, one dict per field; every
    value is bit-identical to ``suite_tqp(ts[j], qs[j], ps[j])``.  A launch per 1 M-point level is bound by launch and pipeline-fill latency
    (12-16 us for 6 us of HBM time); one launch over all levels is not."""
    outputs = tuple(outputs)
    return _b.execute_suite_batch("suite_tqp_batch", (ts, qs, ps), outputs, _slots(SUITE_TQP_OUTPUTS, outputs), out, _ept_id(ept_method))


def suite_ttdp_batch(ts, tds, ps, outputs=DEFAULT_TTDP, out=None, ept_method="ifs"):
    """``suite_ttdp`` over a list of separate fields in one launch (see ``suite_tqp_batch``)."""
    outputs = tuple(outputs)
    return _b.execute_suite_batch("suite_ttdp_batch", (ts, tds, ps), outputs, _slots(SUITE_TTDP_OUTPUTS, outputs), out, _ept_id(ept_method))


def suite_trp_batch(ts, rs, ps, outputs=DEFAULT_TRP, out=None, ept_method="ifs"):
    """``suite_trp`` over a list of separate fields in one launch (see ``suite_tqp_batch``)."""
    outputs = tuple(outputs)
    return _b.execute_suite_batch("suite_trp_batch", (ts, rs, ps), outputs, _slots(SUITE_TRP_OUTPUTS, outputs), out, _ept_id(ept_method))


# Fields of fewer columns than this run a mixed call as the suite launch plus one geopotential_on_hybrid_levels launch per column
# output: the fused walk has one work item per tile of 256 threads x one 16-byte vector of columns (512 columns in float64, 1024 in
# float32), so a small field leaves most of the GPU idle, while the suite launch also splits the levels into work items.  Measured
# on B200, 5 outputs + z x 137 levels, fused / two launches (profiles/r03_kbench_geo_*.log): float64 0.91 at 65 536 columns, 1.20 at
# 32 768; float32 0.81 at 262 144, 1.05 at 131 072.
GEO_FUSED_MIN_COLUMNS = {"float64": 65536, "float32": 262144}


def _out_buffer(out, name, like):
    """out[name] when the caller preallocated it (checked), else a new tensor like `like`."""
    if out is not None and name in out:
        o = out[name]
        if o.dtype != like.dtype or o.shape != like.shape or not o.is_contiguous() or o.device != like.device:
            raise ValueError(f"suite_tq_hybrid: preallocated output {name!r} must be a contiguous {like.dtype} tensor of shape {tuple(like.shape)}")
        return o
    return torch.empty_like(like)


def suite_tq_hybrid(t, q, sp, A, B, outputs=DEFAULT_TQP, out=None, want_p=False, ept_method="ifs", zs=None, alpha_top="ifs", h_type="geometric",
                    h_reference="ground"):
    """The (t, q, p) suite on hybrid model levels with the pressure computed inside the kernel.

    ``t`` and ``q`` are ``[nlev, ...]`` fields, ``sp`` the surface pressure ``[...]``, ``A`` / ``B`` the ``nlev + 1``
    half-level coefficients.  Equals ``suite_tqp(t, q, p)`` with
    ``p = earthkit.meteo.vertical.pressure_on_hybrid_levels(A, B, sp, output="full")`` (reference
    vertical/array/vertical.py:663,708) -- but the ``[nlev, ...]`` pressure array is never written or read:
    56 instead of 64 bytes per point for the five default outputs.  ``want_p=True`` also returns it (key ``"p"``).

    ``outputs`` may also name the column outputs of ``COLUMN_OUTPUTS``, the geopotential of the same levels:
    ``"thickness"`` (``relative_geopotential_thickness_on_hybrid_levels``), ``"z"`` (``geopotential_on_hybrid_levels``) and
    ``"height"`` (``height_on_hybrid_levels`` with ``h_type`` / ``h_reference``: "geometric" or any other h_type for
    geopotential height, "ground" or "sea"), all with ``alpha_top`` ("ifs" / "arpege").  ``zs``, the surface geopotential (a
    tensor of ``sp.shape`` or a Python number), is needed by ``"z"`` and by every height except geopotential height above
    ground.  With suite outputs too, one kernel walks the columns and reads ``t`` and ``q`` once for both (64 instead of 80
    bytes per point for five suite outputs and ``"z"`` in float64).  The column outputs have the dtype of the field: they equal
    the ``ek_thermo.vertical`` functions called with ``A`` / ``B`` given as tensors of that dtype (not the float64 promotion
    those functions apply to Python-list ``A`` / ``B``).
    """
    outputs = tuple(outputs)
    alpha_top_value = _alpha_top_value(alpha_top)
    suite, cols, need_zs = _split_suite_outputs(outputs, h_type, h_reference, zs)
    slots = _slots(SUITE_TQP_OUTPUTS, suite)
    for x in (t, q, sp):
        if not isinstance(x, torch.Tensor):
            raise TypeError("suite_tq_hybrid: t, q and sp must be torch CUDA tensors")
    dev = _b._check_device([t, q, sp])
    dtype = t.dtype
    if dtype not in (torch.float64, torch.float32) or q.dtype != dtype or sp.dtype != dtype:
        raise TypeError("suite_tq_hybrid: t, q and sp must share one dtype (float64 or float32)")
    if t.shape != q.shape or t.dim() < 1 or tuple(t.shape[1:]) != tuple(sp.shape):
        raise ValueError(f"suite_tq_hybrid: expected t, q of shape (nlev,) + sp.shape, got {tuple(t.shape)}, {tuple(q.shape)}, {tuple(sp.shape)}")
    nlev, npl = int(t.shape[0]), int(sp.numel())
    a = torch.as_tensor(A, dtype=dtype, device=dev).contiguous()
    b = torch.as_tensor(B, dtype=dtype, device=dev).contiguous()
    if a.numel() != nlev + 1 or b.numel() != nlev + 1:
        raise ValueError(f"suite_tq_hybrid: A and B need nlev + 1 = {nlev + 1} half-level values")
    if need_zs:
        if isinstance(zs, torch.Tensor):
            _b._check_device([t, zs])
            if zs.dtype != dtype or zs.shape != sp.shape:
                raise ValueError(f"suite_tq_hybrid: zs must be a {dtype} tensor of shape {tuple(sp.shape)} or a Python number")
        elif not isinstance(zs, (int, float)) or isinstance(zs, bool):
            raise TypeError("suite_tq_hybrid: zs must be a torch CUDA tensor or a Python number")
    else:
        zs = None
    tc, qc, spc = t.contiguous(), q.contiguous(), sp.contiguous()
    ptrs = (c_void_p * _b.N_SUITE_SLOTS)()
    mask = 0
    res = {}
    em = _ept_id(ept_method)
    for name in outputs:
        res[name] = _out_buffer(out, name, tc)
    for name, k in zip(suite, slots):
        ptrs[k] = res[name].data_ptr()
        mask |= 1 << k
    p_ptr = None
    if want_p:
        res["p"] = _out_buffer(out, "p", tc)
        p_ptr = res["p"].data_ptr()
    if npl == 0:
        return res
    fused = bool(cols) and (bool(suite) or want_p) and npl >= GEO_FUSED_MIN_COLUMNS["float64" if dtype == torch.float64 else "float32"]
    if not fused and (suite or want_p or not cols):
        _b.call_raw("suite_tq_hybrid", dtype, dev, tc.data_ptr(), qc.data_ptr(), spc.data_ptr(), a.data_ptr(), b.data_ptr(), nlev, npl, ptrs, mask,
                    em, p_ptr)
    if not fused:
        for name, mode in cols.items():
            _column_kernel(tc, qc, mode, 0, sp=spc, A=a, B=b, alpha_top=alpha_top, zs=zs, out=res[name])
        return res
    zsc = None
    if zs is not None:
        zsc = zs.contiguous() if isinstance(zs, torch.Tensor) else torch.full(tuple(sp.shape), float(zs), dtype=dtype, device=dev)
    col_ptr = lambda n: res[n].data_ptr() if n in res else None  # noqa: E731
    _b.call_raw("suite_tq_hybrid_geo", dtype, dev, tc.data_ptr(), qc.data_ptr(), spc.data_ptr(), zsc.data_ptr() if zsc is not None else None,
                a.data_ptr(), b.data_ptr(), nlev, npl, ptrs, mask, em, p_ptr, _top_is_toa(a, b, 0, spc, dtype, dev), alpha_top_value,
                col_ptr("thickness"), col_ptr("z"), col_ptr("height"), cols.get("height", 0))
    return res


def ept_wet_bulb(t, h, p, humidity="q", ept_method="ifs", t_method="direct", potential=True, want_ept=True, want_wb=True):
    """Equivalent potential temperature and wet-bulb (potential) temperature in one pass.

    ``h`` is the specific humidity (``humidity="q"``) or the dewpoint (``"td"``).  Equals
    ``ept_from_*`` and ``wet_bulb[_potential]_temperature_from_*`` of the reference with the same
    ``ept_method`` / ``t_method``.  Returns ``(ept, wb)``, with None for an output not wanted.
    """
    if humidity not in ("q", "td"):
        raise ValueError(f"humidity={humidity!r} must be 'q' or 'td'")
    m = _EPT[ept_method]
    if t_method not in _TM or (t_method == "direct" and not potential):
        raise ValueError(f"temperature_on_moist_adiabat: invalid t_method={t_method} specified!")
    tm = _TM[t_method]
    if tm == 0:
        want_wb = False
    if not (want_ept or want_wb):
        raise ValueError("nothing to compute")
    res = _b.execute("ept_wet_bulb", (t, h, p), (int(humidity == "q"), m, tm, int(bool(potential))), want=(want_ept, want_wb))
    if want_ept and want_wb:
        return res
    return (res, None) if want_ept else (None, res)
