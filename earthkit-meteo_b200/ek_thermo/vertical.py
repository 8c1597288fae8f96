"""``ek_thermo.vertical`` -- hybrid (IFS model) level pressure on torch CUDA tensors (SURVEY.md 8(f)-1).

Drop-in for ``earthkit.meteo.vertical.pressure_on_hybrid_levels`` (reference
src/earthkit/meteo/vertical/array/vertical.py:505-737, "V"): same signature, defaults, outputs and exceptions.
One kernel launch reads ``sp`` once and writes every requested [level, point] array from registers.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _backend as _b

_OUTPUTS = ("full", "half", "alpha", "delta")


def _dtype_of(x):
    """The dtype an argument contributes to numpy-style promotion: tensors and numpy arrays their own, a Python list /
    tuple float64 (``xp.asarray([...])`` in the reference makes a float64 array, V:630-631), a Python number nothing
    (numpy-2 weak scalars)."""
    if x is None or isinstance(x, (int, float)):
        return None
    if isinstance(x, torch.Tensor):
        return x.dtype
    dt = getattr(x, "dtype", None)
    if dt is not None:
        try:
            return getattr(torch, str(dt))
        except (AttributeError, TypeError):
            return torch.float64
    return torch.float64


def _working_dtype(*xs):
    """float64 / float32 by the reference's (numpy) promotion over every array argument: a float64 operand among float32
    ones promotes the computation, it is never cast down."""
    dtype = None
    for x in xs:
        d = _dtype_of(x)
        if d is None:
            continue
        if not d.is_floating_point:
            d = torch.float64
        dtype = d if dtype is None else torch.promote_types(dtype, d)
    return torch.float32 if dtype in (torch.float32, torch.float16, torch.bfloat16) else torch.float64


def _coeff_tensors(A, B, dtype, device):
    a = torch.as_tensor(A, dtype=dtype, device=device).contiguous()
    b = torch.as_tensor(B, dtype=dtype, device=device).contiguous()
    if a.dim() != 1 or a.shape != b.shape or a.numel() < 2:
        raise ValueError("A and B must be 1-D arrays of the same size (one value per half-level, at least 2)")
    return a, b


def _top_is_toa(a, b, top_half, spc, dtype, dev):
    """V:678: does ANY point have p_half[top] <= 0.1 Pa?  A constant when B[top] == 0, else a one-flag reduction kernel -- or, for
    a host (numpy) ``spc`` with ``a`` / ``b`` of its dtype, the same comparison on the host."""
    a_top, b_top = float(a[top_half]), float(b[top_half])
    host = isinstance(spc, np.ndarray)
    if b_top == 0.0 or (spc.size if host else spc.numel()) == 0:
        return int(a_top <= 0.1)
    if host:
        return int(np.any(a[top_half] + b[top_half] * spc <= spc.dtype.type(0.1)))
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    _b.call_raw("hybrid_top_is_toa", dtype, dev, spc.data_ptr(), spc.numel(), a_top, b_top, flag.data_ptr())
    return int(flag.item())


def _alpha_top_value(alpha_top):
    """alpha of the top level when its upper half level is the top of the atmosphere: ln 2 for "ifs", 1 for "arpege" (V:669)."""
    if alpha_top not in ("ifs", "arpege"):
        raise ValueError(f"Unknown method '{alpha_top}' for pressure calculation. Use 'ifs' or 'arpege'.")  # V:626-627
    return math.log(2.0) if alpha_top == "ifs" else 1.0


def pressure_on_hybrid_levels(A, B, sp, levels=None, alpha_top="ifs", output="full", vertical_axis=0):
    """Pressure on full / half levels, ``delta`` and ``alpha`` of hybrid levels.  Reference V:505-737.

    ``sp`` is a torch CUDA tensor (float64 / float32) of any shape; ``A`` / ``B`` are array-likes with one value per
    half-level.  Returns a tensor or a tuple of tensors shaped ``(levels,) + sp.shape`` (vertical axis moved to
    ``vertical_axis``).  dtype as in the reference: the numpy promotion of ``sp``, ``A`` and ``B`` (Python lists count as
    float64); ``alpha`` / ``delta`` are always float64 arrays (V:672,686).
    """
    if isinstance(output, str):
        output = (output,)
    if not output:
        raise ValueError("At least one output type must be specified.")  # V:617-618
    for out in output:
        if out not in _OUTPUTS:
            raise ValueError(f"Unknown output type '{out}'. Allowed values are 'full', 'half', 'alpha' or 'delta'.")  # V:620-624
    alpha_top_value = _alpha_top_value(alpha_top)
    if not isinstance(sp, torch.Tensor):
        raise TypeError("ek_thermo.vertical: sp must be a torch CUDA tensor (no CPU path; use earthkit.meteo.vertical for host arrays)")
    dev = _b._check_device([sp])
    dtype = _working_dtype(sp, A, B)  # V:630-663: A + B * sp promotes as numpy does
    spc = sp.to(dtype).contiguous()
    a, b = _coeff_tensors(A, B, dtype, dev)
    nhalf = a.numel()
    nlev = nhalf - 1
    if levels is not None:  # V:634-654
        lv = [int(x) for x in (levels.tolist() if hasattr(levels, "tolist") else list(levels))]
        lmax, lmin = max(lv), min(lv)
        if lmax > nlev:
            raise ValueError(f"Requested level {lmax} exceeds the maximum number of levels {nlev}.")
        if lmin < 1:
            raise ValueError(f"Level numbering starts at 1. Found level={lmin} < 1.")
        full_rows, half_rows, top_k = [x - 1 for x in lv], lv, lmin - 1
    else:
        full_rows, half_rows, top_k = list(range(nlev)), list(range(nhalf)), 0
    want = {o: True for o in output}
    npl = spc.numel()
    top_toa = 0
    if "delta" in want or "alpha" in want:  # V:678: one decision for the whole field
        top_toa = _top_is_toa(a, b, top_k, spc, dtype, dev)
    rows_f = torch.tensor(full_rows, dtype=torch.int32, device=dev)
    rows_h = torch.tensor(half_rows, dtype=torch.int32, device=dev)
    res = {}
    for name in _OUTPUTS:
        if name in want:
            nrow = len(half_rows) if name == "half" else len(full_rows)
            # alpha / delta: xp.zeros(...) arrays in the reference, i.e. always float64 (V:672,686); the kernel widens on store
            odt = torch.float64 if name in ("alpha", "delta") else dtype
            res[name] = torch.empty((nrow,) + tuple(sp.shape), dtype=odt, device=dev)
    ptr = lambda n: res[n].data_ptr() if n in res else None  # noqa: E731
    if npl > 0:
        _b.call_raw("pressure_on_hybrid_levels", dtype, dev, a.data_ptr(), b.data_ptr(), nhalf, spc.data_ptr(), npl, rows_f.data_ptr(),
                    len(full_rows), rows_h.data_ptr(), len(half_rows), top_k, top_toa, alpha_top_value, ptr("full"), ptr("half"), ptr("delta"),
                    ptr("alpha"), 1)
    outs = [res[o] for o in output]
    if vertical_axis != 0 and outs[0].dim() > 1:  # V:731-733
        outs = [r.movedim(0, vertical_axis) for r in outs]
    return outs[0] if len(outs) == 1 else tuple(outs)


# --------------------------------------------------------------------------------------------------------------------
# SURVEY.md 8(f)-2: geopotential thickness / geopotential / height on hybrid levels (V:741-1188)
# --------------------------------------------------------------------------------------------------------------------
_HM = {"thickness": 0, "geopotential": 1, ("geopotential", "sea"): 2, ("geopotential", "ground"): 3, ("geometric", "sea"): 4,
       ("geometric", "ground"): 5}


def _adds_zs(mode):
    """Does height form `mode` add the surface geopotential zs?  All but the thickness and geopotential height above ground (V:1186)."""
    return mode != _HM["thickness"] and mode != _HM[("geopotential", "ground")]


def _column_kernel(t, q, mode, vertical_axis, sp=None, A=None, B=None, alpha_top="ifs", alpha=None, delta=None, zs=None, out=None):
    """Output form `mode` of the geopotential thickness, one kernel launch.  Computed in the numpy promotion of every array
    argument; returned in the reference's dtype: the thickness lives in ``zeros_like(R(q) * t)`` (V:806), so its dtype is
    that of ``t`` / ``q``, and the forms that add ``np.asarray(zs)`` promote it with ``zs`` (a Python number: float64).  A float64
    computation for float32 ``t`` / ``q`` is rounded once on the way out, as the reference's assignment rounds it.  ``out``, when
    given, receives the working-dtype result as it is."""
    for x in (t, q):
        if not isinstance(x, torch.Tensor):
            raise TypeError("ek_thermo.vertical: t and q must be torch CUDA tensors (no CPU path)")
    tensors = [x for x in (t, q, sp, alpha, delta, zs) if isinstance(x, torch.Tensor)]
    dev = _b._check_device(tensors)
    dtype = _working_dtype(t, q, sp, alpha, delta, zs, A, B)  # numpy promotion over every array argument, never a down-cast
    out_dtype = _working_dtype(t, q)
    if _adds_zs(mode):  # the reference adds np.asarray(zs): a Python number is a float64 array there
        out_dtype = torch.float64 if isinstance(zs, (int, float)) else _working_dtype(t, q, zs)
    if t.shape != q.shape or t.dim() < 1:
        raise ValueError(f"t and q must have the same shape, got {tuple(t.shape)} and {tuple(q.shape)}")
    if vertical_axis != 0:  # V:878-883: work with the vertical axis first
        t, q = t.movedim(vertical_axis, 0), q.movedim(vertical_axis, 0)
        if alpha is not None:
            alpha, delta = alpha.movedim(vertical_axis, 0), delta.movedim(vertical_axis, 0)
    tc, qc = t.to(dtype).contiguous(), q.to(dtype).contiguous()
    nlev = int(tc.shape[0])
    col_shape = tuple(tc.shape[1:])
    npl = int(tc[0].numel()) if nlev else 0
    keep = []

    def col(x, name):  # a per-column field (sp, zs): broadcast to the column shape
        x = torch.as_tensor(x, dtype=dtype, device=dev)
        if tuple(x.shape) != col_shape:
            x = x.expand(col_shape)
        x = x.contiguous()
        keep.append(x)
        return x.data_ptr()

    p_sp = p_a = p_b = p_al = p_de = p_zs = None
    nhalf = top_toa = 0
    alpha_top_value = _alpha_top_value(alpha_top)
    if alpha is not None:
        if alpha.shape != t.shape or delta.shape != t.shape:  # numpy broadcasting of d * alpha, d * delta into zeros_like(d) (V:804-810)
            try:
                alpha, delta = alpha.expand(t.shape), delta.expand(t.shape)
            except RuntimeError:
                raise ValueError(f"operands could not be broadcast together with shapes {tuple(t.shape)} {tuple(alpha.shape)}") from None
        ac, dc = alpha.to(dtype).contiguous(), delta.to(dtype).contiguous()
        keep += [ac, dc]
        p_al, p_de = ac.data_ptr(), dc.data_ptr()
    else:
        a, b = _coeff_tensors(A, B, dtype, dev)
        nhalf = a.numel()
        if nlev > nhalf - 1:
            raise ValueError(f"Requested level {nlev} exceeds the maximum number of levels {nhalf - 1}.")
        keep += [a, b]
        p_a, p_b, p_sp = a.data_ptr(), b.data_ptr(), col(sp, "sp")
        top_toa = _top_is_toa(a, b, nhalf - 1 - nlev, keep[-1], dtype, dev)  # the band is the nlev bottom-most levels (V:1191-1203)
    if _adds_zs(mode):
        p_zs = col(zs, "zs")
    own = out is None
    if own:
        out = torch.empty_like(tc)
    if npl > 0 and nlev > 0:
        _b.call_raw("geopotential_on_hybrid_levels", dtype, dev, tc.data_ptr(), qc.data_ptr(), nlev, npl, p_sp, p_a, p_b, nhalf, top_toa,
                    alpha_top_value, p_al, p_de, p_zs, mode, out.data_ptr())
    del keep
    if own and out.dtype != out_dtype:
        out = out.to(out_dtype)
    return out.movedim(0, vertical_axis) if vertical_axis != 0 else out


def relative_geopotential_thickness_on_hybrid_levels_from_alpha_delta(t, q, alpha, delta, vertical_axis=0):
    """Geopotential thickness between the surface and the full levels, from precomputed alpha/delta.  Reference V:815-891.
    Returned in the dtype of ``t`` / ``q`` whatever the dtype of alpha / delta (the reference's ``zeros_like(d)``)."""
    return _column_kernel(t, q, 0, vertical_axis, alpha=alpha, delta=delta)


def _thickness_axis_as_reference(t, q, A, B, sp, alpha_top, vertical_axis):
    """``vertical_axis != 0`` exactly as the reference computes it (V:970-994): alpha / delta come out of
    ``pressure_on_hybrid_levels`` with their level axis FIRST and are then moved with ``moveaxis(x, vertical_axis, 0)`` like
    t and q -- a second move.  That is shape-consistent only for square fields (as many columns as levels), where it
    scrambles alpha / delta; any other shape fails numpy's broadcast check and raises ``ValueError``.  Replicated, not fixed
    (SURVEY.md 7.3-H5); pinned by the live-reference fixture tests/golden/ref_hybrid_axis.npz."""
    if not isinstance(t, torch.Tensor):
        raise TypeError("ek_thermo.vertical: t and q must be torch CUDA tensors (no CPU path)")
    a_len = len(A)
    nlev_t, nlev = int(t.shape[vertical_axis]), a_len - 1
    levels = None if nlev_t == nlev else list(range(nlev - nlev_t + 1, nlev + 1))  # V:1191-1203
    alpha, delta = pressure_on_hybrid_levels(A, B, sp, alpha_top=alpha_top, levels=levels, output=("alpha", "delta"))
    return _column_kernel(t, q, 0, vertical_axis, alpha=alpha, delta=delta)  # moves t, q, alpha and delta alike (V:981-986)


def _height_form(dphi, zs, mode):
    """Output form `mode` of a thickness already in memory, with numpy's broadcasting of zs (and its ValueError).  Geopotential
    height above ground does not read zs in the reference (V:1186), so there zs neither broadcasts nor promotes."""
    if not _adds_zs(mode):
        return _b.execute("height_from_thickness", (dphi, 0.0), (mode,))
    # np.asarray(zs) in the reference: a Python number is a float64 array, an array keeps its dtype
    zs_t = torch.as_tensor(zs, dtype=torch.float64 if isinstance(zs, (int, float)) else None, device=dphi.device)
    try:
        torch.broadcast_shapes(tuple(dphi.shape), tuple(zs_t.shape))
    except RuntimeError:
        raise ValueError(f"operands could not be broadcast together with shapes {tuple(dphi.shape)} {tuple(zs_t.shape)}") from None
    return _b.execute("height_from_thickness", (dphi, zs_t), (mode,))


def geopotential_height_from_geopotential(z):
    """z / g.  Reference V:330-353."""
    return _b.execute("height_from_thickness", (z, 0.0), (3,))


def geometric_height_from_geopotential(z):
    """R z/g / (R - z/g) with the reference's Earth radius.  Reference V:472-502."""
    return _b.execute("height_from_thickness", (z, 0.0), (6,))


def relative_geopotential_thickness_on_hybrid_levels(t, q, A, B, sp, alpha_top="ifs", vertical_axis=0):
    """Same, with alpha/delta computed inside the kernel from sp and A/B (never materialised).  Reference V:894-994.

    Computed in the numpy promotion of every argument (float64 for Python-list ``A`` / ``B``); returned in the reference's dtype,
    that of ``t`` / ``q``.  ``geopotential_on_hybrid_levels`` and ``height_on_hybrid_levels`` return that dtype promoted with
    ``zs`` where they add it (a Python number counts as float64, as ``np.asarray(zs)`` in the reference).

    ``t``/``q`` may hold only the bottom-most contiguous levels of the model (V:1191-1203).  ``vertical_axis != 0`` behaves as
    in the reference (see ``_thickness_axis_as_reference``)."""
    if vertical_axis != 0:
        return _thickness_axis_as_reference(t, q, A, B, sp, alpha_top, vertical_axis)
    return _column_kernel(t, q, 0, vertical_axis, sp=sp, A=A, B=B, alpha_top=alpha_top)


def geopotential_on_hybrid_levels(t, q, zs, A, B, sp, alpha_top="ifs", vertical_axis=0):
    """Geopotential on the full levels: thickness + surface geopotential, one kernel.  Reference V:997-1069."""
    if vertical_axis != 0:
        return _height_form(_thickness_axis_as_reference(t, q, A, B, sp, alpha_top, vertical_axis), zs, 1)
    return _column_kernel(t, q, 1, vertical_axis, sp=sp, A=A, B=B, alpha_top=alpha_top, zs=zs)


def _height_mode(h_type, h_reference):
    """The EK_HM_* form of height_on_hybrid_levels' h_type / h_reference (V:1163-1188)."""
    if h_reference not in ["sea", "ground"]:
        raise ValueError(f"Unknown '{h_reference=}'. Use 'sea' or 'ground'.")  # V:1163-1164
    return _HM[("geometric" if h_type == "geometric" else "geopotential", h_reference)]  # any other h_type -> geopotential (V:1175-1186)


# column outputs of fused.suite_tq_hybrid and hostpipe.HostSuite.suite_tq_hybrid: the geopotential of the suite's levels, from the
# same walk of the columns
COLUMN_OUTPUTS = (
    "thickness",  # relative_geopotential_thickness_on_hybrid_levels(t, q, A, B, sp, alpha_top)                      V:894-994
    "z",  # geopotential_on_hybrid_levels(t, q, zs, A, B, sp, alpha_top)                                            V:997-1069
    "height",  # height_on_hybrid_levels(t, q, zs, A, B, sp, alpha_top, h_type, h_reference)                        V:1072-1188
)


def _split_suite_outputs(outputs, h_type, h_reference, zs):
    """``outputs`` of a hybrid-level suite call as (suite outputs, {column output: height mode}, whether zs is read).  Raises
    ValueError when a column output needs zs and none is given."""
    modes = dict(zip(COLUMN_OUTPUTS, (_HM["thickness"], _HM["geopotential"], _height_mode(h_type, h_reference))))
    suite = tuple(o for o in outputs if o not in modes)
    cols = {o: modes[o] for o in outputs if o in modes}
    need_zs = any(_adds_zs(m) for m in cols.values())
    if need_zs and zs is None:
        raise ValueError("suite_tq_hybrid: 'z' and every 'height' except geopotential height above ground need the surface geopotential zs")
    return suite, cols, need_zs


def height_on_hybrid_levels(t, q, zs, A, B, sp, alpha_top="ifs", h_type="geometric", h_reference="ground", vertical_axis=0):
    """Geometric / geopotential height above sea level / ground, one kernel.  Reference V:1072-1188."""
    mode = _height_mode(h_type, h_reference)
    if vertical_axis != 0:
        return _height_form(_thickness_axis_as_reference(t, q, A, B, sp, alpha_top, vertical_axis), zs, mode)
    return _column_kernel(t, q, mode, vertical_axis, sp=sp, A=A, B=B, alpha_top=alpha_top, zs=zs)
