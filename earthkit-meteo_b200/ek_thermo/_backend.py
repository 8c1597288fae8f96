"""ctypes binding of libek_thermo.so and the generic "launch one entry point" helper.

PyTorch is used for tensor handles, allocation and streams only.  There is NO CPU path: if the
shared library is missing, or an argument is not a CUDA tensor, the call fails loudly.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_int, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = os.environ.get("EK_THERMO_LIB", "libek_thermo.so")
LIB_PATH = LIB_NAME if os.path.isabs(LIB_NAME) else os.path.join(_HERE, LIB_NAME)


class ek_operand(ctypes.Structure):
    """Mirror of ``struct ek_operand`` (include/ek_thermo.h): device pointer or broadcast scalar."""

    _fields_ = [("ptr", c_void_p), ("value", c_double)]


class EkThermoError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"ek_thermo: CUDA library {LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C earthkit-meteo_b200/csrc`. There is no CPU fallback."
    )
_lib = ctypes.CDLL(LIB_PATH)
_lib.ek_thermo_version.restype = c_int
_lib.ek_thermo_last_error.restype = ctypes.c_char_p
_lib.ek_thermo_launch_count.restype = c_uint64
_lib.ek_thermo_set_launch_config.argtypes = [c_int, c_int]
_lib.ek_thermo_shard_range.argtypes = [c_int64, c_int, c_int, c_int64, ctypes.POINTER(c_int64), ctypes.POINTER(c_int64)]

_SUFFIX = {torch.float64: "f64", torch.float32: "f32"}
_TORCH = {np.dtype("float64"): torch.float64, np.dtype("float32"): torch.float32}  # the host-array dtypes and their tensor dtypes
# ept_method -> EK_EPT_* (T:1319-1323); an unknown method is a KeyError, as in the reference (T:1024-1026)
_EPT = {"ifs": 0, "bolton35": 1, "bolton39": 2}

# option kinds of every entry point, in C argument order:  operands..., options..., outputs..., n, stream
# name -> (n_inputs, option ctypes, n_outputs)
SIGNATURES = {
    "celsius_to_kelvin": (1, (), 1),
    "kelvin_to_celsius": (1, (), 1),
    "specific_humidity_from_mixing_ratio": (1, (), 1),
    "mixing_ratio_from_specific_humidity": (1, (), 1),
    "vapour_pressure_from_specific_humidity": (2, (), 1),
    "vapour_pressure_from_mixing_ratio": (2, (), 1),
    "specific_humidity_from_vapour_pressure": (2, (c_double,), 1),
    "mixing_ratio_from_vapour_pressure": (2, (c_double,), 1),
    "saturation_vapour_pressure": (1, (c_int,), 1),
    "saturation_vapour_pressure_slope": (1, (c_int,), 1),
    "saturation_mixing_ratio": (2, (c_int,), 1),
    "saturation_specific_humidity": (2, (c_int,), 1),
    "saturation_mixing_ratio_slope": (4, (c_int, c_int, c_int, c_double), 1),
    "saturation_specific_humidity_slope": (4, (c_int, c_int, c_int, c_double), 1),
    "temperature_from_saturation_vapour_pressure": (1, (), 1),
    "relative_humidity_from_dewpoint": (2, (), 1),
    "relative_humidity_from_specific_humidity": (3, (), 1),
    "specific_humidity_from_dewpoint": (2, (), 1),
    "mixing_ratio_from_dewpoint": (2, (), 1),
    "specific_humidity_from_relative_humidity": (3, (), 1),
    "dewpoint_from_relative_humidity": (2, (), 1),
    "dewpoint_from_specific_humidity": (2, (), 1),
    "virtual_temperature": (2, (), 1),
    "virtual_potential_temperature": (3, (), 1),
    "potential_temperature": (2, (), 1),
    "temperature_from_potential_temperature": (2, (), 1),
    "pressure_on_dry_adiabat": (3, (), 1),
    "temperature_on_dry_adiabat": (3, (), 1),
    "lcl_temperature": (2, (c_int,), 1),
    "lcl": (3, (c_int,), 2),
    "specific_gas_constant": (1, (), 1),
    "ept_from_dewpoint": (3, (c_int,), 1),
    "ept_from_specific_humidity": (3, (c_int,), 1),
    "saturation_ept": (2, (c_int,), 1),
    "temperature_on_moist_adiabat": (2, (c_int, c_int), 1),
    "wet_bulb_temperature_from_dewpoint": (3, (c_int, c_int), 1),
    "wet_bulb_temperature_from_specific_humidity": (3, (c_int, c_int), 1),
    "wet_bulb_potential_temperature_from_dewpoint": (3, (c_int, c_int), 1),
    "wet_bulb_potential_temperature_from_specific_humidity": (3, (c_int, c_int), 1),
    "ept_wet_bulb": (3, (c_int, c_int, c_int, c_int), 2),
    # wind (SURVEY.md 8(f)-3)
    "wind_speed": (2, (), 1),
    "wind_direction": (2, (c_int, c_int), 1),
    "wind_xy_to_polar": (2, (c_int,), 2),
    "wind_polar_to_xy": (2, (c_int,), 2),
    "w_from_omega": (3, (), 1),
    "coriolis": (1, (), 1),
    # height forms of a geopotential (SURVEY.md 8(f)-2)
    "height_from_thickness": (2, (c_int,), 1),
}

for _name, (_nin, _opts, _nout) in SIGNATURES.items():
    for _sfx in ("f64", "f32"):
        _fn = getattr(_lib, f"ek_thermo_{_name}_{_sfx}")
        _fn.argtypes = [ek_operand] * _nin + list(_opts) + [c_void_p] * _nout + [c_int64, c_void_p]
        _fn.restype = c_int
for _name in ("suite_tqp", "suite_ttdp", "suite_trp"):
    for _sfx in ("f64", "f32"):
        _fn = getattr(_lib, f"ek_thermo_{_name}_{_sfx}")
        _fn.argtypes = [ek_operand] * 3 + [ctypes.POINTER(c_void_p), c_uint32, c_int, c_int64, c_void_p]
        _fn.restype = c_int
for _name in ("suite_tqp_batch", "suite_ttdp_batch", "suite_trp_batch"):
    for _sfx in ("f64", "f32"):
        _fn = getattr(_lib, f"ek_thermo_{_name}_{_sfx}")
        _fn.argtypes = [c_int, c_void_p, c_void_p, c_void_p, ctypes.POINTER(c_double), ctypes.POINTER(c_double), ctypes.POINTER(c_void_p), c_uint32, c_int,
                        c_int64, c_void_p]
        _fn.restype = c_int
_c_int_p = ctypes.POINTER(c_int)
for _sfx in ("f64", "f32"):
    _fn = getattr(_lib, f"ek_thermo_pressure_on_hybrid_levels_{_sfx}")
    _fn.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_double,
                    c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]
    _fn.restype = c_int
    _fn = getattr(_lib, f"ek_thermo_hybrid_top_is_toa_{_sfx}")
    _fn.argtypes = [c_void_p, c_int64, c_double, c_double, c_void_p, c_void_p]
    _fn.restype = c_int
    _fn = getattr(_lib, f"ek_thermo_geopotential_on_hybrid_levels_{_sfx}")
    _fn.argtypes = [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_void_p, c_void_p,
                    c_int, c_void_p, c_void_p]
    _fn.restype = c_int
    _fn = getattr(_lib, f"ek_thermo_suite_tq_hybrid_{_sfx}")
    _fn.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, ctypes.POINTER(c_void_p), c_uint32, c_int, c_void_p,
                    c_void_p]
    _fn.restype = c_int
    _fn = getattr(_lib, f"ek_thermo_suite_tq_hybrid_geo_{_sfx}")
    _fn.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, ctypes.POINTER(c_void_p), c_uint32, c_int, c_void_p,
                    c_int, c_double, c_void_p, c_void_p, c_void_p, c_int, c_void_p]
    _fn.restype = c_int
for _sfx in ("f64", "f32"):
    _fn = getattr(_lib, f"ek_thermo_host_suite_{_sfx}")
    _fn.argtypes = [c_int, c_void_p, c_void_p, c_void_p, ctypes.POINTER(c_void_p), c_uint32, c_int, c_int64, c_void_p, c_size_t, c_int]
    _fn.restype = c_int
    _fn = getattr(_lib, f"ek_thermo_host_suite_tq_hybrid_{_sfx}")
    _fn.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, ctypes.POINTER(c_void_p), c_uint32, c_int, c_void_p,
                    c_size_t, c_int]
    _fn.restype = c_int
    _fn = getattr(_lib, f"ek_thermo_host_suite_tq_hybrid_geo_{_sfx}")
    _fn.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, ctypes.POINTER(c_void_p), c_uint32, c_int, c_int,
                    c_double, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_int]
    _fn.restype = c_int


def version() -> int:
    return int(_lib.ek_thermo_version())


def launch_count() -> int:
    """Kernels launched by the library since it was loaded."""
    return int(_lib.ek_thermo_launch_count())


def set_launch_config(threads: int = 0, ctas_per_sm: int = 0) -> None:
    _check(_lib.ek_thermo_set_launch_config(threads, ctas_per_sm))


def _check(rc: int) -> None:
    if rc == 0:
        return
    msg = (_lib.ek_thermo_last_error() or b"").decode()
    if rc == -3:  # EK_ERR_EPS: the reference raises ValueError (T:189-190)
        raise ValueError(msg)
    if rc < 0:
        raise ValueError(f"ek_thermo: {msg} (code {rc})")
    raise EkThermoError(f"ek_thermo: {msg} (cudaError {rc})")


# ----------------------------------------------------------------------------------------------
# argument preparation
# ----------------------------------------------------------------------------------------------
def _check_device(tensors):
    """Every array argument must be a CUDA tensor on one device.  No CPU path exists."""
    dev = None
    for t in tensors:
        if not t.is_cuda:
            raise TypeError(
                "ek_thermo: got a CPU tensor. This package only runs on CUDA tensors (no CPU fallback); "
                "use earthkit.meteo.thermo for host arrays."
            )
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise ValueError(f"ek_thermo: tensors are on different devices ({dev} and {t.device})")
    return dev


_Tensor = torch.Tensor


def _on_device(t):
    return t.is_cuda


def _prepare(args):
    """Operands of a launch.  Fast path for the normal whole-field call -- every array argument a contiguous CUDA tensor
    of one dtype (float64 / float32), shape and device, the rest Python numbers -- and `_prepare_general` for everything
    else (broadcasting, promotion, non-contiguous views, errors).  The eager call of a 1 M-point field is bound by this
    host code, not by the kernel."""
    first = None
    ops = []
    for a in args:
        if isinstance(a, _Tensor):
            if first is None:
                first = a
                dtype = a.dtype
                shape = a.shape
                dev = a.device
                if dtype not in _SUFFIX:
                    return _prepare_general(args)
            elif a.dtype != dtype or a.shape != shape or a.device != dev:
                return _prepare_general(args)
            if not a.is_contiguous():
                return _prepare_general(args)
            ops.append(ek_operand(a.data_ptr(), 0.0))
        elif type(a) is float:
            ops.append(ek_operand(None, a))
        else:
            return _prepare_general(args)
    if first is None or not _on_device(first):
        return _prepare_general(args)  # raises the TypeError of the no-CPU-path rule
    return ops, (), dtype, dev, shape, first.numel()


def _prepare_general(args):
    """Split positional array-likes into (tensors | python scalars), find dtype, device, broadcast shape."""
    items = []
    tensors = []
    for a in args:
        if isinstance(a, torch.Tensor):
            items.append(a)
            tensors.append(a)
        elif isinstance(a, (int, float)) and not isinstance(a, bool):
            items.append(float(a))
        elif a is None:
            items.append(None)
        else:
            raise TypeError(
                f"ek_thermo: unsupported argument type {type(a).__name__}; expected torch CUDA tensors or Python numbers "
                "(numpy / host arrays are served by earthkit.meteo.thermo, there is no CPU path here)"
            )
    if not tensors:
        raise TypeError("ek_thermo: at least one argument must be a torch CUDA tensor")
    dev = _check_device(tensors)
    first = tensors[0]
    dtype, shape = first.dtype, first.shape
    uniform = True  # fast path: same dtype, same shape, contiguous -- the normal whole-field call
    for t in tensors:
        if t.dtype != dtype or t.shape != shape or not t.is_contiguous():
            uniform = False
            break
    if not uniform:
        for t in tensors[1:]:
            dtype = torch.promote_types(dtype, t.dtype)
        shape = torch.broadcast_shapes(*[t.shape for t in tensors])
    if dtype not in _SUFFIX:
        uniform = False
        dtype = torch.float64 if not dtype.is_floating_point else (torch.float32 if dtype in (torch.float16, torch.bfloat16) else dtype)
    n = first.numel() if uniform else int(torch.Size(shape).numel())
    ops = []
    keep = []
    for it in items:
        if it is None:
            ops.append(ek_operand(None, 0.0))
        elif isinstance(it, float):
            ops.append(ek_operand(None, it))
        elif uniform:
            ops.append(ek_operand(it.data_ptr(), 0.0))
        else:
            t = it
            if t.numel() == 1 and n > 1:
                ops.append(ek_operand(None, float(t.item())))  # broadcast by value, never materialised
                continue
            if t.dtype != dtype:
                t = t.to(dtype)
            if t.shape != shape:
                t = t.expand(shape)
            if not t.is_contiguous():
                t = t.contiguous()
            keep.append(t)
            ops.append(ek_operand(t.data_ptr(), 0.0))
    return ops, keep, dtype, dev, shape, n


# torch's raw accessors (no Stream / device objects built per call): the eager ERA5-level call is bound by host time
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)
_FN_CACHE = {}


def _stream_ptr(device):
    if _raw_stream is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


def _call(symbol: str, dtype, device, c_args):
    """The one place where the C ABI is entered.  (Tests patch this to check the host logic on CPU.)"""
    fn = _FN_CACHE.get((symbol, dtype))
    if fn is None:
        fn = _FN_CACHE[(symbol, dtype)] = getattr(_lib, f"ek_thermo_{symbol}_{_SUFFIX[dtype]}")
    cur = _raw_device() if _raw_device is not None else torch.cuda.current_device()
    if cur == device.index:  # the usual case: no device switch needed
        rc = fn(*c_args, _stream_ptr(device))
        if rc != 0:
            _check(rc)
        return
    with torch.cuda.device(device):
        _check(fn(*c_args, _stream_ptr(device)))


def call_raw(symbol: str, dtype, device, *c_args):
    """Entry points whose argument list does not follow the operands/options/outputs pattern (stream appended)."""
    _call(symbol, dtype, device, list(c_args))


def _empty(shape, dtype, device):
    return torch.empty(shape, dtype=dtype, device=device)


def execute(symbol: str, args, options=(), want=None):
    """Run entry point `symbol` on positional array args; returns a tensor or a tuple of tensors.

    `want` optionally selects which outputs to allocate (tuple of bools), for the two-output kernels.
    Pointers, sizes and options are handed to ctypes as plain ints (the entry points' argtypes convert them).
    """
    nin, opt_types, nout = SIGNATURES[symbol]
    assert len(args) == nin and len(options) == len(opt_types), symbol
    ops, keep, dtype, dev, shape, n = _prepare(args)
    if nout == 1:  # the common case: one output, no selection
        o = torch.empty(shape, dtype=dtype, device=dev)
        if n > 0:  # empty in -> empty out, nothing to launch (empty tensors have a NULL data_ptr)
            _call(symbol, dtype, dev, [*ops, *options, o.data_ptr(), n])
        del keep
        return o
    if want is None:
        want = (True,) * nout
    outs = [_empty(shape, dtype, dev) if w else None for w in want]
    c_args = [*ops, *options]
    c_args += [o.data_ptr() if o is not None else None for o in outs]
    c_args.append(n)
    if n > 0:
        _call(symbol, dtype, dev, c_args)
    del keep
    res = tuple(o for o in outs if o is not None)
    return res[0] if len(res) == 1 else res


N_SUITE_SLOTS = 10  # EK_S_NSLOTS (include/ek_thermo.h)


def execute_suite(symbol: str, args, out_names, slots, out=None, ept_method=0):
    """Run a fused suite; `slots` are the output slot numbers wanted; returns {name: tensor}."""
    ops, keep, dtype, dev, shape, n = _prepare(args)
    ptrs = (c_void_p * N_SUITE_SLOTS)()
    mask = 0
    res = {}
    for name, k in zip(out_names, slots):
        t = out.get(name) if out is not None else None
        if t is not None:
            if t.dtype != dtype or t.shape != shape or not t.is_contiguous() or t.device != dev:
                raise ValueError(f"ek_thermo: preallocated output {name!r} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {dev}")
        else:
            t = torch.empty(shape, dtype=dtype, device=dev)
        res[name] = t
        ptrs[k] = t.data_ptr()
        mask |= 1 << k
    if n > 0:
        _call(symbol, dtype, dev, [*ops, ptrs, mask, ept_method, n])
    del keep
    return res


def execute_suite_batch(symbol: str, seg_args, out_names, slots, outs=None, ept_method=0):
    """Run a fused suite over a list of separate fields in one launch.  seg_args: three items, each a list of same-shape
    contiguous CUDA tensors (one per field) or a Python number (broadcast); the LAST item may also be a list of Python numbers,
    one per field (pressure-level data: one pressure per level).  Returns a list of {name: tensor}, one per field."""
    def _numbers(a):
        return isinstance(a, (list, tuple)) and len(a) > 0 and all(isinstance(v, (int, float)) and not isinstance(v, bool) for v in a)

    level_scalars = None
    if _numbers(seg_args[-1]):
        level_scalars = [float(v) for v in seg_args[-1]]
        seg_args = (*seg_args[:-1], 0.0)
    lists = [a for a in seg_args if isinstance(a, (list, tuple))]
    if not lists:
        raise TypeError("ek_thermo: a batched suite needs at least one list of CUDA tensors")
    n_seg = len(lists[0])
    if any(len(a) != n_seg for a in lists) or (level_scalars is not None and len(level_scalars) != n_seg):
        raise ValueError("ek_thermo: the input lists of a batched suite must have one length")
    res = [dict() for _ in range(n_seg)]
    if n_seg == 0:
        return res
    for a in lists:
        for t in a:
            if not isinstance(t, torch.Tensor):
                raise TypeError("ek_thermo: batched suite arguments are lists of torch CUDA tensors or Python numbers")
    dev = _check_device([t for a in lists for t in a])  # every field a CUDA tensor on one device: no CPU path
    first = lists[0][0]
    dtype, shape = first.dtype, first.shape
    if dtype not in _SUFFIX:
        raise TypeError("ek_thermo: batched suites take float64 or float32 tensors")
    keep = []
    ptr_arrays = []
    scalars = (c_double * 3)(0.0, 0.0, 0.0)
    for k, a in enumerate(seg_args):
        if isinstance(a, (list, tuple)):
            for t in a:
                if t.dtype != dtype or t.shape != shape or not t.is_contiguous():
                    raise ValueError("ek_thermo: the fields of a batched suite must share dtype, device and shape and be contiguous")
            ptr_arrays.append((c_void_p * n_seg)(*[t.data_ptr() for t in a]))
        elif isinstance(a, (int, float)) and not isinstance(a, bool):
            scalars[k] = float(a)
            ptr_arrays.append(None)
        else:
            raise TypeError("ek_thermo: batched suite arguments are lists of CUDA tensors or Python numbers")
    out_tab = (c_void_p * N_SUITE_SLOTS)()
    mask = 0
    for name, k in zip(out_names, slots):
        col = []
        for j in range(n_seg):
            t = outs[j].get(name) if outs is not None else None
            if t is not None:
                if t.dtype != dtype or t.shape != shape or not t.is_contiguous() or t.device != dev:
                    raise ValueError(f"ek_thermo: preallocated output {name!r} of field {j} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {dev}")
            else:
                t = torch.empty(shape, dtype=dtype, device=dev)
            res[j][name] = t
            col.append(t.data_ptr())
        arr = (c_void_p * n_seg)(*col)
        keep.append(arr)
        out_tab[k] = ctypes.cast(arr, c_void_p)
        mask |= 1 << k
    n = first.numel()
    if n > 0:
        lv = (c_double * n_seg)(*level_scalars) if level_scalars is not None else None
        _call(symbol, dtype, dev, [n_seg, *ptr_arrays, scalars, lv, out_tab, mask, ept_method, n])
    del keep
    return res


def shard_range(n: int, world: int, rank: int, align: int = 1):
    b, e = c_int64(0), c_int64(0)
    _check(_lib.ek_thermo_shard_range(n, world, rank, align, ctypes.byref(b), ctypes.byref(e)))
    return int(b.value), int(e.value)


def host_pipeline(symbol: str, dtype, workspace: torch.Tensor, n_slots: int, *c_args):
    """Run host-array pipeline entry point `symbol` (ek_thermo_host_suite*): `c_args` up to the workspace, which the pipeline
    splits into `n_slots` stream slots."""
    fn = getattr(_lib, f"ek_thermo_{symbol}_{_SUFFIX[dtype]}")
    with torch.cuda.device(workspace.device):
        torch.cuda.current_stream().synchronize()  # the pipeline runs on its own streams: nothing may be pending on the workspace
        _check(fn(*c_args, workspace.data_ptr(), workspace.numel() * workspace.element_size(), n_slots))
