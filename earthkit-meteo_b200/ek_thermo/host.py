"""``ek_thermo.host`` -- the same functions for HOST arrays: numpy in, numpy out, computed on the GPU.

The reference's callers hold numpy arrays (``earthkit.meteo.thermo.array`` is array-namespace code, and
``xr.apply_ufunc(potential_temperature, t, p)`` hands it the numpy data of xarray objects, reference
tests/vertical/test_xr_theta.py:34).  This module is the data-format adapter on that side of the path
(SURVEY.md 8(f)-4): ``host.thermo.<fn>`` and ``host.wind.<fn>`` take what the reference takes -- numpy arrays, nested
lists, numpy / Python scalars, with numpy broadcasting and dtype promotion -- stream the arrays through the device
in chunks on two CUDA streams (H2D copy, the one kernel of ``ek_thermo.thermo.<fn>``, D2H copy), and return numpy
arrays of the broadcast shape.  Options (``method=``, ``phase=``, ``eps=`` ...) and error behaviour are those of the
device functions, i.e. of the reference.

There is no CPU arithmetic here: without a CUDA device every call raises ``RuntimeError``.  Arrays of 4 Mi elements
or more go through page-locked staging buffers that worker threads fill and drain (a pageable ``cudaMemcpy`` is limited
to 7-8 GB/s by the driver's single staging buffer); page-locked inputs (``hostpipe.pinned_empty``) are copied directly.
Measured on one B200: 1.0-1.15 Gpt/s for pageable float64 arrays (0.22-0.30 without the staging threads), against
0.010 Gpt/s for the reference on one core.  For the fused suites on whole fields use ``hostpipe.HostSuite`` (one C
call, three streams, no Python per chunk).
"""
from __future__ import annotations

import functools
import math
import threading

import numpy as np
import torch

from . import fused as _fused
from . import thermo as _thermo
from . import wind as _wind
from ._backend import _TORCH

__all__ = ["thermo", "wind", "fused", "set_chunk_elements", "set_pinned_results", "release_staging"]

_CHUNK = 1 << 25  # elements per array per chunk (256 MB of float64): bounds device memory, amortises launch latency


def set_chunk_elements(n):
    """Elements per array and chunk of the host pipeline (default 2**25).  Returns the previous value."""
    global _CHUNK
    old = _CHUNK
    if int(n) < 1:
        raise ValueError("set_chunk_elements: n must be >= 1")
    _CHUNK = int(n)
    return old


def _is_arraylike(v):
    if isinstance(v, (list, tuple)):  # nested numbers are arrays; ("theta", "rh") is an option
        return not (len(v) > 0 and isinstance(v[0], str))
    return isinstance(v, (np.ndarray, np.generic))


def _run(fn, args, kwargs, device):
    if not torch.cuda.is_available():
        raise RuntimeError("ek_thermo.host: no CUDA device. The arithmetic runs on the GPU only; there is no CPU fallback "
                           "(use earthkit.meteo for CPU arrays).")
    args = list(args)
    kwargs = {k: (v.item() if isinstance(v, np.generic) else v) for k, v in kwargs.items()}  # numpy scalars as options
    slots = [("a", i) for i, v in enumerate(args) if _is_arraylike(v)] + [("k", k) for k, v in kwargs.items() if _is_arraylike(v)]
    if not slots:  # all Python numbers: the reference returns a numpy scalar
        for i, v in enumerate(args):
            if isinstance(v, (int, float)) and not isinstance(v, bool):
                args[i] = np.asarray(float(v))
                slots = [("a", i)]
                break
        if not slots:
            raise TypeError("ek_thermo.host: expected at least one array or number argument")

    def get(slot):
        return args[slot[1]] if slot[0] == "a" else kwargs[slot[1]]

    def put(slot, v):
        if slot[0] == "a":
            args[slot[1]] = v
        else:
            kwargs[slot[1]] = v

    arrs = [np.asarray(get(s)) for s in slots]
    dt = np.result_type(*arrs)  # Python scalars among the arguments do not up-cast float32 arrays (numpy semantics)
    if dt not in _TORCH:
        dt = np.dtype("float64")  # integer / bool / float16 input: computed in float64, as numpy would promote
    shape = np.broadcast_shapes(*[a.shape for a in arrs])
    n = int(math.prod(shape))
    flat = []
    for s, a in zip(slots, arrs):
        a = a.astype(dt, copy=False)
        if a.size == 1 and n != 1:
            put(s, float(a.reshape(-1)[0]))  # broadcast by value inside the kernel, never materialised
            continue
        if a.shape != shape:
            a = np.broadcast_to(a, shape)
        a = np.ascontiguousarray(a)
        if not a.flags.writeable:  # torch.from_numpy wants a writable buffer (it is only read here)
            a = a.copy()
        flat.append((s, a.reshape(-1)))
    if n == 0:
        probe = fn(*[torch.empty(0, dtype=_TORCH[dt], device=device) if ("a", i) in slots else v for i, v in enumerate(args)],
                   **{k: (torch.empty(0, dtype=_TORCH[dt], device=device) if ("k", k) in slots else v) for k, v in kwargs.items()})
        many = isinstance(probe, tuple)
        outs = [np.empty(shape, dt) for _ in (probe if many else (probe,))]
        return tuple(outs) if many else outs[0]

    if n >= _STAGE_MIN:
        outs, many = _pipeline_staged(fn, args, kwargs, put, flat, dt, n, device)
    else:
        outs, many = _pipeline_direct(fn, args, kwargs, put, flat, dt, n, device)
    outs = [o.reshape(shape)[()] if shape == () else o.reshape(shape) for o in outs]
    return tuple(outs) if many else outs[0]


def _pipeline_direct(fn, args, kwargs, put, flat, dt, n, device):
    """Chunks copied straight from / to the caller's arrays on two streams (asynchronous when they are page-locked)."""
    streams = [torch.cuda.Stream(device=device) for _ in range(2)]
    outs = None
    many = False
    chunk = max(1, _CHUNK)
    for ci, b in enumerate(range(0, n, chunk)):
        e = min(n, b + chunk)
        st = streams[ci % 2]
        with torch.cuda.stream(st):
            for s, a in flat:
                put(s, torch.from_numpy(a[b:e]).to(device, non_blocking=True))
            res = fn(*args, **kwargs)
            many = isinstance(res, tuple)
            res = res if many else (res,)
            if outs is None:
                outs = [np.empty(n, dt) for _ in res]
            for o, r in zip(outs, res):
                torch.from_numpy(o[b:e]).copy_(r.reshape(-1), non_blocking=True)
    for st in streams:
        st.synchronize()
    return outs, many


# ---- staged pipeline for large pageable arrays ---------------------------------------------------------------------
# A pageable cudaMemcpy goes through the driver's single staging buffer at 7-8 GB/s.  Here worker threads copy each
# input chunk into page-locked staging buffers (numpy releases the GIL for the copy) while the copies to and from the
# device run asynchronously on the slot's stream.  The RESULT arrays are page-locked themselves (numpy views of pinned
# torch tensors from torch's caching host allocator: the first call pays cudaHostAlloc, later calls reuse the blocks of
# results the caller has dropped), so the D2H copy lands in the array that is returned -- no second copy of the outputs.
# `set_pinned_results(False)` returns ordinary pageable numpy arrays instead (outputs then pass through staging too).
#
# Re-entrancy: every running call checks a private _StagingSet out of a free list under a lock (dask's threaded
# scheduler and xr.apply_ufunc call these functions from several threads at once); the worker pool is shared.
_STAGE_MIN = 1 << 22    # elements: below this the direct path is used
_STAGE_CHUNK = 1 << 22  # elements per array and staged chunk (32 MB of float64)
_STAGE_SLOTS = 5        # chunks in flight (measured on a 16-vCPU host, theta: 3 slots 0.83, 4 slots 0.97-1.09, 5 slots 1.15 Gpt/s)
_STAGE_LAG = 1          # (pageable results) a chunk is copied out of staging this many chunks after it was issued
_STAGE_WORKERS = 12     # upper bound; never more than the CPUs this process may run on
_PINNED_RESULTS = True
_pool = None
_pool_size = 0
_lock = threading.Lock()
_free_sets = []   # _StagingSet objects no call is using
_generation = 0   # bumped by release_staging(): sets of an older generation are dropped when their call returns


class _StagingSet:
    """The page-locked staging buffers of ONE running call: (dtype, slot, role, k) -> pinned tensor of _STAGE_CHUNK elements."""

    def __init__(self, generation):
        self.generation = generation
        self.bufs = {}

    def buf(self, dt, slot, role, k):
        key = (dt, slot, role, k)
        t = self.bufs.get(key)
        if t is None or t.numel() < _STAGE_CHUNK:
            t = self.bufs[key] = torch.empty(_STAGE_CHUNK, dtype=_TORCH[dt], pin_memory=True)
        return t


def _checkout():
    with _lock:
        while _free_sets:
            s = _free_sets.pop()
            if s.generation == _generation:
                return s
        return _StagingSet(_generation)


def _checkin(s):
    with _lock:
        if s.generation == _generation:
            _free_sets.append(s)


def _workers():
    global _pool, _pool_size
    with _lock:
        if _pool is None:
            import os
            from concurrent.futures import ThreadPoolExecutor

            _pool_size = max(2, min(_STAGE_WORKERS, len(os.sched_getaffinity(0))))
            _pool = ThreadPoolExecutor(max_workers=_pool_size, thread_name_prefix="ek_host")
        return _pool


def set_pinned_results(flag):
    """Large results as page-locked numpy arrays (default) or ordinary pageable ones.  Returns the previous setting."""
    global _PINNED_RESULTS
    old = _PINNED_RESULTS
    _PINNED_RESULTS = bool(flag)
    return old


def release_staging():
    """Free the page-locked staging buffers of the host pipeline (they are kept between calls).  Safe while other threads
    are inside a call: their sets are private and are dropped, not reused, when those calls return."""
    global _generation
    with _lock:
        _generation += 1
        _free_sets.clear()
    empty = getattr(torch._C, "_host_emptyCache", None)  # hand cached page-locked blocks back to the OS where torch can
    if empty is not None:
        empty()


def _result_array(n, dt):
    if _PINNED_RESULTS:
        return torch.empty(n, dtype=_TORCH[dt], pin_memory=True).numpy()  # the numpy view keeps the pinned tensor alive
    return np.empty(n, dt)


def _pipeline_staged(fn, args, kwargs, put, flat, dt, n, device):
    st_set = _checkout()
    try:
        return _pipeline_staged_run(st_set, fn, args, kwargs, put, flat, dt, n, device)
    finally:
        torch.cuda.synchronize(device)  # nothing of this call may still read or write the set's buffers (error paths too)
        _checkin(st_set)


def _pipeline_staged_run(st_set, fn, args, kwargs, put, flat, dt, n, device):
    pool = _workers()
    S = _STAGE_SLOTS
    pinned = [torch.from_numpy(a[:1]).is_pinned() for _, a in flat]  # the caller's own page-locked arrays skip staging
    streams = [torch.cuda.Stream(device=device) for _ in range(S)]
    h2d_done = [None] * S  # event: the slot's input staging buffers have been read by the device
    events = [torch.cuda.Event() for _ in range(S)]
    pending = [[] for _ in range(S)]  # (pageable results) copy-out futures of the chunk that used the slot last
    ranges = [None] * S
    outs = None
    out_pinned = False
    many = False
    nres = 0
    nchunks = -(-n // _STAGE_CHUNK)

    n_pageable = sum(1 for x in pinned if not x)
    # every array's chunk is copied in pieces by several workers at once: one memcpy stream per array (3 for a suite) leaves
    # most of the host's memory bandwidth unused and makes the staging step the bottleneck of the whole pipeline
    parts = max(1, min(4, _pool_size // max(1, n_pageable)))

    def fill(ci):
        """Worker threads copy chunk ci of every pageable input into the slot's staging buffers."""
        slot = ci % S
        b = ci * _STAGE_CHUNK
        e = min(n, b + _STAGE_CHUNK)
        if h2d_done[slot] is not None:
            h2d_done[slot].synchronize()
        futs = []
        step = -(-(e - b) // parts)
        for k, (_, a) in enumerate(flat):
            if pinned[k]:
                continue
            dst = st_set.buf(dt, slot, "in", k).numpy()
            for o in range(0, e - b, step):
                m = min(step, e - b - o)
                futs.append(pool.submit(np.copyto, dst[o:o + m], a[b + o:b + o + m]))
        return futs

    def copy_out(slot):
        b, e = ranges[slot]
        events[slot].synchronize()
        step = -(-(e - b) // max(1, min(4, _pool_size // max(1, nres))))
        pending[slot] = [pool.submit(np.copyto, outs[j][b + o:min(e, b + o + step)], st_set.buf(dt, slot, "out", j).numpy()[o:min(e - b, o + step)])
                         for j in range(nres) for o in range(0, e - b, step)]

    futs = fill(0)
    for ci in range(nchunks):
        b = ci * _STAGE_CHUNK
        e = min(n, b + _STAGE_CHUNK)
        m = e - b
        slot = ci % S
        nxt = fill(ci + 1) if ci + 1 < nchunks else []  # the next chunk is staged while this one is issued
        for f in futs:
            f.result()
        for f in pending[slot]:
            f.result()  # (pageable results) the slot's output staging buffers are free again
        pending[slot] = []
        with torch.cuda.stream(streams[slot]):
            for k, (s, a) in enumerate(flat):
                src = torch.from_numpy(a[b:e]) if pinned[k] else st_set.buf(dt, slot, "in", k)[:m]
                put(s, src.to(device, non_blocking=True))
            h2d_done[slot] = torch.cuda.Event()
            h2d_done[slot].record()
            res = fn(*args, **kwargs)
            many = isinstance(res, tuple)
            res = res if many else (res,)
            if outs is None:
                nres = len(res)
                out_pinned = _PINNED_RESULTS
                outs = [_result_array(n, dt) for _ in res]
            for j, r in enumerate(res):
                dst = torch.from_numpy(outs[j][b:e]) if out_pinned else st_set.buf(dt, slot, "out", j)[:m]
                dst.copy_(r.reshape(-1), non_blocking=True)
            events[slot].record()
        ranges[slot] = (b, e)
        futs = nxt
        if not out_pinned and ci >= _STAGE_LAG:  # an earlier chunk has had the staging time of the chunks after it to finish
            copy_out((ci - _STAGE_LAG) % S)
    if not out_pinned:
        for k in range(max(0, nchunks - _STAGE_LAG), nchunks):
            copy_out(k % S)
        for p in pending:
            for f in p:
                f.result()
    for st in streams:
        st.synchronize()
    return outs, many


class _HostNamespace:
    """Attribute access returns the host-array version of the device function of the same name."""

    def __init__(self, module, names, what):
        self._module = module
        self.__all__ = list(names)
        self.__doc__ = f"Host-array (numpy) front end of ``ek_thermo.{what}``: same names, signatures and options."
        self.device = None  # None: the current CUDA device at call time
        for name in names:
            setattr(self, name, self._wrap(getattr(module, name)))

    def _wrap(self, fn):
        @functools.wraps(fn)
        def host_fn(*args, **kwargs):
            dev = torch.device("cuda", torch.cuda.current_device()) if self.device is None and torch.cuda.is_available() else self.device
            return _run(fn, args, kwargs, dev)

        host_fn.__doc__ = (fn.__doc__ or "") + "\n\nHost-array version: numpy arrays / scalars in, numpy out; computed on the GPU in chunks."
        return host_fn


class _HostFused:
    """Host-array versions of the fused kernels: one pass over PCIe for all requested fields."""

    device = None

    def _dev(self):
        return torch.device("cuda", torch.cuda.current_device()) if self.device is None and torch.cuda.is_available() else self.device

    def _suite(self, fn, a, b, c, outputs, ept_method):
        outputs = tuple(outputs)
        res = _run(lambda x, y, z: tuple(fn(x, y, z, outputs=outputs, ept_method=ept_method).values()), (a, b, c), {}, self._dev())
        return dict(zip(outputs, res if isinstance(res, tuple) else (res,)))

    def suite_tqp(self, t, q, p, outputs=_fused.DEFAULT_TQP, ept_method="ifs"):
        """``fused.suite_tqp`` for numpy arrays: returns ``{name: numpy array}``."""
        return self._suite(_fused.suite_tqp, t, q, p, outputs, ept_method)

    def suite_ttdp(self, t, td, p, outputs=_fused.DEFAULT_TTDP, ept_method="ifs"):
        """``fused.suite_ttdp`` for numpy arrays: returns ``{name: numpy array}``."""
        return self._suite(_fused.suite_ttdp, t, td, p, outputs, ept_method)

    def suite_trp(self, t, r, p, outputs=_fused.DEFAULT_TRP, ept_method="ifs"):
        """``fused.suite_trp`` for numpy arrays: returns ``{name: numpy array}``."""
        return self._suite(_fused.suite_trp, t, r, p, outputs, ept_method)

    def ept_wet_bulb(self, t, h, p, humidity="q", ept_method="ifs", t_method="direct", potential=True):
        """``fused.ept_wet_bulb`` for numpy arrays: returns ``(ept, wet_bulb)`` as numpy arrays."""
        return _run(lambda x, y, z: _fused.ept_wet_bulb(x, y, z, humidity=humidity, ept_method=ept_method, t_method=t_method, potential=potential),
                    (t, h, p), {}, self._dev())


fused = _HostFused()
thermo = _HostNamespace(_thermo, _thermo.__all__, "thermo")
thermo.array = thermo  # the reference exposes the functions under ``thermo`` and ``thermo.array``
wind = _HostNamespace(_wind, _wind.__all__, "wind")
wind.array = wind
