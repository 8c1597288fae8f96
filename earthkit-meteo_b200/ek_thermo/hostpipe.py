"""Host-buffer front end: the fused suite over numpy / host arrays, streamed through the GPU.

This is the "reference-facing" call measured as ``e2e`` by bench.py: inputs and outputs live in HOST
memory; the C library overlaps H2D copies, the suite kernel and D2H copies of successive chunks on
several streams (ek_thermo_host_suite_*).  All arithmetic still happens on the GPU.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _backend as _b
from .fused import COLUMN_OUTPUTS, DEFAULT_TQP, DEFAULT_TTDP, SUITE_TQP_OUTPUTS, SUITE_TTDP_OUTPUTS

_TORCH = {np.dtype("float64"): torch.float64, np.dtype("float32"): torch.float32}


def pinned_empty(n, dtype=np.float64):
    """A page-locked host array (numpy view of a pinned torch tensor), for full-speed PCIe copies."""
    t = torch.empty(int(n), dtype=_TORCH[np.dtype(dtype)], pin_memory=True)
    return t.numpy()


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_host_to_device(device="cuda:0"):
    """Restrict the calling process to the CPUs next to `device` (its PCIe root's NUMA node).

    Page-locked buffers allocated afterwards land in that node's memory (Linux allocates on the node of the
    allocating thread), so H2D / D2H copies do not cross the socket interconnect.  Matters when one process per GPU
    streams host fields through several GPUs of a multi-socket box at once.  Returns the CPU set it bound to, or
    None when the topology cannot be read (no sysfs entry, no overlap with the allowed CPUs) -- never raises.
    """
    import os

    try:
        pr = torch.cuda.get_device_properties(torch.device(device))
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/local_cpulist") as f:
            local = _parse_cpulist(f.read())
        allowed = os.sched_getaffinity(0)
        cpus = local & allowed
        if not cpus or cpus == allowed:
            return sorted(cpus) or None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except (OSError, AttributeError, ValueError, RuntimeError, AssertionError):
        return None


_EPT = {"ifs": 0, "bolton35": 1, "bolton39": 2}


class HostSuite:
    """Reusable pipeline: owns the device workspace (allocated once through torch) and the stream slots."""

    def __init__(self, device="cuda:0", workspace_bytes=1 << 30, n_slots=3):
        self.device = torch.device(device)
        self.n_slots = int(n_slots)
        self.workspace = torch.empty(int(workspace_bytes), dtype=torch.uint8, device=self.device)

    @staticmethod
    def _outputs(table, outputs, out, shape, dt):
        n = int(np.prod(shape))
        ptrs = [0] * _b.N_SUITE_SLOTS
        mask = 0
        res = {}
        for name in outputs:
            k = table[name]
            o = out[name] if out is not None and name in out else np.empty(shape, dtype=dt)
            if o.dtype != dt or o.size != n or not o.flags.c_contiguous:
                raise ValueError(f"host suite: output {name!r} must be a contiguous {dt} array of {n} elements")
            res[name] = o
            ptrs[k] = o.ctypes.data
            mask |= 1 << k
        return res, ptrs, mask

    def _run(self, kind, table, a, b, c, outputs, out, ept_method):
        arrs = [np.ascontiguousarray(x) for x in (a, b, c)]
        dt = arrs[0].dtype
        if dt not in _TORCH or any(x.dtype != dt or x.shape != arrs[0].shape for x in arrs):
            raise TypeError("host suite: the three inputs must be float64 or float32 numpy arrays of one shape")
        res, ptrs, mask = self._outputs(table, outputs, out, arrs[0].shape, dt)
        _b.host_suite(kind, _TORCH[dt], [x.ctypes.data for x in arrs], ptrs, mask, _EPT[ept_method], arrs[0].size, self.workspace, self.n_slots)
        return res

    def suite_tqp(self, t, q, p, outputs=DEFAULT_TQP, out=None, ept_method="ifs"):
        return self._run(0, SUITE_TQP_OUTPUTS, t, q, p, tuple(outputs), out, ept_method)

    def suite_ttdp(self, t, td, p, outputs=DEFAULT_TTDP, out=None, ept_method="ifs"):
        return self._run(1, SUITE_TTDP_OUTPUTS, t, td, p, tuple(outputs), out, ept_method)

    def suite_tq_hybrid(self, t, q, sp, A, B, outputs=DEFAULT_TQP, out=None, ept_method="ifs", zs=None, alpha_top="ifs", h_type="geometric",
                        h_reference="ground"):
        """``fused.suite_tq_hybrid`` for host arrays: t, q ``[nlev, npl]``, sp ``[npl]``, A / B ``nlev + 1`` half-level values.
        The pressure field crosses PCIe in neither direction (sp travels instead: 16 + 8/nlev bytes per point in).  The column
        outputs ``"thickness"``, ``"z"`` and ``"height"`` with ``zs`` (a ``[npl]`` array or a Python number), ``alpha_top``,
        ``h_type`` and ``h_reference`` as there; they come from the same kernel pass over each chunk."""
        from .vertical import _height_mode, _top_is_toa

        outputs = tuple(outputs)
        cols = tuple(o for o in outputs if o in COLUMN_OUTPUTS)
        suite = tuple(o for o in outputs if o not in COLUMN_OUTPUTS)
        if alpha_top not in ("ifs", "arpege"):
            raise ValueError(f"Unknown method '{alpha_top}' for pressure calculation. Use 'ifs' or 'arpege'.")
        hmode = _height_mode(h_type, h_reference)
        t, q, sp = (np.ascontiguousarray(x) for x in (t, q, sp))
        dt = t.dtype
        if dt not in _TORCH or q.dtype != dt or sp.dtype != dt or t.ndim != 2 or q.shape != t.shape or sp.shape != t.shape[1:]:
            raise TypeError("host suite: t, q must be [nlev, npl] and sp [npl] float64 or float32 numpy arrays of one dtype")
        nlev, npl = t.shape
        a = np.ascontiguousarray(np.asarray(A, dtype=dt))
        b = np.ascontiguousarray(np.asarray(B, dtype=dt))
        if a.shape != (nlev + 1,) or b.shape != (nlev + 1,):
            raise ValueError(f"host suite: A and B need nlev + 1 = {nlev + 1} half-level values")
        res, ptrs, mask = self._outputs(SUITE_TQP_OUTPUTS, suite, out, t.shape, dt)
        if not cols:
            _b.host_suite_tq_hybrid(_TORCH[dt], t.ctypes.data, q.ctypes.data, sp.ctypes.data, a.ctypes.data, b.ctypes.data, nlev, npl, ptrs, mask,
                                    _EPT[ept_method], self.workspace, self.n_slots)
            return res
        modes = {"thickness": 0, "z": 1, "height": hmode}
        zs_ptr = None
        if any(modes[c] not in (0, 3) for c in cols):
            if zs is None:
                raise ValueError("host suite: 'z' and every 'height' except geopotential height above ground need the surface geopotential zs")
            zs = np.full(sp.shape, zs, dtype=dt) if isinstance(zs, (int, float)) and not isinstance(zs, bool) else np.ascontiguousarray(zs)
            if zs.dtype != dt or zs.shape != sp.shape:
                raise TypeError(f"host suite: zs must be a {dt} array of shape {sp.shape} or a Python number")
            zs_ptr = zs.ctypes.data
        col_res, _, _ = self._outputs({c: 0 for c in cols}, cols, out, t.shape, dt)
        res.update(col_res)
        res = {name: res[name] for name in outputs}
        _b.host_suite_tq_hybrid_geo(_TORCH[dt], t.ctypes.data, q.ctypes.data, sp.ctypes.data, zs_ptr, a.ctypes.data, b.ctypes.data, nlev, npl, ptrs,
                                    mask, _EPT[ept_method], _top_is_toa(a, b, 0, sp, None, None), math.log(2.0) if alpha_top == "ifs" else 1.0,
                                    [res[c].ctypes.data if c in res else None for c in COLUMN_OUTPUTS], hmode, self.workspace, self.n_slots)
        return res
