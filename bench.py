#!/usr/bin/env python
"""bench.py -- thermo grid-points/s and achieved HBM GB/s vs roofline (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input.  Default workload (N=1) is
BASELINE.json configs[1]: the fused thermo suite (t,q,p -> theta, es, rh, td, Tv) on IFS O1280
(6 599 680 points) x 137 model levels, float64 = 904 156 160 points, 64 algorithmic bytes per point.
Inputs are generated ON DEVICE before the timed region (58 GB resident, far larger than the 126 MB L2,
so every step streams from HBM).  For N>1 (torchrun, one process per GPU) the default workloads run the same
per-GPU field on every rank (weak scaling); `conv_ens_o640_f64` (BASELINE.json configs[3]) is PARTITIONED: the
51 x 137 slabs of the ensemble are sharded over the ranks by ek_thermo.partition, results stay resident, and a
cross-shard check recomputes probe slabs of every shard on rank 0.  There is no data-path collective -- NCCL is
only used for the barrier and the max-over-ranks of the device time (a gloo group carries the shard check).

Printed JSON line: see the keys below; `roofline`, `cpu_baseline`, `e2e`, `parity`, `clocks`, `gpu_launches` are
described in DESIGN.md section 6.  `--impl reference` times the UNMODIFIED reference (installed in oracle/_ref by
oracle/build_ref.py; the numpy oracle port if that install is absent) on all host cores, on level slabs of the
same synthetic field (same generator, same seed), after running the reference's own thermo tests against it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, "earthkit-meteo_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

from synthetic import N_LEVELS, O640_POINTS, O1280_POINTS, IfsField, sample_levels  # noqa: E402

METRIC = "thermo grid-points/s"  # BASELINE.json metric; the achieved HBM GB/s vs roofline half of it is the `roofline` object

SUITE5_Q = ("theta", "es", "rh", "td", "tv")
SUITE5_TD = ("theta", "es", "rh", "q", "tv")


def _w(kind, outputs, levels, npl, dtype, members=1, sharded=False, slabs=None):
    return dict(kind=kind, outputs=tuple(outputs), levels=levels, npl=npl, dtype=dtype, members=members, sharded=sharded,
                slabs=slabs or members * levels)


WORKLOADS = {
    # BASELINE.json configs[1] (the configuration the metric is quoted on) and its float32 / dewpoint twins
    "suite_tqp_o1280x137_f64": _w("tqp", SUITE5_Q, N_LEVELS, O1280_POINTS, "f64"),
    "suite_tqp_o1280x137_f32": _w("tqp", SUITE5_Q, N_LEVELS, O1280_POINTS, "f32"),
    "suite_ttdp_o1280x137_f64": _w("ttdp", SUITE5_TD, N_LEVELS, O1280_POINTS, "f64"),
    # the single pass of north_star item 3: one read of (t, q, p) -> theta, rh, td, theta_e, theta_w (64 B/pt) and the
    # same with es and Tv as well (80 B/pt): configs[1] + configs[2] in one launch
    "single_pass_tqp_o1280x137_f64": _w("tqp", ("theta", "rh", "td", "ept", "wbpt"), N_LEVELS, O1280_POINTS, "f64"),
    "suite7_tqp_o1280x137_f64": _w("tqp", SUITE5_Q + ("ept", "wbpt"), N_LEVELS, O1280_POINTS, "f64"),
    "suite7_tqp_o1280x137_f32": _w("tqp", SUITE5_Q + ("ept", "wbpt"), N_LEVELS, O1280_POINTS, "f32"),
    "suite7_ttdp_o1280x137_f64": _w("ttdp", SUITE5_TD + ("ept", "wbpt"), N_LEVELS, O1280_POINTS, "f64"),
    # BASELINE.json configs[0]: theta + rh on one ERA5 0.25 degree level
    "theta_rh_era5_f64": _w("tqp", ("theta", "rh"), 1, 721 * 1440, "f64"),
    # BASELINE.json configs[2]: ept + wet-bulb potential temperature ("direct"), the two-output kernel
    "ept_wbpt_o1280x137_f64": _w("ept", ("ept", "wbpt"), N_LEVELS, O1280_POINTS, "f64"),
    "ept_wbpt_o1280x137_f32": _w("ept", ("ept", "wbpt"), N_LEVELS, O1280_POINTS, "f32"),
    # SURVEY.md 8(f)-1: the same suite with the pressure computed in-kernel from sp and the L137 A/B (56 B/pt)
    "suite_tq_hybrid_o1280x137_f64": _w("hybrid", SUITE5_Q, N_LEVELS, O1280_POINTS, "f64"),
    # BASELINE.json configs[3]: ENS 51 members x O640 x 137 levels, humidity / dewpoint conversions.  `_shard_` = one
    # GPU's eighth of it on every rank (weak); without: the whole ensemble partitioned over the ranks (see module docstring)
    "conv_ens_o640_shard_f64": _w("tqp", ("rh", "td", "w"), N_LEVELS, O640_POINTS, "f64", members=7, slabs=874),
    "conv_ens_o640_f64": _w("tqp", ("rh", "td", "w"), N_LEVELS, O640_POINTS, "f64", members=51, sharded=True),
}
DEFAULT_WORKLOAD = "suite_tqp_o1280x137_f64"

L2_FLUSH_BYTES = 384 << 20  # rotate small workloads over at least this many bytes (3 x the 126 MB L2)
HBM_BUDGET_BYTES = 150e9    # resident arrays per GPU (of 180 GB): a shard larger than this is capped and reported so
DUMP_BYTES = 64 << 20       # --dump-outputs writes at most this much in all

# output name -> the public reference function it equals, on module m (the reference's earthkit.meteo.thermo or the
# oracle, which mirrors its names): this is how a user of the reference computes the same fields
OUT_FNS = {
    "tqp": {
        "theta": lambda m, t, q, p: m.potential_temperature(t, p),
        "es": lambda m, t, q, p: m.saturation_vapour_pressure(t),
        "rh": lambda m, t, q, p: m.relative_humidity_from_specific_humidity(t, q, p),
        "td": lambda m, t, q, p: m.dewpoint_from_specific_humidity(q, p),
        "tv": lambda m, t, q, p: m.virtual_temperature(t, q),
        "w": lambda m, t, q, p: m.mixing_ratio_from_specific_humidity(q),
        "e": lambda m, t, q, p: m.vapour_pressure_from_specific_humidity(q, p),
        "thetav": lambda m, t, q, p: m.virtual_potential_temperature(t, q, p),
        "ept": lambda m, t, q, p: m.ept_from_specific_humidity(t, q, p),
        "wbpt": lambda m, t, q, p: m.wet_bulb_potential_temperature_from_specific_humidity(t, q, p),
    },
    "ttdp": {
        "theta": lambda m, t, td, p: m.potential_temperature(t, p),
        "es": lambda m, t, td, p: m.saturation_vapour_pressure(t),
        "rh": lambda m, t, td, p: m.relative_humidity_from_dewpoint(t, td),
        "q": lambda m, t, td, p: m.specific_humidity_from_dewpoint(td, p),
        "tv": lambda m, t, td, p: m.virtual_temperature(t, m.specific_humidity_from_dewpoint(td, p)),
        "w": lambda m, t, td, p: m.mixing_ratio_from_dewpoint(td, p),
        "ept": lambda m, t, td, p: m.ept_from_dewpoint(t, td, p),
        "wbpt": lambda m, t, td, p: m.wet_bulb_potential_temperature_from_dewpoint(t, td, p),
    },
}
OUT_FNS["hybrid"] = OUT_FNS["ept"] = OUT_FNS["tqp"]


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(workload):
    """DRAM bytes per launch of the workload's kernel, from the committed `ncu --set full` capture of this round (if any)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(workload)
    return None


def cpu_module():
    """(module, kind): the unmodified reference from oracle/_ref when it is installed, else the numpy oracle port."""
    import build_ref

    if build_ref.installed():
        for p in reversed(build_ref.sys_path_entries()):
            if p not in sys.path:
                sys.path.insert(0, p)
        from earthkit.meteo import thermo as ref_thermo

        assert os.path.realpath(ref_thermo.__file__).startswith(os.path.realpath(build_ref.DEST)), ref_thermo.__file__
        return ref_thermo, "reference"
    import thermo_oracle

    return thermo_oracle, "port"


def cpu_step(kind, outputs, module):
    fns = OUT_FNS[kind]

    def step(a, b, c):
        return [fns[o](module, a, b, c) for o in outputs]

    return step


# --------------------------------------------------------------------------------------------------
# the hot-path step on the device
# --------------------------------------------------------------------------------------------------
def build_step(kind, outputs, arrays, hyb=None):
    """Returns (step callable, bytes per point, output tensors).  Output buffers are allocated once and reused."""
    import torch

    from ek_thermo import _backend, fused

    t, h, p = arrays
    esz = t.element_size()
    if kind == "hybrid":
        sp, a, b = hyb
        nlev = a.numel() - 1
        t2, h2 = t.reshape(nlev, -1), h.reshape(nlev, -1)
        out = {name: torch.empty_like(t2) for name in outputs}

        def step():
            fused.suite_tq_hybrid(t2, h2, sp, a, b, outputs=outputs, out=out)

        # per point: t, q read, outputs written; sp is read once per point COLUMN (8/nlev B per point)
        return step, esz * (2 + len(outputs)) + esz / nlev, {k: v.reshape(-1) for k, v in out.items()}
    if kind in ("tqp", "ttdp"):
        out = {name: torch.empty_like(t) for name in outputs}
        fn = fused.suite_tqp if kind == "tqp" else fused.suite_ttdp
        bpp = esz * (3 + len(outputs))
        # a field that fits the 126 MB L2 (one ERA5 level: 41.5 MB) is rotated over enough copies that no launch finds
        # its inputs in L2 (SURVEY 8(d): "rotating buffers > 126 MB")
        n_sets = 1 if bpp * t.numel() >= L2_FLUSH_BYTES else -(-L2_FLUSH_BYTES // (bpp * t.numel()))
        sets = [(t, h, p, out)] + [(t.clone(), h.clone(), p.clone(), {k: torch.empty_like(t) for k in outputs}) for _ in range(n_sets - 1)]
        state = {"i": 0}

        def step():
            a, b, c, o = sets[state["i"] % n_sets]
            state["i"] += 1
            fn(a, b, c, outputs=outputs, out=o)

        step.n_sets = n_sets
        step.last_out = lambda: sets[(state["i"] - 1) % n_sets][3]
        return step, bpp, out
    # ept + wet-bulb potential temperature ("direct"), BASELINE.json configs[2]: the two-output kernel
    from ctypes import c_int, c_int64, c_void_p

    ept, wb = torch.empty_like(t), torch.empty_like(t)
    ops = [_backend.ek_operand(x.data_ptr(), 0.0) for x in (t, h, p)]
    c_args = ops + [c_int(1), c_int(0), c_int(1), c_int(1), c_void_p(ept.data_ptr()), c_void_p(wb.data_ptr()), c_int64(t.numel())]

    def step():
        _backend._call("ept_wet_bulb", t.dtype, t.device, c_args)

    return step, esz * 5, {"ept": ept, "wbpt": wb}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms; only samples that arrive inside the timed
    region [mark_begin, mark_end] are reported."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.t0, self.t1 = index, None, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [ln for ts, ln in self.lines if self.t0 <= ts <= self.t1 + 0.06]
        if not inside:  # a timed region shorter than one sampling period: take the sample closest to it
            inside = [min(self.lines, key=lambda x: abs(x[0] - self.t1))[1]] if self.lines else []
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# parity of the TIMED buffers: a strided sample of what the timed steps wrote, against the oracle
# --------------------------------------------------------------------------------------------------
def parity_sample(kind, outputs, arrays, hyb, out, npl, dtype, n_target=1 << 20):
    """>= n_target points taken at a fixed odd stride from the buffers the timed steps read and wrote; the oracle (numpy
    restatement of the reference, oracle/thermo_oracle.py) is evaluated on the same input values in the working dtype."""
    import torch

    import thermo_oracle as oracle

    n = arrays[0].numel()
    stride = max(1, n // n_target) | 1
    idx = torch.arange(0, n, stride, device=arrays[0].device)
    t, h = (arrays[k][idx].cpu().numpy() for k in (0, 1))
    if kind == "hybrid":  # p = ph_k + 0.5 (ph_k+1 - ph_k), ph = A + B sp (reference vertical.py:663,708), in the working dtype
        sp, a, b = (x.cpu().numpy() for x in hyb)
        ii = idx.cpu().numpy()
        k, col = ii // npl, ii % npl
        ph0, ph1 = a[k] + b[k] * sp[col], a[k + 1] + b[k + 1] * sp[col]
        p = ph0 + t.dtype.type(0.5) * (ph1 - ph0)
    else:
        p = arrays[2][idx].cpu().numpy()
    limit = 1e-12 if dtype == "f64" else 1e-5
    res = {"n": int(idx.numel()), "stride": int(stride), "limit": limit, "max_rel": 0.0, "n_over_limit": 0, "nan_mismatches": 0,
           "inf_mismatches": 0, "n_nan": 0, "checker": "oracle/thermo_oracle.py on the timed buffers' own input values", "per_output": {}}
    fns = OUT_FNS[kind]
    with np.errstate(all="ignore"):
        for name in outputs:
            got = out[name][idx].cpu().numpy().astype(np.float64)
            want = np.asarray(fns[name](oracle, t, h, p)).astype(np.float64)
            nan_g, nan_w = np.isnan(got), np.isnan(want)
            inf_bad = int(np.sum((np.isinf(got) | np.isinf(want)) & ~(got == want) & ~(nan_g | nan_w)))
            fin = np.isfinite(got) & np.isfinite(want)
            rel = np.abs(got[fin] - want[fin]) / np.maximum(np.abs(want[fin]), 1e-300)
            po = {"max_rel": float(rel.max()) if rel.size else 0.0, "n_over_limit": int(np.sum(rel > limit)),
                  "nan_mismatches": int(np.sum(nan_g != nan_w)), "n_nan": int(nan_w.sum())}
            res["per_output"][name] = po
            res["max_rel"] = max(res["max_rel"], po["max_rel"])
            res["n_over_limit"] += po["n_over_limit"]
            res["nan_mismatches"] += po["nan_mismatches"]
            res["inf_mismatches"] += inf_bad
            res["n_nan"] += po["n_nan"]
    res["ok"] = bool(res["n_over_limit"] == 0 and res["nan_mismatches"] == 0 and res["inf_mismatches"] == 0)
    return res


def dump_outputs(path, out, seed=0):
    """Every output of one step as <path>/<name>.npy (flat, in the working dtype): all points when the outputs fit in
    DUMP_BYTES, else the same sample of points for every output, drawn from `seed` and fixed by the field size, the dtype and
    the number of outputs -- so two builds of the project run with the same arguments can be compared output for output."""
    import torch

    os.makedirs(path, exist_ok=True)
    first = next(iter(out.values()))
    n = first.numel()
    k = min(n, (DUMP_BYTES - (64 << 10)) // (first.element_size() * len(out)))  # 64 KB left for the .npy headers
    idx = None
    if k < n:
        idx = torch.from_numpy(np.sort(np.random.default_rng(seed).choice(n, k, replace=False))).to(first.device)
    for name, x in out.items():
        x = x.reshape(-1)
        np.save(os.path.join(path, f"{name}.npy"), (x if idx is None else x[idx]).cpu().numpy())


# --------------------------------------------------------------------------------------------------
# CPU legs: the reference (oracle/_ref) on level slabs of the same field
# --------------------------------------------------------------------------------------------------
def cpu_field(kind, npl, levels, seed):
    """The generator of the GPU arm, on the device when there is one (same values as the GPU arm's field), else on the CPU."""
    import torch

    dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    return IfsField("tqp" if kind == "ept" else kind, npl, levels=levels, seed=seed, device=dev), dev


def cpu_baseline_single_core(kind, outputs, npl, levels, dtype, budget_s=12.0):
    """The reference on ONE core (as it ships: numpy is single-threaded) over level slabs spread through the column."""
    module, mkind = cpu_module()
    field, dev = cpu_field(kind, npl, levels, 0)
    lv = sample_levels(levels, 4)
    t, h, p = field.slabs_numpy(lv, np.float64 if dtype == "f64" else np.float32)
    fn = cpu_step(kind, outputs, module)
    with np.errstate(all="ignore"):
        fn(t[:10000], h[:10000], p[:10000])
        done, t0 = 0, time.perf_counter()
        while True:
            fn(t, h, p)
            done += 1
            el = time.perf_counter() - t0
            if el > budget_s or done >= 4:
                break
    return {"value": done * t.size / el, "unit": "grid-points/s", "cores": 1, "kind": mkind,
            "sample": f"{done} pass(es) over levels {lv} of the workload's field ({t.size} points, {dtype}, generated on {dev}, seed 0), "
                      f"{'unmodified reference from oracle/_ref' if mkind == 'reference' else 'numpy oracle port'}, {el:.1f} s"}


_W = {}


def _worker_run(args):
    b, e = args
    with np.errstate(all="ignore"):
        res = _W["fn"](*(x[b:e] for x in _W["arr"]))
    return float(sum(np.nansum(r[:8]) for r in res))  # results stay in the worker (as they would stay in RAM)


def run_reference(args, wl):
    import multiprocessing as mp

    import build_ref

    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    kind, outputs, levels, npl, dtype = wl["kind"], wl["outputs"], wl["levels"], wl["npl"], wl["dtype"]
    tests_line = None
    if build_ref.installed():
        n_files, bad = build_ref.verify()
        assert not bad, f"oracle/_ref differs from the reference it was installed from: {bad[:3]}"
        ok, tests_line = build_ref.run_reference_tests()
        print(f"[reference arm] {n_files} installed files verified against their source hashes; reference tests/thermo/test_thermo.py: {tests_line}",
              file=sys.stderr, flush=True)
        assert ok, tests_line
    module, mkind = cpu_module()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    field, dev = cpu_field(kind, npl, levels, 0)
    lv = sample_levels(levels, 8)
    npd = np.float64 if dtype == "f64" else np.float32
    # one step = one slab of npl points made of equal parts of eight levels spread through the column (top, mixed-phase band,
    # boundary layer): every step costs the same and represents the whole field, whatever --steps is
    part = npl // len(lv)
    pieces = [[x[:part] for x in field.slabs_numpy([k], npd)] for k in lv]
    _W["arr"] = [np.ascontiguousarray(np.concatenate([pc[i] for pc in pieces])) for i in range(3)]
    n_step = int(_W["arr"][0].size)
    _W["fn"] = cpu_step(kind, outputs, module)
    del field, pieces
    ctx = mp.get_context("fork")  # the workers inherit the input slab and the imported reference; they never touch CUDA
    with ctx.Pool(cores) as pool:
        edges = np.linspace(0, n_step, cores * 4 + 1).astype(np.int64)
        chunks = [(int(b), int(e)) for b, e in zip(edges[:-1], edges[1:])]
        for _ in range(max(args.warmup, 1)):
            pool.map(_worker_run, chunks)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_worker_run, chunks)
        el = time.perf_counter() - t0
    npl = n_step
    value = args.steps * npl / el
    src = "unmodified reference (oracle/_ref, earthkit.meteo.thermo public functions)" if mkind == "reference" else "numpy oracle port of the reference"
    sample = (f"{npl} points per step: {part} points from each of the levels {lv} of the workload's own field "
              f"(generated on {dev}, seed 0, same generator as the GPU arm), {src}, {cores} processes")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "grid-points/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": dtype, "data": "synthetic",
        "config": {"workload": args.workload, "outputs": list(outputs), "levels": levels, "points_per_level": npl,
                   "points_per_step": int(npl), "l2": "n/a (CPU)"},
        "cpu_baseline": {"value": value, "unit": "grid-points/s", "cores": cores, "kind": mkind, "sample": sample},
        "e2e": {"value": value, "unit": "grid-points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_tests": tests_line, "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def shard_plan(wl, world, rank):
    """(first slab, number of slabs, capped?) of this rank.  Weak workloads: `members` x levels slabs on every rank.
    Sharded workloads: the rank's ek_thermo.partition shard of all members x levels slabs, capped to what fits in HBM."""
    from ek_thermo import partition

    npl, slabs_total = wl["npl"], wl["slabs"]
    if not wl["sharded"]:
        return 0, slabs_total, False
    b, e = partition.shard_range(slabs_total * npl, world, rank, align=npl)
    first, count = b // npl, (e - b) // npl
    esz = 8 if wl["dtype"] == "f64" else 4
    cap = int(HBM_BUDGET_BYTES // (esz * (3 + len(wl["outputs"])) * npl))
    return first, min(count, cap), count > cap


def slab_stats(out, outputs, j, npl):
    """Per-output (NaN count, sum of the finite values) of slab j of the resident results: the cross-shard checksum."""
    import torch

    res = []
    for name in outputs:
        x = out[name][j * npl:(j + 1) * npl]
        res.append((int(torch.isnan(x).sum().item()), float(torch.nansum(x.double()).item())))
    return res


def run_ours(args, wl):
    import torch

    import ek_thermo
    from ek_thermo import hostpipe

    kind, outputs, levels, npl, dtype = wl["kind"], wl["outputs"], wl["levels"], wl["npl"], wl["dtype"]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    numa_cpus = hostpipe.bind_host_to_device(device) if world > 1 else None  # pinned e2e buffers next to the rank's GPU
    dist = gloo = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=device)
        gloo = dist.new_group(backend="gloo")  # host-side object exchange of the shard check; no tensor data travels

    tdt = torch.float64 if dtype == "f64" else torch.float32
    first, n_slabs, capped = shard_plan(wl, world, rank)
    field = IfsField("tqp" if kind == "ept" else kind, npl, levels=levels, seed=(0 if wl["sharded"] else rank), device=device)
    arrays = field.materialise(first, n_slabs, tdt)
    n = n_slabs * npl
    hyb = None
    if kind == "hybrid":
        hyb = (field.sp(0).to(tdt), torch.tensor(field.A_half, dtype=tdt, device=device), torch.tensor(field.B_half, dtype=tdt, device=device))
        arrays[2] = None  # the pressure field is never materialised for the kernel
    step, bytes_per_pt, out = build_step(kind, outputs, arrays, hyb)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        tt = torch.tensor([x], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = ek_thermo.launch_count()
    barrier()
    sampler.mark_begin()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    sampler.mark_end()
    launches = ek_thermo.launch_count() - launches0
    ms_own = ev0.elapsed_time(ev1) / args.steps
    ms_step = max_over_ranks(ms_own)
    n_all = sum_over_ranks(float(n))
    clocks = sampler.stop() if rank == 0 else None
    value = n_all / (ms_step * 1e-3)

    # ---- parity of the timed buffers (rank 0's field; every rank's for the sharded workload through the shard check)
    parity = parity_sample(kind, outputs, arrays, hyb, out, npl, dtype) if (rank == 0 and not args.no_parity) else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step.last_out() if hasattr(step, "last_out") else out)

    # ---- cross-shard check (SURVEY.md 8(e)): probe slabs of every shard are recomputed on rank 0 from the same seed
    shard_check = None
    if wl["sharded"]:
        probes = sorted({0, n_slabs // 2, n_slabs - 1})
        mine = [(first + j, slab_stats(out, outputs, j, npl)) for j in probes]
        gathered = [mine]
        if dist is not None:
            gathered = [None] * world
            dist.all_gather_object(gathered, mine, group=gloo)
        if rank == 0:
            from ek_thermo import fused

            bad = []
            for r, lst in enumerate(gathered):
                for s, stats in lst:
                    t1, h1, p1 = (x.to(tdt) for x in field.slab(s))
                    o1 = fused.suite_tqp(t1, h1, p1, outputs=outputs)
                    if slab_stats(o1, outputs, 0, npl) != stats:
                        bad.append((r, s))
            n_probe = sum(len(x) for x in gathered)
            shard_check = (f"ok ({n_probe} probe slabs of {world} shard(s) recomputed on rank 0 from the seed: per-output NaN counts and checksums identical)"
                           if not bad else f"MISMATCH at (rank, slab) {bad[:8]}")

    # ---- e2e: the host-buffer call (host arrays in, host arrays out), copies inside the timed region
    e2e = e2e_pageable = None
    if not args.no_e2e:
        e2e, e2e_pageable = run_e2e(args, wl, arrays, hyb, out, n_slabs, device, world, barrier, max_over_ranks, field)

    if rank == 0:
        peak, peak_src = load_peaks()
        achieved = bytes_per_pt * n / (ms_own * 1e-3) / 1e9  # rank 0's GPU: one kernel per step
        cpu = cpu_baseline_single_core(kind, outputs, npl, levels, dtype) if world == 1 and not args.no_cpu else None
        scaling = "weak"
        if wl["sharded"]:
            scaling = "strong" if not capped else "strong (capped: this N cannot hold the whole ensemble, see config.shard)"
        line = {
            "metric": METRIC, "value": value, "unit": "grid-points/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": {"workload": args.workload, "outputs": list(outputs), "levels": levels, "points_per_level": npl,
                       "points_per_gpu": n, "points_all_gpus": int(n_all), "bytes_per_point": bytes_per_pt,
                       "parallelism": f"shard x{world} (no data-path collective; NCCL only for the barrier and the max of the device time)",
                       "shard": (f"rank 0 owns slabs [{first}, {first + n_slabs}) of {wl['slabs']} (member x level slabs of {npl} points)"
                                 + (f"; capped to {n_slabs} slabs = {HBM_BUDGET_BYTES / 1e9:.0f} GB per GPU" if capped else "")) if wl["sharded"]
                       else f"every rank runs its own {wl['slabs']} level slabs (seed = rank)",
                       "host_cpus_rank0": (f"{len(numa_cpus)} CPUs local to the GPU" if numa_cpus else "unbound"),
                       "l2": ("inputs+outputs per step (%.1f GB) exceed the 126 MB L2; no flush needed" % (bytes_per_pt * n / 1e9)
                              if getattr(step, "n_sets", 1) == 1 else
                              "inputs+outputs per step are %.1f MB (< 126 MB L2): steps rotate over %d buffer sets (%.0f MB), so no launch finds its inputs in L2"
                              % (bytes_per_pt * n / 1e6, step.n_sets, step.n_sets * bytes_per_pt * n / 1e6))},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": load_traffic(args.workload), "peak_source": peak_src,
                         "kernel": {"ept": "ew_kernel<OpEptWb>", "tqp": "ew_kernel<OpSuiteTQPm>", "ttdp": "ew_kernel<OpSuiteTTdPm>",
                                    "hybrid": "suite_hybrid_kernel<OpSuiteTQPm>"}[kind],
                         "algorithmic_bytes_per_launch": bytes_per_pt * n, "avg_launch_ms": ms_own},
            "parity": parity, "cpu_baseline": cpu, "e2e": e2e, "e2e_pageable": e2e_pageable, "clocks": clocks, "gpu_launches": int(launches),
        }
        if shard_check is not None:
            line["shard_check"] = shard_check
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def run_e2e(args, wl, arrays, hyb, out, n_slabs, device, world, barrier, max_over_ranks, field):
    """`e2e`: page-locked host arrays -> ek_thermo.hostpipe.HostSuite (one C call: chunked H2D, kernel, D2H on 3 streams) ->
    page-locked host arrays.  `e2e_pageable`: ordinary numpy arrays -> ek_thermo.host.fused (staging threads) -> fresh result
    arrays: the drop-in call of a numpy user.  Both are timed with the copies inside, on the first levels of the field."""
    import torch

    from ek_thermo import host, hostpipe

    kind, outputs, npl, dtype = wl["kind"], wl["outputs"], wl["npl"], wl["dtype"]
    lv = max(1, min(n_slabs, args.e2e_levels))
    n_e2e = lv * npl
    npd = np.float64 if dtype == "f64" else np.float32
    esz = np.dtype(npd).itemsize
    steps = max(2, min(args.steps, args.e2e_steps))
    hs = hostpipe.HostSuite(device, workspace_bytes=args.e2e_workspace_mb << 20, n_slots=3)
    h_out = {name: hostpipe.pinned_empty(n_e2e, npd) for name in outputs}
    if kind == "hybrid":  # the lv bottom-most levels of the column (the band needs its own half-level coefficients)
        nlev = n_slabs
        rows = slice((nlev - lv) * npl, nlev * npl)
        h_t, h_q = (hostpipe.pinned_empty(n_e2e, npd) for _ in range(2))
        h_t[:] = arrays[0][rows].cpu().numpy()
        h_q[:] = arrays[1][rows].cpu().numpy()
        h_sp = hostpipe.pinned_empty(npl, npd)
        h_sp[:] = hyb[0].cpu().numpy()
        a, b = hyb[1][nlev - lv:].cpu().numpy(), hyb[2][nlev - lv:].cpu().numpy()
        o2 = {k: v.reshape(lv, npl) for k, v in h_out.items()}

        def call():
            hs.suite_tq_hybrid(h_t.reshape(lv, npl), h_q.reshape(lv, npl), h_sp, a, b, outputs=outputs, out=o2)

        h2d = esz * (2 * n_e2e + npl)
        check_rows = rows
        pageable_call = None
    else:
        h_in = [hostpipe.pinned_empty(n_e2e, npd) for _ in range(3)]
        for hbuf, d in zip(h_in, arrays):
            hbuf[:] = d[:n_e2e].cpu().numpy()
        fn = hs.suite_ttdp if kind == "ttdp" else hs.suite_tqp

        def call():
            fn(*h_in, outputs=outputs, out=h_out)  # blocks until the outputs are in host memory

        h2d = 3 * esz * n_e2e
        check_rows = slice(0, n_e2e)
        p_in = [np.array(x) for x in h_in]  # ordinary (pageable) numpy copies
        pfn = host.fused.suite_ttdp if kind == "ttdp" else host.fused.suite_tqp

        def pageable_call():
            return pfn(*p_in, outputs=outputs)

    per_step = []

    def timed(f):
        f()
        barrier()
        per_step.clear()
        t0 = time.perf_counter()
        for _ in range(steps):
            t1 = time.perf_counter()
            f()
            per_step.append(round(time.perf_counter() - t1, 4))
        torch.cuda.synchronize()
        return max_over_ranks(time.perf_counter() - t0)

    el = timed(call)
    e2e = {"value": world * steps * n_e2e / el, "unit": "grid-points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": len(outputs) * esz * n_e2e,
           "steps": steps, "step_seconds_rank0": list(per_step), "value_median_step_rank0": n_e2e / float(np.median(per_step)),
           "pcie_gbs_all_gpus": world * (h2d + len(outputs) * esz * n_e2e) * steps / el / 1e9,
           "sample": f"{lv} of {n_slabs} level slabs per step ({n_e2e} points) through ek_thermo.hostpipe.HostSuite, page-locked host buffers"}
    # the device result of the timed steps and the host-pipeline result agree bit for bit on the shared slab
    name0 = outputs[0]
    dev_res = out[name0][check_rows][:100000].cpu().numpy()
    assert np.array_equal(h_out[name0][:100000], dev_res, equal_nan=True), "host pipeline and device path differ"
    e2e_pageable = None
    if pageable_call is not None and not args.no_e2e_pageable:
        res = {}

        def pc():
            res.clear()  # the previous step's result arrays are dropped, as a caller's loop would
            res.update(pageable_call())

        el = timed(pc)
        assert np.array_equal(res[name0][:100000], dev_res, equal_nan=True), "host.fused and device path differ"
        e2e_pageable = {"value": world * steps * n_e2e / el, "unit": "grid-points/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": len(outputs) * esz * n_e2e, "steps": steps, "step_seconds_rank0": list(per_step),
                        # the staging threads share the VM's cores: single steps of 3-8 x the median turn up on busy hosts
                        "value_median_step_rank0": n_e2e / float(np.median(per_step)),
                        "sample": f"{n_e2e} points per step through ek_thermo.host.fused: pageable numpy arrays in (staged by worker threads), "
                                  "fresh page-locked result arrays out (torch's caching host allocator; first call excluded as warm-up)"}
        host.release_staging()
    return e2e, e2e_pageable


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--levels", type=int, default=0, help="override the number of levels (smaller field: the lowest N model levels)")
    ap.add_argument("--members", type=int, default=0, help="override the number of members of an ensemble workload")
    ap.add_argument("--e2e-levels", type=int, default=16)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-workspace-mb", type=int, default=768)
    ap.add_argument("--no-cpu", action="store_true", help="skip the single-core CPU baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer legs")
    ap.add_argument("--no-e2e-pageable", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed buffers")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) to DIR/<name>.npy, "
                    "at most 64 MB in all: a fixed seeded sample of points when the whole outputs are larger")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the device path (--impl ours)")
    wl = dict(WORKLOADS[args.workload])
    if args.levels:
        wl["levels"] = args.levels
        wl["slabs"] = wl["members"] * wl["levels"]
    if args.members:
        wl["members"] = args.members
        wl["slabs"] = wl["members"] * wl["levels"]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
