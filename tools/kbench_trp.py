#!/usr/bin/env python
"""kbench_trp.py -- the fused (t, r, p) suite against the chain of launches it replaces, alternated in one session on one GPU.

    python tools/kbench_trp.py [--steps 10] [--reps 5] [--only o1280_f64_default,...]

A caller holding (t, r, p) who wants the default fields without the suite runs three kernels:
    q  = specific_humidity_from_relative_humidity(t, r, p)     reads t, r, p  writes q
    td = dewpoint_from_relative_humidity(t, r)                 reads t, r     writes td
    suite_tqp(t, q, p, outputs=("theta", "es", "tv"))          reads t, q, p  writes three fields
= 13 arrays per point (104 B in float64) against the suite's 8 (64 B).  The single pass (theta, td, q, ept, wbpt) has the same
counts.  Workloads:
  * o1280_{f64,f32}_{default,single}: O1280 x 137 IFS-shaped model-level fields (tools/synthetic.IfsField, r from
    relative_humidity_from_specific_humidity of its physical q), one array per input;
  * era5_37_f64_default: 37 ERA5 pressure levels of 721 x 1440 points, one allocation per level, pressure one number per level:
    one suite_trp_batch launch against the chain level by level (111 launches).
Each repetition times `--steps` calls of the fused form, then `--steps` calls of the chain, with CUDA events; reported are the
median and range over the repetitions of ms per call, Gpt/s and the fraction of the algorithmic-bytes roofline (arrays touched
x element size x points over the HBM bandwidth: MEASURED_PEAKS.json when present, else 6551 GB/s as tools/kbench.py).  The
fused outputs are checked against the chain's: bit-identical wherever no output of the point is NaN.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "earthkit-meteo_b200"), os.path.join(ROOT, "tools")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ek_thermo  # noqa: E402
from ek_thermo import fused, thermo  # noqa: E402
from synthetic import N_LEVELS, O1280_POINTS, IfsField  # noqa: E402

DEV = "cuda:0"
ERA5_LEVELS_HPA = [1, 2, 3, 5, 7, 10, 20, 30, 50, 70, 100, 125, 150, 175, 200, 225, 250, 300, 350, 400, 450, 500, 550, 600, 650, 700, 750, 775,
                   800, 825, 850, 875, 900, 925, 950, 975, 1000]
ERA5_POINTS = 721 * 1440


def _peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6551.0


def _gpu():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception:
        return torch.cuda.get_device_name(0)


def _chain(t, r, p, names, keep):
    """The launches a caller without the suite makes for `names`; `keep` holds the outputs (reused across calls)."""
    keep["q"] = thermo.specific_humidity_from_relative_humidity(t, r, p)
    keep["td"] = thermo.dewpoint_from_relative_humidity(t, r)
    rest = tuple(k for k in names if k not in ("q", "td"))
    keep.update(fused.suite_tqp(t, keep["q"], p, outputs=rest))
    return keep


def _ifs_field(dtype):
    """O1280 x 137 (t, r, p) as flat device arrays of `dtype`."""
    f = IfsField("tqp", O1280_POINTS, levels=N_LEVELS, seed=0, device=DEV)
    t, q, p = f.materialise(0, N_LEVELS, dtype)
    r = thermo.relative_humidity_from_specific_humidity(t, q, p)
    del q
    torch.cuda.synchronize()
    return t, r, p


def _era5():
    """37 levels of (t, r) in separate allocations, float64, and the level pressures in Pa."""
    g = torch.Generator(device=DEV).manual_seed(1)
    ts, rs, ps = [], [], []
    for hpa in ERA5_LEVELS_HPA:
        p = 100.0 * hpa
        t = (288.15 * (p / 101325.0) ** 0.19 + torch.empty(ERA5_POINTS, dtype=torch.float64, device=DEV).uniform_(-15, 15, generator=g)).clamp_(180, 320)
        ts.append(t)
        rs.append(torch.empty(ERA5_POINTS, dtype=torch.float64, device=DEV).uniform_(1.0, 100.0, generator=g))
        ps.append(p)
    return ts, rs, ps


def _same_where_finite(a, b):
    """(bit-identical where both are free of NaN, NaN positions equal)"""
    ok = ~torch.isnan(a) & ~torch.isnan(b)
    return bool(torch.equal(torch.isnan(a), torch.isnan(b))) and bool((a[ok] == b[ok]).all())


def _time(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run(name, fused_fn, chain_fn, n, esz, arrays_fused, arrays_chain, check, steps, reps, peak):
    for fn in (fused_fn, chain_fn):  # warm-up: module load, allocator, the lean tables
        fn()
        fn()
    torch.cuda.synchronize()
    ms = {"fused": [], "chain": []}
    for _ in range(reps):  # alternated in one session
        ms["fused"].append(_time(fused_fn, steps))
        ms["chain"].append(_time(chain_fn, steps))
    res = {"workload": name, "points": n, "steps": steps, "reps": reps}
    for k, arrays in (("fused", arrays_fused), ("chain", arrays_chain)):
        v = np.array(ms[k])
        med = float(np.median(v))
        res[k] = {"ms_median": round(med, 4), "ms_min": round(float(v.min()), 4), "ms_max": round(float(v.max()), 4),
                  "gpts": round(n / med / 1e6, 2), "bytes_per_point": arrays * esz,
                  "frac_roofline": round(arrays * esz * n / med / 1e6 / peak, 3)}
    res["speedup"] = round(res["chain"]["ms_median"] / res["fused"]["ms_median"], 3)
    res["fused_equals_chain"] = check()
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    only = [s for s in a.only.split(",") if s]
    peak = _peak()
    print(json.dumps({"gpu": _gpu(), "lib": os.path.basename(ek_thermo._backend.LIB_PATH), "peak_gbs": peak, "torch": torch.__version__}), flush=True)
    sets = {"default": fused.DEFAULT_TRP, "single": fused.SINGLE_PASS_TRP}
    for dname, dtype, esz in (("f64", torch.float64, 8), ("f32", torch.float32, 4)):
        names = [f"o1280_{dname}_{s}" for s in sets]
        if only and not any(x in only for x in names):
            continue
        t, r, p = _ifs_field(dtype)
        n = t.numel()
        for sname, outs in sets.items():
            name = f"o1280_{dname}_{sname}"
            if only and name not in only:
                continue
            fo = {k: torch.empty_like(t) for k in outs}
            keep = {}

            def check(outs=outs, fo=fo, keep=keep):
                return all(_same_where_finite(fo[k], keep[k]) for k in outs)

            run(name, lambda outs=outs, fo=fo: fused.suite_trp(t, r, p, outputs=outs, out=fo), lambda outs=outs, keep=keep: _chain(t, r, p, outs, keep),
                n, esz, 3 + len(outs), 13, check, a.steps, a.reps, peak)
            del fo, keep
        del t, r, p
        torch.cuda.empty_cache()
    name = "era5_37_f64_default"
    if not only or name in only:
        ts, rs, ps = _era5()
        outs = fused.DEFAULT_TRP
        fo = [{k: torch.empty_like(ts[0]) for k in outs} for _ in ts]
        keep = [dict() for _ in ts]

        def chain():
            for j in range(len(ts)):
                _chain(ts[j], rs[j], ps[j], outs, keep[j])

        def check():
            return all(_same_where_finite(fo[j][k], keep[j][k]) for j in range(len(ts)) for k in outs)

        # fused: t, r in + 5 out; chain: q (t, r -> q), td (t, r -> td), suite_tqp (t, q -> 3): 11 arrays; p is one number per level
        run(name, lambda: fused.suite_trp_batch(ts, rs, ps, outputs=outs, out=fo), chain, len(ts) * ERA5_POINTS, 8, 7, 11, check, a.steps * 5,
            a.reps, peak)


if __name__ == "__main__":
    main()
