#!/usr/bin/env python
"""kbench_hybrid.py -- timing of the hybrid-level kernels (SURVEY.md 8(f)-1/2) on O1280 x 137 levels, one GPU.

    python tools/kbench_hybrid.py [--f32]                 every hybrid kernel on O1280 x 137
    python tools/kbench_hybrid.py --geo [--f32] [--columns N,...]
        "suite_tq_hybrid 5 outputs + z, fused" against "suite_tq_hybrid then geopotential_on_hybrid_levels", alternated in one
        run, on O1280 and ERA5 x 137 and on small fields on both sides of GEO_FUSED_MIN_COLUMNS (default), or on the given
        column counts.  The fused rows force the fused kernel; "wrapper" says which of the two suite_tq_hybrid picks there."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "earthkit-meteo_b200"), os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from ek_thermo import fused, vertical  # noqa: E402

dev = "cuda:0"
nlev = 137
dtype = torch.float64 if "--f32" not in sys.argv else torch.float32
esz = 8 if dtype == torch.float64 else 4
ab = np.load(os.path.join(ROOT, "tests", "golden", "ifs_l137_ab.npz"))
A, B = torch.tensor(ab["A"], dtype=dtype, device=dev), torch.tensor(ab["B"], dtype=dtype, device=dev)
peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
print(f"device={torch.cuda.get_device_name(0)} dtype={dtype} peak={peak} GB/s")


def fields(npl, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    sp = torch.empty(npl, device=dev, dtype=dtype).uniform_(5.0e4, 1.05e5, generator=g)
    zs = torch.empty(npl, device=dev, dtype=dtype).uniform_(-300.0, 3.0e4, generator=g)
    p = vertical.pressure_on_hybrid_levels(A, B, sp)
    t = (288.15 * (p / 101325.0) ** 0.19 + torch.empty_like(p).uniform_(-15, 15, generator=g)).clamp_(180, 320)
    q = torch.empty_like(p).uniform_(1.0e-6, 0.02, generator=g)
    del p
    return sp, zs, t, q


def time_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        r = fn()
        del r
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def geo_main():
    """The fused suite + geopotential call against the two launches it replaces, alternated (rounds x reps calls each)."""
    key = "float64" if dtype == torch.float64 else "float32"
    thr = fused.GEO_FUSED_MIN_COLUMNS[key]
    # O1280, ERA5 0.25 deg (721 x 1440), and small fields: the wrapper's threshold and half of it (one case on each side)
    cols = [int(x) for x in sys.argv[sys.argv.index("--columns") + 1].split(",")] if "--columns" in sys.argv else \
        [4 * 1280 * 1289, 1038240, 262144, thr, thr // 2]
    names = fused.DEFAULT_TQP + ("z",)
    for npl in cols:
        sp, zs, t, q = fields(npl)
        n = npl * nlev
        bpp = esz * (2 + len(fused.DEFAULT_TQP) + 1) + esz * 2 / nlev  # t, q, 5 outputs, z per element; sp, zs per column

        def fused_call():
            fused.GEO_FUSED_MIN_COLUMNS[key] = 0
            return fused.suite_tq_hybrid(t, q, sp, A, B, outputs=names, zs=zs)

        def two_calls():
            return fused.suite_tq_hybrid(t, q, sp, A, B), vertical.geopotential_on_hybrid_levels(t, q, zs, A, B, sp)

        variants = {"suite_tq_hybrid 5 outputs + z, fused": fused_call, "suite_tq_hybrid then geopotential_on_hybrid_levels": two_calls}
        reps = 5 if n > 1e8 else 50
        for fn in variants.values():
            for _ in range(2):
                r = fn()
            del r
        torch.cuda.synchronize()
        ms = {k: [] for k in variants}
        for _ in range(5):  # alternate the two variants
            for k, fn in variants.items():
                ms[k].append(time_ms(fn, reps))
        fused.GEO_FUSED_MIN_COLUMNS[key] = thr
        for k, v in ms.items():
            best, med = min(v), sorted(v)[len(v) // 2]
            gbs = bpp * n / med / 1e6
            print(f"columns={npl:8d} x {nlev} {k:52s} median {med:8.3f} ms (best {best:8.3f}) {gbs:8.1f} GB/s frac={gbs / peak:.3f}")
        f, s2 = (sorted(v)[len(v) // 2] for v in ms.values())
        print(f"columns={npl:8d} x {nlev} fused / two launches = {f / s2:.3f}; the wrapper runs the {'fused kernel' if npl >= thr else 'two launches'}")
        del sp, zs, t, q
        torch.cuda.empty_cache()


def main():
    npl = 4 * 1280 * 1289
    sp, zs, t, q = fields(npl)
    n = npl * nlev
    kernels = {
        # name: (callable, algorithmic bytes per [level, point] element)
        "pressure full": (lambda: vertical.pressure_on_hybrid_levels(A, B, sp), esz * (1 + 1 / nlev)),
        # delta and alpha are float64 arrays whatever the dtype of sp (as in the reference)
        "pressure full+half+delta+alpha": (lambda: vertical.pressure_on_hybrid_levels(A, B, sp, output=("full", "half", "delta", "alpha")), esz * (2 + 2 / nlev) + 16),
        "thickness (alpha/delta in registers)": (lambda: vertical.relative_geopotential_thickness_on_hybrid_levels(t, q, A, B, sp), esz * (3 + 1 / nlev)),
        "geometric height above ground": (lambda: vertical.height_on_hybrid_levels(t, q, zs, A, B, sp), esz * (3 + 2 / nlev)),
        "suite_tq_hybrid (5 outputs)": (lambda: fused.suite_tq_hybrid(t, q, sp, A, B), esz * (7 + 1 / nlev)),
    }
    print(f"points={n}")
    for name, (fn, bpp) in kernels.items():
        for _ in range(2):
            r = fn()
        del r
        torch.cuda.synchronize()
        ms = time_ms(fn, 5)
        gbs = bpp * n / ms / 1e6
        print(f"{name:40s} {ms:8.3f} ms {n / ms / 1e6:8.2f} Gpt/s {gbs:8.1f} GB/s frac={gbs / peak:.3f}")


if __name__ == "__main__":
    geo_main() if "--geo" in sys.argv else main()
