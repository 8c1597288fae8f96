#!/usr/bin/env python
"""hostbench_hybrid.py -- HostSuite.suite_tq_hybrid on host arrays, with and without the geopotential "z", one GPU.

    python tools/hostbench_hybrid.py [--columns 262144] [--f32]

Page-locked numpy arrays of [137, columns] in and out; wall-clock per call, best and median of 5, after a warm-up call.
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "earthkit-meteo_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from ek_thermo import fused, hostpipe  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--columns", type=int, default=1 << 18)
    ap.add_argument("--f32", action="store_true")
    a = ap.parse_args()
    dt = np.float32 if a.f32 else np.float64
    npl, nlev = a.columns, 137
    ab = np.load(os.path.join(ROOT, "tests", "golden", "ifs_l137_ab.npz"))
    A, B = ab["A"].astype(dt), ab["B"].astype(dt)
    rng = np.random.default_rng(0)

    def pinned(x):
        p = hostpipe.pinned_empty(x.size, dt).reshape(x.shape)
        p[...] = x
        return p

    sp = pinned(rng.uniform(5.0e4, 1.05e5, npl))
    zs = pinned(rng.uniform(-300.0, 3.0e4, npl))
    t = pinned(rng.uniform(200.0, 300.0, (nlev, npl)))
    q = pinned(rng.uniform(1.0e-6, 0.02, (nlev, npl)))
    hs = hostpipe.HostSuite("cuda:0")
    print(f"device={torch.cuda.get_device_name(0)} dtype={np.dtype(dt).name} columns={npl} levels={nlev}")
    for label, names in (("5 outputs", fused.DEFAULT_TQP), ("5 outputs + z", fused.DEFAULT_TQP + ("z",))):
        out = {k: pinned(np.empty((nlev, npl))) for k in names}
        hs.suite_tq_hybrid(t, q, sp, A, B, outputs=names, out=out, zs=zs)
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            hs.suite_tq_hybrid(t, q, sp, A, B, outputs=names, out=out, zs=zs)
            ts.append(time.perf_counter() - t0)
        ts.sort()
        moved = np.dtype(dt).itemsize * nlev * npl * (2 + len(names)) + np.dtype(dt).itemsize * npl * 2
        print(f"HostSuite.suite_tq_hybrid {label:14s} best {ts[0] * 1e3:8.2f} ms median {ts[2] * 1e3:8.2f} ms  {moved / ts[2] / 1e9:6.2f} GB/s over PCIe")


if __name__ == "__main__":
    main()
