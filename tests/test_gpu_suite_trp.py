"""The (t, r, p) suite on the GPU: parity with the oracle composition, bit-identity with the single-function kernels and the
(t, q, p) suite it stands for, the batched and pressure-level forms, the host-array front ends, and both libraries."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import thermo_oracle as oracle
from cases import edge_inputs, random_inputs
from trp_parity import check_suite

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
N_RANDOM = 256 * 4 * 37 + 77  # several tiles, a scalar tail and a ragged end
METHODS = ["ifs", "bolton35", "bolton39"]


@pytest.fixture(scope="module")
def ek():
    import ek_thermo

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return ek_thermo


def _same(a, b):
    """Bit-identical, NaN positions included."""
    return a.shape == b.shape and bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def _ifs(n_per_level=96, seed=0):
    """IFS-shaped (t, r, p) over all 137 levels: physical r from the reference's relative_humidity_from_specific_humidity."""
    from synthetic import ifs_point_inputs

    d = ifs_point_inputs(n_per_level, seed=seed)
    with np.errstate(all="ignore"):
        r = oracle.relative_humidity_from_specific_humidity(d["t"], d["q"], d["p"])
    return d["t"], r, d["p"]


def _edge(n=4099):
    """edge_inputs' special values (r = 0, r > 100, negative r, NaN, +-inf, band edges) plus p - e straddling the eps rule."""
    with np.errstate(all="ignore"):
        d = edge_inputs(n=n, seed=21)
        t = np.repeat(np.array([300.0, 273.0, 250.0, 230.0]), 16)
        r = np.tile(np.array([100.0, 37.5, 120.0, 1.0]), 16)
        e = r * oracle.saturation_vapour_pressure(t) / 100.0
        p = e + np.tile(np.array([-1e-4, 0.0, 5e-5, 1e-4 - 1e-9, 1e-4, 1e-4 + 1e-9, 2e-4, 1.0]), 8)
    return np.concatenate([d["t"], t]), np.concatenate([d["r"], r]), np.concatenate([d["p"], p])


def _inputs(kind):
    if kind == "random":
        d = random_inputs(N_RANDOM, seed=5)
        return d["t"], d["r"], d["p"]
    return _ifs() if kind == "ifs" else _edge()


def _dev(args, dtype):
    with np.errstate(all="ignore"):
        a = [np.ascontiguousarray(np.asarray(x).astype(dtype)) for x in args]
    return a, [torch.from_numpy(x).to(DEV) for x in a]


# ---- oracle parity -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ept_method", METHODS)
@pytest.mark.parametrize("kind", ["random", "ifs", "edge"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_matches_oracle(ek, dtype, kind, ept_method):
    """All ten outputs in one launch, the default set and the single pass against the composition trp_parity.suite_trp under the
    parity rule of tests/compare.py: NaN and inf positions identical in float64."""
    from ek_thermo import fused

    a, d = _dev(_inputs(kind), dtype)
    sets = [tuple(fused.SUITE_TRP_OUTPUTS)] + ([fused.DEFAULT_TRP, fused.SINGLE_PASS_TRP] if ept_method == "ifs" else [])
    for outputs in sets:
        before = ek.launch_count()
        got = fused.suite_trp(*d, outputs=outputs, ept_method=ept_method)
        assert ek.launch_count() == before + 1 and tuple(got) == outputs
        check_suite({k: v.cpu().numpy() for k, v in got.items()}, a, ept_method, edge=(kind == "edge"))


# ---- bit-identity with the kernels each output stands for -----------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["random", "ifs"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_bits_equal_single_functions_and_tqp_suite(ek, dtype, kind):
    """q and td are the bits of specific_humidity_from_relative_humidity and dewpoint_from_relative_humidity; theta, tv, w, thetav,
    ept and wbpt are the bits of suite_tqp on that q -- wherever every output of the point is finite and below 1e30.  The other
    points are NaN, or unphysical ones (q near 1 at 320 K and 10 hPa in the random set) whose Bolton theta_e reaches 1e40-1e80 K
    or overflows: there a lean primitive leaves its fast domain, the kernel recomputes the point as a whole with the exact
    functor, and the single-function kernels (which never see that theta_e) agree to rounding instead."""
    from ek_thermo import fused

    _, (t, r, p) = _dev(_inputs(kind), dtype)
    chain = ("theta", "tv", "w", "thetav", "ept", "wbpt")
    rtol = 1e-5 if dtype == np.float32 else 1e-11
    for em in METHODS:
        for outputs in ((tuple(fused.SUITE_TRP_OUTPUTS),) + ((fused.DEFAULT_TRP, fused.SINGLE_PASS_TRP) if em == "ifs" else ())):
            got = fused.suite_trp(t, r, p, outputs=outputs, ept_method=em)
            vals = torch.stack(list(got.values()))
            fast = (torch.isfinite(vals) & (vals.abs() < 1e30)).all(0)
            assert float(fast.float().mean()) > 0.9
            pairs = []
            if "q" in got:
                pairs.append(("q", ek.thermo.specific_humidity_from_relative_humidity(t, r, p)))
            if "td" in got:
                pairs.append(("td", ek.thermo.dewpoint_from_relative_humidity(t, r)))
            q = got["q"] if "q" in got else fused.suite_trp(t, r, p, outputs=("q",))["q"]
            names = tuple(k for k in chain if k in got)
            pairs += list(fused.suite_tqp(t, q, p, outputs=names, ept_method=em).items())
            for k, want in pairs:
                assert _same(got[k][fast], want[fast]), (em, outputs, k)
                torch.testing.assert_close(got[k], want, rtol=rtol, atol=0, equal_nan=True, msg=f"{em} {outputs} {k}")


# ---- batched, pressure-level and position -----------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_batch_equals_per_field_calls(ek, dtype):
    """suite_trp_batch over separate fields equals one suite_trp call per field, bit for bit, with a list of pressure fields, one
    pressure per field (pressure-level data) and one scalar pressure; 150 fields take two launches."""
    from ek_thermo import fused

    n_seg, npl = 150, 4099
    t, r, p = _ifs(n_per_level=(n_seg * npl) // 137 + 1, seed=3)
    _, (t, r, p) = _dev((t[:n_seg * npl], r[:n_seg * npl], p[:n_seg * npl]), dtype)
    ts, rs, ps = ([x[j * npl:(j + 1) * npl].clone() for j in range(n_seg)] for x in (t, r, p))
    ts[64][::97] = float("nan")  # missing values: the exact recompute inside the batched kernel
    levels = [float(x) for x in np.linspace(100.0, 101325.0, n_seg)]
    levels[3] = 3.0  # p - e < eps on most points: the NaN rule
    for outputs, em in ((fused.DEFAULT_TRP, "ifs"), (("theta", "td"), "ifs"), (fused.SINGLE_PASS_TRP, "ifs"), (tuple(fused.SUITE_TRP_OUTPUTS), "bolton35")):
        for pp in (ps, levels, 85000.0):
            before = ek.launch_count()
            got = fused.suite_trp_batch(ts, rs, pp, outputs=outputs, ept_method=em)
            assert ek.launch_count() == before + 2 and len(got) == n_seg
            for j in range(n_seg):
                pj = pp[j] if isinstance(pp, list) else pp
                want = fused.suite_trp(ts[j], rs[j], pj, outputs=outputs, ept_method=em)
                for k in outputs:
                    assert _same(got[j][k], want[k]), (outputs, j, k, type(pp))


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_scalar_pressure_equals_materialised_pressure(ek, dtype):
    """The pressure-level tile loop (p one number) gives the bits of the same call with p materialised, for the compile-time and
    the run-time-mask instantiations."""
    from ek_thermo import fused

    _, (t, r, _) = _dev(_inputs("random"), dtype)
    for p0 in (85000.0, 500.0):
        pf = torch.full_like(t, p0)
        for outputs, em in ((fused.DEFAULT_TRP, "ifs"), (fused.SINGLE_PASS_TRP, "ifs"), (tuple(fused.SUITE_TRP_OUTPUTS), "ifs"), (("td", "ept"), "bolton39")):
            a = fused.suite_trp(t, r, p0, outputs=outputs, ept_method=em)
            b = fused.suite_trp(t, r, pf, outputs=outputs, ept_method=em)
            for k in outputs:
                assert _same(a[k], b[k]), (p0, outputs, k)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_result_does_not_depend_on_position(ek, dtype):
    """A point gives the same bits in the vector body or the scalar tail, in a whole-field launch or in pieces with aligned and
    unaligned starts (unaligned views take the scalar load/store path)."""
    from ek_thermo import fused

    _, (t, r, p) = _dev(_inputs("ifs"), dtype)
    for outputs in (fused.DEFAULT_TRP, fused.SINGLE_PASS_TRP, tuple(fused.SUITE_TRP_OUTPUTS)):
        whole = fused.suite_trp(t, r, p, outputs=outputs)
        for lo, hi in ((1, 5001), (2, 8194), (3, t.numel()), (4096, t.numel() - 7)):
            part = fused.suite_trp(t[lo:hi], r[lo:hi], p[lo:hi], outputs=outputs)
            for k in outputs:
                assert _same(part[k], whole[k][lo:hi]), (lo, hi, k)
        shift = 1001
        rolled = fused.suite_trp(*(torch.roll(x, shift) for x in (t, r, p)), outputs=outputs)
        for k in outputs:
            assert _same(rolled[k], torch.roll(whole[k], shift)), k


# ---- host-array front ends ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_host_front_ends_equal_device_call(ek, dtype):
    """HostSuite.suite_trp (host_suite kind 2, many chunks) and host.fused.suite_trp return the device call's bits."""
    from ek_thermo import fused, host, hostpipe

    n = 1_000_003
    src = random_inputs(n, seed=23)
    hs = hostpipe.HostSuite(DEV, workspace_bytes=16 << 20, n_slots=3)
    h = {}
    for k in ("t", "r", "p"):
        h[k] = hostpipe.pinned_empty(n, dtype)
        h[k][:] = src[k]
    d = [torch.from_numpy(h[k]).to(DEV) for k in ("t", "r", "p")]
    for outputs, em in ((fused.DEFAULT_TRP, "ifs"), (fused.SINGLE_PASS_TRP, "ifs"), (("td", "e", "ept"), "bolton39")):
        want = fused.suite_trp(*d, outputs=outputs, ept_method=em)
        got = hs.suite_trp(h["t"], h["r"], h["p"], outputs=outputs, ept_method=em)
        got2 = host.fused.suite_trp(h["t"], h["r"], h["p"], outputs=outputs, ept_method=em)
        assert tuple(got) == tuple(got2) == outputs
        for k in outputs:
            assert got[k].dtype == dtype and got2[k].dtype == dtype
            assert _same(torch.from_numpy(got[k]), want[k].cpu()), ("HostSuite", k)
            assert _same(torch.from_numpy(np.asarray(got2[k])), want[k].cpu()), ("host.fused", k)
    out = {"td": np.empty(n, dtype=dtype)}
    got = hs.suite_trp(h["t"], h["r"], h["p"], outputs=("td",), out=out)
    assert got["td"] is out["td"]


# ---- coverage -------------------------------------------------------------------------------------------------------------------
def test_preallocated_empty_and_unaligned(ek):
    from ek_thermo import fused

    a, (t, r, p) = _dev(_inputs("random"), np.float64)
    out = {"td": torch.empty_like(t), "ept": torch.empty_like(t)}
    got = fused.suite_trp(t, r, p, outputs=("td", "q", "ept"), out=out)
    assert got["td"].data_ptr() == out["td"].data_ptr() and got["ept"].data_ptr() == out["ept"].data_ptr()
    check_suite({k: v.cpu().numpy() for k, v in got.items()}, a)
    before = ek.launch_count()
    e = fused.suite_trp(t[:0], r[:0], p[:0])
    assert ek.launch_count() == before and all(v.shape == (0,) for v in e.values()) and tuple(e) == fused.DEFAULT_TRP
    assert fused.suite_trp_batch([t[:0]], [r[:0]], [p[:0]])[0]["td"].shape == (0,)
    # an unaligned view (8 bytes past a 16-byte boundary): the scalar load/store path of the same kernel
    v = [x[1:] for x in (t, r, p)]
    got = fused.suite_trp(*v, outputs=tuple(fused.SUITE_TRP_OUTPUTS))
    check_suite({k: x.cpu().numpy() for k, x in got.items()}, [x[1:] for x in a])
    with pytest.raises(ValueError):
        fused.suite_trp(t, r, p, outputs=("td",), out={"td": torch.empty(3, dtype=torch.float64, device=DEV)})


def test_exact_library_passes_the_same_checks():
    """libek_thermo_exact.so, the libdevice-math twin of the product library, through the parity, bit-identity, batch and
    position tests in a child process (one library per process)."""
    import ek_thermo

    if os.path.basename(ek_thermo._backend.LIB_PATH) == "libek_thermo_exact.so":
        pytest.skip("already running against the exact build")
    assert os.path.exists(os.path.join(os.path.dirname(ek_thermo._backend.LIB_PATH), "libek_thermo_exact.so"))
    env = dict(os.environ, EK_THERMO_LIB="libek_thermo_exact.so")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-x", "-p", "no:cacheprovider", "-k",
                        "not exact_library and (ifs or random or bits or batch or position or scalar_pressure or host_front or preallocated)"],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
