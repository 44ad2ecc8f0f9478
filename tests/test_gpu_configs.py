"""GPU tests at the BASELINE.json configurations: oracle comparisons at sizes the oracle finishes in seconds, and
size-independent properties (conservation, partition / order invariance, exact accumulation, null field) at the
full C2 size (1e7 rays, 512^3)."""
import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import synthpy_oracle as O

pytestmark = pytest.mark.gpu
C_LIGHT = 299792458.0
LWL = 1064e-9
LENGTHS = (10e-3, 10e-3, 20e-3)
EXT = 10e-3


@pytest.fixture(scope="module")
def mods():
    assert torch.cuda.is_available()
    from synthpy_b200 import beam, diagnostics, domain, engine, field_generator, legacy, propagator
    return dict(B=beam, D=diagnostics, Dm=domain, E=engine, FG=field_generator, L=legacy, P=propagator)


def _oracle(ne, dims, phaseshift=False):
    x, y, z = (np.linspace(-L / 2, L / 2, n) for L, n in zip(LENGTHS, dims))
    o = O.Domain(x, y, z, EXT, phaseshift=phaseshift)
    o.external_ne(ne)
    o.calc_dndr(LWL)
    return o


def test_C1_gaussian_column_shadowgraphy(mods):
    """configs[0]: 128^3 analytic Gaussian column (formula of minimal_solver.test_lens), shadowgraphy, bin_scale 10;
    1e4 of the 1e5 rays against the oracle, the full 1e5 for count conservation."""
    P, D, Dm, L = mods["P"], mods["D"], mods["Dm"], mods["L"]
    n = 128
    dom = Dm.ScalarDomain(LENGTHS, n)
    XX, YY, _ = np.meshgrid(*dom._axes64, indexing="ij")
    ne = 1e24 * np.exp(-(XX ** 2 + YY ** 2) / (1e-3) ** 2)
    dom.external_ne(ne)
    np.random.seed(0)
    s0 = L.init_beam(100000, 5e-3, 5e-5, EXT, "circular", "z")
    n_steps = 2 * (n - 1)
    sub = s0[:, :10000]
    rf, _, _ = P.solve(sub, dom, EXT, lwl=LWL, method="rk4", n_steps=n_steps, early_exit=False)
    o = _oracle(ne, (n, n, n))
    rf_o, _ = O.ray_to_jones(o.solve_rk4(sub, n_steps)[0], EXT)
    assert rel_err(rf, rf_o, floor=1e-7) < 1e-9
    sh = D.Shadowgraphy(LWL, rf)
    sh.single_lens_solve()
    sh.histogram(bin_scale=10)
    H_o = O.histogram(O.run_chain(rf_o, O.chain("shadow_single")), bin_scale=10)
    assert sh.H.sum() == H_o.sum() and np.abs(sh.H - H_o).sum() <= 1e-3 * H_o.sum()
    # all 1e5 rays, fused, default step (half a cell) with early exit == explicit n_steps without (same line)
    spec = D.spec("shadow_single", bin_scale=10)
    stats, _ = P.solve_and_image(dom, s0, EXT, [spec], lwl=LWL)
    assert stats["rays_binned"] + stats["rays_rejected"] <= 100000 and stats["rays_binned"] == int(spec.image.counts.sum())
    assert stats["rays_binned"] > 0.5 * 100000


def test_C3_interferometry_phase(mods):
    """configs[2] at reduced size: phase accumulation (float64 aux grid) + two-lens interferogram vs the oracle."""
    P, D, Dm, FG, L = mods["P"], mods["D"], mods["Dm"], mods["FG"], mods["L"]
    n = 48
    ne = FG.turbulent_ne(n // 2, noise="torch", seed=3).cpu().numpy()
    dom = Dm.ScalarDomain(LENGTHS, n, phaseshift=True)
    dom.external_ne(ne)
    np.random.seed(1)
    s0 = L.init_beam(6000, 4e-3, 5e-5, EXT, "circular", "z")
    n_steps = 2 * (n - 1)
    rf, Jf, _ = P.solve(s0, dom, EXT, lwl=LWL, return_E=True, method="rk4", n_steps=n_steps, early_exit=False, phase_f64=True)
    o = _oracle(ne, (n, n, n), phaseshift=True)
    sf_o, _ = o.solve_rk4(s0, n_steps)
    rf_o, J_o = O.ray_to_jones(sf_o, EXT)
    assert rel_err(rf, rf_o, floor=1e-7) < 1e-9
    assert np.max(np.abs(Jf - J_o)) < 3e-7                      # |phase| ~ 1e3 rad: 1e-10 relative phase parity
    it = D.Interferometry(LWL, rf, Jf)
    it.two_lens_solve(ref_beam=None)
    it.interferogram(bin_scale=40)
    r_o, E_o = O.run_chain(rf_o, O.chain("interf_two"), E=J_o, wl=LWL)
    H_o = O.interferogram(r_o, E_o, bin_scale=40)
    assert it.H.shape == H_o.shape and np.abs(it.H - H_o).sum() <= 1e-3 * H_o.sum()
    # float32 aux lane (the fast default): phase within 1e-6 relative, image within the L1 budget
    rf2, Jf2, _ = P.solve(s0, dom, EXT, lwl=LWL, return_E=True, method="rk4", n_steps=n_steps, early_exit=False)
    ph_o = sf_o[7]
    dphi = np.angle(Jf2[1] * np.exp(-1j * ph_o))
    assert np.max(np.abs(dphi)) < 2e-6 * np.abs(ph_o).max() + 1e-9
    # reference-beam variant of the current API (pinned by golden g9, test_gpu_parity::test_current_generation_diagnostics)
    it2 = D.Interferometry(LWL, rf, Jf)
    it2.two_lens_solve()
    it2.interferogram(bin_scale=40)
    r_o2, E_o2 = O.run_chain(rf_o, O.chain("interf_two"), E=O.interfere_ref_beam(rf_o, J_o, 10, 20), wl=LWL)
    H_o2 = O.interferogram(r_o2, E_o2, bin_scale=40)
    assert np.abs(it2.H - H_o2).sum() <= 1e-3 * H_o2.sum()


def test_C4_refractometry_knife_edge_and_tolerance_sweep(mods):
    """configs[3] at reduced size: refractometer + knife-edge schlieren chains vs the oracle, and the adaptive
    tolerance sweep: work grows, images converge towards the tightest tolerance."""
    P, D, Dm, FG, L = mods["P"], mods["D"], mods["Dm"], mods["FG"], mods["L"]
    n = 48
    ne = FG.turbulent_ne(n // 2, noise="torch", seed=4).cpu().numpy()
    dom = Dm.ScalarDomain(LENGTHS, n)
    dom.external_ne(ne)
    np.random.seed(2)
    s0 = L.init_beam(20000, 4e-3, 5e-5, EXT, "circular", "z")
    n_steps = 2 * (n - 1)
    rf, _, _ = P.solve(s0, dom, EXT, lwl=LWL, method="rk4", n_steps=n_steps, early_exit=False)
    o = _oracle(ne, (n, n, n))
    rf_o, _ = O.ray_to_jones(o.solve_rk4(s0, n_steps)[0], EXT)
    assert rel_err(rf, rf_o, floor=1e-7) < 1e-9
    rm = D.Refractometry(LWL, rf)
    rm.incoherent_solve()
    rm.histogram(bin_scale=20)
    H_o = O.histogram(O.run_chain(rf_o, O.chain("refracto_incoherent")), bin_scale=20)
    assert rm.H.sum() == H_o.sum() and np.abs(rm.H - H_o).sum() <= 1e-3 * H_o.sum()
    for off in (0.0, 0.1, 0.5):
        sc = D.Schlieren(LWL, rf)
        sc.knife_solve(offset=off, axis="y", direction=1)
        sc.histogram(bin_scale=20)
        H_o = O.histogram(O.run_chain(rf_o, O.chain("schlieren_knife", offset=off, axis=2, direction=1)), bin_scale=20)
        assert sc.H.sum() == H_o.sum() and np.abs(sc.H - H_o).sum() <= 1e-3 * H_o.sum()
    # adaptive sweep (rtol, atol) as in SURVEY 8d-C4
    imgs, work = [], []
    for rtol, atol in [(1e-3, 1e-6), (1e-5, 1e-8), (1e-7, 1e-9), (1e-9, 1e-12)]:
        spec = D.spec("refracto_incoherent", bin_scale=20)
        stats, _ = P.solve_and_image(dom, s0, EXT, [spec], lwl=LWL, method="rk45", rtol=rtol, atol=atol, max_steps=200000,
                                     early_exit=False)
        assert stats["rays_capped"] == 0
        imgs.append(spec.image.result().cpu().numpy())
        work.append(stats["ray_steps"] / s0.shape[1])
    assert work[0] < work[1] < work[2] < work[3]
    l1 = [np.abs(h - imgs[-1]).sum() / imgs[-1].sum() for h in imgs[:-1]]
    assert l1[2] <= l1[0] + 1e-12 and l1[2] < 0.05


def test_field_generator_on_device(mods, golden):
    """SURVEY 8f-1 on the GPU: (a) the cuFFT path reproduces the field the reference's gaussian3D.domain_fft produced for
    np.random.seed(1) (tests/golden/g3_turb.npz, made by the real module); (b) at the benchmarked 512^3 size the radially
    averaged power spectrum of the generated field follows the requested k^-11/3 law inside the band and is empty outside;
    (c) the CPU and GPU FFTs of the same (torch, seeded) noise give the same grid."""
    FG = mods["FG"]
    g = golden("g3_turb")
    np.random.seed(1)
    ne = FG.turbulent_ne(16, noise="numpy", device="cuda")
    assert ne.is_cuda and tuple(ne.shape) == g["ne"].shape
    assert np.max(np.abs(ne.cpu().numpy() - g["ne"])) < 1e-6 * np.abs(g["ne"]).max()
    a = FG.turbulent_ne(32, noise="torch", seed=5, device="cuda").cpu()
    b = FG.turbulent_ne(32, noise="torch", seed=5, device="cpu")
    assert float((a - b).abs().max()) < 1e-6 * float(b.abs().max())      # float32 |k| (gaussian3D.py:240): sqrt differs by an ulp between cuFFT box and host
    # spectrum of the C2 field: f = (ne - 1e25) / 9e24, extent 5 (mm), res 256 -> dx = 5 / 256
    n, res, extent = 512, 256, 5.0
    f = (FG.turbulent_ne(res, noise="torch", seed=1, device="cuda") - 1e25) / 9e24
    P = torch.fft.fftn(f).abs() ** 2
    del f
    k1 = 2 * np.pi * torch.fft.fftfreq(n, d=extent / res, device="cuda", dtype=torch.float64)
    k = torch.sqrt(k1[:, None, None] ** 2 + k1[None, :, None] ** 2 + k1[None, None, :] ** 2)
    k_min, k_max = 2 * np.pi / 1.0, 2 * np.pi / 0.01
    inside = (k >= k_min) & (k <= k_max)
    assert float(P[~inside].sum()) < 1e-20 * float(P[inside].sum())                 # band-limited (gaussian3D.py:252-256)
    edges = torch.logspace(np.log10(k_min * 1.5), np.log10(float(k.max()) * 0.5), 13, device="cuda", dtype=torch.float64)
    kc, pk = [], []
    for lo, hi in zip(edges[:-1], edges[1:]):
        m = (k >= lo) & (k < hi)
        kc.append(float(k[m].mean())); pk.append(float(P[m].mean()))
    slope = np.polyfit(np.log(kc), np.log(pk), 1)[0]
    assert abs(slope + 11.0 / 3.0) < 0.1, slope                                     # |noise|^2 averages to a constant per shell


@pytest.fixture(scope="module")
def c2(mods):
    """The C2 workload at full size: 512^3 turbulent field, 1e7 device-generated rays."""
    Dm, FG, B = mods["Dm"], mods["FG"], mods["B"]
    ne = FG.turbulent_ne(256, noise="torch", seed=1)
    dom = Dm.ScalarDomain(LENGTHS, 512)
    dom.external_ne(ne)
    dom.device_field(LWL)
    beam = B.Beam(int(1e7), 5e-3, 5e-5, EXT, device=True, seed=2)
    return dom, beam


def _images(mods, dom, beam, n, off, **kw):
    D, P = mods["D"], mods["P"]
    specs = [D.spec("shadow_two", bin_scale=1), D.spec("schlieren_DF", bin_scale=1, R_stop=1)]
    stats, _ = P.solve_and_image(dom, beam, EXT, specs, lwl=LWL, n_rays=n, ray_offset=off, **kw)
    return [s.image.counts.clone() for s in specs], stats


def test_C2_full_size_properties(mods, c2):
    dom, beam = c2
    N = int(1e7)
    whole, st = _images(mods, dom, beam, N, 0)
    # conservation: every ray is either binned, rejected by an element, or misses the detector
    for img in whole:
        assert 0 < int(img.sum()) <= N
    assert st["rays_binned"] == sum(int(i.sum()) for i in whole)
    assert st["ray_steps"] > 900 * N                                 # ~2 steps per cell over 511 cells, early exit
    # partition invariance (what multi-GPU sharding relies on): 3 uneven shards sum to the whole, bit for bit
    acc = [torch.zeros_like(i) for i in whole]
    steps = 0
    for off, cnt in ((0, 3333333), (3333333, 4000000), (7333333, 2666667)):
        part, s = _images(mods, dom, beam, cnt, off)
        steps += s["ray_steps"]
        for a, p_ in zip(acc, part):
            a += p_
    assert all(torch.equal(a, w) for a, w in zip(acc, whole)) and steps == st["ray_steps"]
    # order invariance: bundling rays (sort) must not change any per-ray result
    unsorted, s2 = _images(mods, dom, beam, N, 0, sort=False)
    assert all(torch.equal(a, w) for a, w in zip(unsorted, whole)) and s2["ray_steps"] == st["ray_steps"]


def test_C2_null_field_is_identity_at_full_size(mods):
    """NULL test (full_solver.py:12-54) at 512^3 / 1e6 rays: no density => exit angles are exactly the entry angles."""
    Dm, B, P = mods["Dm"], mods["B"], mods["P"]
    dom = Dm.ScalarDomain(LENGTHS, 512)
    dom.external_ne(torch.zeros((512, 512, 512), dtype=torch.float32, device="cuda"))
    beam = B.Beam(int(1e6), 5e-3, 5e-5, EXT, device=True, seed=5)
    s0 = beam.materialise()
    rf, _, _ = P.solve(s0, dom, EXT, lwl=LWL)
    assert torch.equal(rf[1], torch.atan(s0[3] / s0[5])) and torch.equal(rf[3], torch.atan(s0[4] / s0[5]))
    x_exit = s0[0] - s0[3] * ((s0[2] - EXT) / s0[5])
    assert torch.max(torch.abs(rf[0] - x_exit)) < 1e-14


def test_C5_grid_1024_properties(mods):
    """BASELINE configs[4] at its full GRID size on one GPU (1024^3: 17 GB packed field, the largest grid the configs
    name), with a 2e6-ray shard: conservation, two-shard partition invariance bit for bit, steps ~ 2 per cell."""
    Dm, FG, B, D, P = mods["Dm"], mods["FG"], mods["B"], mods["D"], mods["P"]
    free, _ = torch.cuda.mem_get_info()
    if free < 90e9:
        pytest.skip("needs ~90 GB of free device memory while the field is generated (FFT) and packed")
    ne = FG.turbulent_ne(512, noise="torch", seed=3)
    dom = Dm.ScalarDomain(LENGTHS, 1024)
    dom.external_ne(ne)
    fld = dom.device_field(LWL)
    del ne
    dom.release_ne()
    torch.cuda.empty_cache()
    assert fld.nbytes >= 16 * 1024 ** 3
    N = 2000000
    beam = B.Beam(N, 5e-3, 5e-5, EXT, device=True, seed=2)

    def run(n, off):
        spec = D.spec("shadow_two", bin_scale=1)
        st, _ = P.solve_and_image(dom, beam, EXT, [spec], lwl=LWL, n_rays=n, ray_offset=off)
        return spec.image.counts.clone(), st
    whole, st = run(N, 0)
    assert st["rays_binned"] == int(whole.sum()) and 0 < int(whole.sum()) <= N
    assert 1900 * N < st["ray_steps"] < 2100 * N                     # 2 steps per cell over 1023 cells, early exit
    a, sa = run(1200000, 0)
    b, sb = run(800000, 1200000)
    assert torch.equal(a + b, whole) and sa["ray_steps"] + sb["ray_steps"] == st["ray_steps"]


def test_quickstart_example_runs(mods):
    """examples/quickstart.py = the reference notebook's walkthrough; must run unchanged on the GPU."""
    import importlib.util
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "quickstart.py")
    spec = importlib.util.spec_from_file_location("quickstart", path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    rf = m.main(20000)
    assert rf.shape == (4, 20000) and np.isfinite(rf).all()


def test_bench_contract_on_a_small_workload():
    """bench.py prints ONE JSON line with every key the driver reads (small grid / few rays so it runs in seconds)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--grid", "64", "--rays", "2e5", "--steps", "2",
                          "--warmup", "3", "--cpu-rays-per-worker", "50", "--parity-rays", "500"], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "cpu_baseline", "same_integrator", "e2e", "parity", "gpu_launches", "clocks",
              "rays_per_s"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"]
    r = d["roofline"]
    assert r["bound"] == "fp64_pipe" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert 0 < r["frac"] <= 1.0 and 20 < r["peak"] < 60                      # B200 FP64: ~37 TFLOP/s FMA
    assert r["hbm_algorithmic"]["bytes_per_ray_step"] == 512 and r["hbm_algorithmic"]["frac"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] > 0
    assert d["same_integrator"]["value"] > 0 and d["cpu_baseline"]["rays_per_s"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 72 * 200000 and e["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] >= 2 * 4 and d["value"] > 0
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    p = d["parity"]
    assert p["n"] == 500 and p["max_rel"] < 1e-9 and p["steps_equal"] and p["hist_equal"]


def test_bench_dump_outputs_and_step_count(tmp_path):
    """--steps sets the number of timed passes (launches scale with it), and --dump-outputs writes the same images and
    stats for the same arguments whatever the step count: every pass traces the same seeded rays through the same field."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lines = {}
    for steps in (2, 3):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--grid", "64", "--rays", "2e5", "--steps", str(steps),
                              "--warmup", "3", "--no-cpu-baseline", "--no-parity", "--no-e2e", "--dump-outputs",
                              str(tmp_path / f"s{steps}")], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        lines[steps] = json.loads([l for l in out.stdout.strip().splitlines() if l.startswith("{")][0])
        assert lines[steps]["steps"] == steps
    assert lines[2]["gpu_launches"] * 3 == lines[3]["gpu_launches"] * 2 and lines[2]["gpu_launches"] > 0
    files = sorted(os.listdir(tmp_path / "s2"))
    assert files == ["schlieren_DF.npy", "schlieren_DF_index.npy", "shadow_two.npy", "shadow_two_index.npy", "stats.npy"]
    assert sum(os.path.getsize(tmp_path / "s2" / f) for f in files) <= 64_000_000
    for f in files:
        a, b = np.load(tmp_path / "s2" / f), np.load(tmp_path / "s3" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b), f
    stats = dict(zip(("ray_steps", "ray_steps_acc", "rays_capped", "rays_binned", "rays_rejected", "rhs_evals"),
                     np.load(tmp_path / "s2" / "stats.npy")))
    assert stats["ray_steps"] == lines[2]["ray_steps_per_pass_per_gpu"] and stats["rays_binned"] == lines[2]["rays_binned_last_pass"]


def test_bench_C1_line():
    """--workload C1 (BASELINE configs[0], the reference's own CPU-runnable case) prints a full line with parity over ALL
    its rays' first 2000."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "C1", "--cpu-rays-per-worker", "200"],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads([l for l in out.stdout.strip().splitlines() if l.startswith("{")][0])
    assert d["config"]["grid"] == 128 and d["config"]["rays_per_gpu"] == 100000 and d["value"] > 0
    assert d["parity"]["max_rel"] < 1e-9 and d["parity"]["steps_equal"] and d["parity"]["hist_equal"]
    assert d["e2e"]["h2d_bytes_per_step"] == 72 * 100000


def test_pvti_field_equals_direct_field_and_driver_example_runs(mods, tmp_path, monkeypatch):
    """SURVEY 8f-4: a density grid written to .pvti and streamed back into HBM gives bit-identical gradients and
    images to the same grid handed over directly; examples/pvti_trace.py (the reference's
    pvti_trace_multiprocess.py driver) runs on it and conserves rays."""
    import importlib.util
    import os
    import pickle
    import sys
    from synthpy_b200 import handle_filetypes as io
    B, D, Dm, P = mods["B"], mods["D"], mods["Dm"], mods["P"]
    n = 64
    ax = np.linspace(-1, 1, n)
    X, Y, Z = np.meshgrid(ax, ax, ax, indexing="ij")
    ne = (3e24 * np.exp(-(X ** 2 + Z ** 2) / 0.3 ** 2) * (1 + 0.2 * np.cos(9 * Y))).astype(np.float32)
    io.export_pvti(ne, fname=str(tmp_path / "dump"), extent_x=5e-3, extent_y=5e-3, extent_z=5e-3)
    t, dim, sp = io.pvti_readin(str(tmp_path / "dump.pvti"), device="cuda")
    assert t.is_cuda and t.is_contiguous() and dim == (n, n, n) and torch.equal(t.cpu(), torch.from_numpy(ne))
    dom_f, ext = io.domain_from_pvti(str(tmp_path / "dump.pvti"), probing_direction="y")
    dom_d = Dm.ScalarDomain([2 * e for e in ext], n, probing_direction="y")
    dom_d.external_ne(ne)
    ga, gb = dom_f.device_field(LWL).export_gradients(), dom_d.device_field(LWL).export_gradients()
    assert all(torch.equal(a, b) for a, b in zip(ga[:3], gb[:3]))
    imgs = []
    for dom in (dom_f, dom_d):
        s = D.spec("shadow_single", bin_scale=8)
        P.solve_and_image(dom, B.Beam(200000, ext[0], 5e-5, ext[1], probing_direction="y", device=True, seed=4), ext[1], [s])
        imgs.append(s.image.result())
    assert torch.equal(imgs[0], imgs[1]) and imgs[0].sum() > 0
    # the driver, end to end, in the reference's units (ne * 1e12)
    io.export_pvti(ne * 1e-12, fname=str(tmp_path / "drv"), extent_x=5e-3, extent_y=5e-3, extent_z=5e-3)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("pvti_trace", os.path.join(root, "examples", "pvti_trace.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    monkeypatch.setattr(sys, "argv", ["pvti_trace.py", "3e5", str(tmp_path / "drv.pvti"), str(tmp_path / "out_"), "--chunk", "1e5",
                                      "--bin-scale", "8"])
    sh_H, r_H = m.main()
    assert sh_H.shape == (2574 // 8, 3448 // 8) and 0 < sh_H.sum() <= 3e5 and 0 < r_H.sum() <= 3e5
    assert np.array_equal(pickle.load(open(tmp_path / "out_shadow.pkl", "rb")), sh_H)
    # three chunks of 1e5 == one launch of 3e5 (device rays depend on (seed, index) only)
    monkeypatch.setattr(sys, "argv", ["pvti_trace.py", "3e5", str(tmp_path / "drv.pvti"), str(tmp_path / "one_"), "--bin-scale", "8"])
    sh1, r1 = m.main()
    assert np.array_equal(sh1, sh_H) and np.array_equal(r1, r_H)


def test_interference_driver_example(mods, tmp_path, monkeypatch):
    """examples/interference_mpi.py (the reference's interference_MPI.py driver): the coherent sum does not depend on the
    chunking; --sum-magnitudes reproduces the driver's `sh.H += sh_split.H` accumulation."""
    import importlib.util
    import os
    import sys
    from synthpy_b200 import handle_filetypes as io
    n = 48
    ax = np.linspace(-1, 1, n)
    X, Y, Z = np.meshgrid(ax, ax, ax, indexing="ij")
    ne = (2e18 * np.exp(-(X ** 2 + Z ** 2) / 0.4 ** 2)).astype(np.float32)        # x 1e6 below
    io.export_pvti(ne, fname=str(tmp_path / "f"), extent_x=8e-3, extent_y=8e-3, extent_z=8e-3)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("interference_mpi", os.path.join(root, "examples", "interference_mpi.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)

    def run(*extra):
        monkeypatch.setattr(sys, "argv", ["interference_mpi.py", "6e4", "1e6", str(tmp_path / "f.pvti"), str(tmp_path / "o_"),
                                          "--bin-scale", "16", "--fringes", "10", "--deg", "20", *extra])
        return m.main()
    one = run("--chunk", "6e4")
    three = run("--chunk", "2e4")
    assert one.shape == (2574 // 16 - 1, 3448 // 16 - 1) and one.max() > 0
    assert np.abs(one - three).max() <= 1e-9 * one.max()                          # coherent sum: chunking is irrelevant
    mags = run("--chunk", "2e4", "--sum-magnitudes")
    assert np.abs(mags - one).max() > 1e-3 * one.max()                            # the driver's accumulation is not
    assert (mags >= one - 1e-9 * one.max()).all()                                 # |a| + |b| + |c| >= |a + b + c| per plane pair
