"""CPU tests of host-side pieces that need no GPU: field generator restatement, Beam host RNG stream, API shapes,
bench.py's reference arm contract."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_field_generator_matches_reference_realisation(golden):
    """synthpy_b200.field_generator.domain_fft (torch FFT) reproduces the field the reference's
    gaussian3D.domain_fft produced for np.random.seed(1) (stored in tests/golden/g3_turb.npz)."""
    from synthpy_b200 import field_generator as fg
    g = golden("g3_turb")
    np.random.seed(1)
    ne = fg.turbulent_ne(16, noise="numpy", device="cpu").numpy()
    assert ne.shape == g["ne"].shape
    assert np.max(np.abs(ne - g["ne"])) < 1e-6 * np.abs(g["ne"]).max()
    a = fg.turbulent_ne(8, noise="torch", seed=5, device="cpu")
    b = fg.turbulent_ne(8, noise="torch", seed=5, device="cpu")
    assert bool((a == b).all()) and float(a.min()) > 0


def test_beam_host_stream_and_shapes():
    from synthpy_b200 import beam as B, legacy
    b = B.Beam(1000, 5e-3, 5e-5, 10e-3, seeded=True)
    assert b.s0.shape == (9, 1000) and np.all(b.s0[2] == -10e-3) and np.all(b.s0[6] == 1.0)
    # seeded draws re-seed before every draw (utils.py:8-24): t, u and chi come from the same stream start
    np.random.seed(0)
    t = 2 * np.pi * np.random.rand(1000)
    np.random.seed(0)
    u = np.random.power(2, 1000)
    assert np.allclose(b.s0[0], 5e-3 * u * np.cos(t)) and np.allclose(b.s0[1], 5e-3 * u * np.sin(t))
    for pd, row in (("x", 0), ("y", 1), ("z", 2)):
        bb = B.Beam(64, 1e-3, 1e-4, 2e-3, probing_direction=pd)
        assert np.all(bb.s0[row] == -2e-3) and np.allclose(np.linalg.norm(bb.s0[3:6], axis=0), 299792458.0)
    np.random.seed(3)
    s0 = legacy.init_beam(50, (1e-3, 2e-3), 1e-4, 5e-3, "rectangular", "z")
    assert np.abs(s0[0]).max() <= 1e-3 and np.abs(s0[1]).max() <= 2e-3
    d = B.Beam(10, 5e-3, 5e-5, 10e-3, device=True, seed=3)
    assert d.s0 is None and d.spec.start == -10e-3


def test_domain_api_shapes():
    from synthpy_b200 import domain as D
    dom = D.ScalarDomain([10e-3, 10e-3, 20e-3], [16, 12, 20], ne_type="test_exponential_cos")
    assert dom.ne.shape == (16, 12, 20) and dom.x.dtype == np.float32 and dom.region_count == 1
    assert np.array_equal(dom.z, np.float32(np.linspace(-10e-3, 10e-3, 20)))
    assert abs(dom.cell_size() - 20e-3 / 19) < 1e-18
    dom2 = D.ScalarDomain(1e-2, 8)
    dom2.test_slab(s=2)
    assert dom2.ne.shape == (8, 8, 8) and np.all(np.diff(dom2.ne[:, 0, 0]) > 0)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` prints one JSON line with the agreed keys (tiny grid so it runs in seconds)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "32", "--steps", "1",
                          "--warmup", "1", "--cpu-rays-per-worker", "40"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "rays*steps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["rays_per_s"] > 0 and line["cpu_baseline"]["rays_per_s"] == line["rays_per_s"]


def test_bench_reference_arm_maps_no_product_code():
    """VERDICT r1: the reference process must not import the product package (whose import dlopens the CUDA library).
    Run the arm under an import hook that refuses `synthpy_b200`, for the turbulent (C2) and the analytic (C1) field."""
    hook = ("import sys, importlib.abc\n"
            "class Deny(importlib.abc.MetaPathFinder):\n"
            "    def find_spec(self, name, path=None, target=None):\n"
            "        if name.split('.')[0] == 'synthpy_b200': raise ImportError('reference arm imported the product package')\n"
            "sys.meta_path.insert(0, Deny())\n"
            "import runpy; sys.argv = ['bench.py'] + sys.argv[1:]; runpy.run_path(%r, run_name='__main__')\n" % os.path.join(ROOT, "bench.py"))
    for extra in (["--grid", "32"], ["--workload", "C1", "--grid", "32", "--rays", "400"]):
        out = subprocess.run([sys.executable, "-c", hook, "--impl", "reference", "--steps", "1", "--warmup", "0",
                              "--cpu-rays-per-worker", "24"] + extra, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["impl"] == "reference" and line["value"] > 0
        maps_check = "libsynthpy_b200" not in out.stdout + out.stderr
        assert maps_check


def test_gaussian_column_profiles():
    """test_lens / test_liner (minimal_solver.py:192-212) in both API generations, against the closed form."""
    from synthpy_b200 import domain as Dm, legacy
    d = Dm.ScalarDomain([2e-3, 2e-3, 4e-3], [9, 11, 13])
    d.test_lens(ne_0=3e24, LR=5e-4)
    X, Y, Z = np.meshgrid(np.linspace(-1e-3, 1e-3, 9), np.linspace(-1e-3, 1e-3, 11), np.linspace(-2e-3, 2e-3, 13), indexing="ij")
    assert d.ne.shape == (9, 11, 13) and np.allclose(d.ne, 3e24 * np.exp(-(X ** 2 + Y ** 2) / 5e-4 ** 2), rtol=1e-12)
    d.test_liner(ne_0=3e24, LR=5e-4)
    assert np.allclose(d.ne, 3e24 * np.exp(-(X ** 2 + Z ** 2) / 5e-4 ** 2), rtol=1e-12)
    x, y, z = np.linspace(-1e-3, 1e-3, 9), np.linspace(-1e-3, 1e-3, 11), np.linspace(-2e-3, 2e-3, 13)
    ld = legacy.ScalarDomain(x, y, z, 2e-3)
    ld.test_lens(n_e0=3e24, LR=5e-4)
    assert np.allclose(ld.ne, 3e24 * np.exp(-(X ** 2 + Y ** 2) / 5e-4 ** 2), rtol=1e-12)
    ld.test_liner(n_e0=3e24, LR=5e-4)
    assert np.allclose(ld.ne, 3e24 * np.exp(-(X ** 2 + Z ** 2) / 5e-4 ** 2), rtol=1e-12)


def test_reference_held_fixture_product_profiles():
    """The same reference fixture (integratedPy.npy) against the PRODUCT's profile generators, both API generations."""
    from conftest import GOLDEN
    from synthpy_b200 import domain as Dm, legacy
    ref = np.load(os.path.join(GOLDEN, "integratedPy.npy"))
    dims, spcs = np.array([100, 1000, 100]), np.array([1e-4, 1e-5, 1e-4])
    ax = [np.linspace(-(n - 1) * s / 2, (n - 1) * s / 2, n) for n, s in zip(dims, spcs)]
    ld = legacy.ScalarDomain(ax[0], ax[1], ax[2], (dims[2] - 1) * spcs[2] / 2)
    ld.test_linear_cos(s1=-1, s2=1, n_e0=1e26, Ly=5e-3)
    assert np.array_equal(np.asarray(ld.ne).sum(axis=2), ref)
    d = Dm.ScalarDomain((dims - 1) * spcs, dims)
    d.test_linear_cos(s1=-1, s2=1, ne_0=1e26, Ly=5e-3)
    # the current-generation signature normalises x by x_length = 2 * extent where the legacy code uses the half-width,
    # so the two generations differ by design (domain.py:392-451 vs full_solver.py:148-157); the legacy one is the fixture's
    assert d.ne.shape == (100, 1000, 100)


def test_beam_types_rect_trackers_and_even():
    from synthpy_b200 import beam as B
    np.random.seed(3)
    a = B.Beam(100, (1e-3, 2e-3), 1e-4, 5e-3, beam_type="rectangular").s0
    np.random.seed(3)
    b = B.Beam(100, (1e-3, 2e-3), 1e-4, 5e-3, beam_type="rect_trackers").s0           # beam.py:228-286 == rectangular
    assert np.array_equal(a, b)
    e = B.Beam(100, 1e-3, 1e-4, 5e-3, beam_type="even")                                # beam.py:210-227
    n_c = int((-1 + np.sqrt(1 + 8 * (100 // 6))) / 2)
    assert e.Np == 3 * (n_c + 1) * n_c + 1 == e.s0.shape[1]
    r = np.hypot(e.s0[0], e.s0[1])
    assert r[0] == 0 and abs(r.max() - 1e-3) < 1e-15 and np.all(e.s0[2] == -5e-3) and np.all(e.s0[6] == 1.0)
    rings = np.round(r / 1e-3 * n_c).astype(int)
    assert all((rings == i).sum() == 6 * i for i in range(1, n_c + 1))



def test_beam_matches_current_generation_source(golden):
    """g10: src/simulator/beam.py + utils.py executed from their own source (oracle/gen_golden.py::import_simulator, NumPy
    standing in for jax.numpy; the draws are NumPy's global RNG upstream too).  Every beam type upstream can construct x
    probing direction x seeded / unseeded: bit for bit.  ('linear' and 'even' raise upstream -- beam.py:291, :222 -- and
    are this package's reading of the intent: test_beam_types_rect_trackers_and_even.)"""
    from synthpy_b200 import beam as B
    g = golden("g10_beam")
    sizes = {"circular": 4e-3, "square": 3e-3, "rectangular": (1e-3, 2.5e-3), "rect_trackers": (2e-3, 0.5e-3)}
    assert len(g) == 24
    for key, ref in g.items():
        bt, pd, seeded = key.rsplit("_", 2)
        np.random.seed(17)
        b = B.Beam(96, sizes[bt], 2e-4, 6e-3, probing_direction=pd, beam_type=bt, seeded=bool(int(seeded)))
        assert np.array_equal(b.s0, ref), key



def test_domain_matches_current_generation_source(golden):
    """g11: src/simulator/domain.py executed from its own source (oracle/gen_golden.py::import_simulator).  The float32
    axes are identical; the named profiles, which upstream evaluates in float32 on the float32-rounded mesh
    (domain.py:392-451) and this package in float64 (domain.py docstring here), agree to float32 rounding."""
    from synthpy_b200 import domain as Dm
    g = golden("g11_domain")
    for name in ("test_null", "test_slab", "test_linear_cos", "test_exponential_cos"):
        d = Dm.ScalarDomain(tuple(g["lengths"]), tuple(g["dims"]), ne_type=name)
        ref = g[name]
        assert ref.dtype == np.float32 and np.asarray(d.ne).shape == ref.shape
        assert np.max(np.abs(np.asarray(d.ne) - ref)) <= 1e-6 * np.abs(ref).max(), name
        assert all(getattr(d, k).dtype == np.float32 and np.array_equal(getattr(d, k), g[k]) for k in "xyz")
    assert np.abs(g["test_exponential_cos"]).max() > 1e26 and np.ptp(g["test_slab"]) > 1e23      # the fixture is not trivial
    d = Dm.ScalarDomain(5e-3, 7)                                             # scalar lengths / dims
    assert np.array_equal(d.x, g["cube_x"]) and tuple(d.dims) == g["cube_XX"].shape


def test_bench_ncu_evidence_is_tied_to_the_kernel_source(tmp_path, monkeypatch):
    """VERDICT r1: static ncu numbers in the bench line must not survive a kernel change.  attach_ncu_static accepts a
    capture only while its stored hash equals the hash of ray_core.h + synthpy_b200.cu, and reports its DRAM bytes as
    `traffic` only for a launch of the same number of rays."""
    import bench
    prof = tmp_path / "profiles"
    prof.mkdir()
    cap = {"source_sha16": bench.source_sha16(), "rays_per_launch": 10000000, "dram__bytes_read.sum": ["2.5", "Gbyte"],
           "dram__bytes_write.sum": ["120", "Mbyte"], "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active": ["53.1", "%"]}
    (prof / "r2_c2_k_propagate_ncu_full.json").write_text(json.dumps(cap))
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "source_sha16", lambda: cap["source_sha16"])
    a = bench.parse([])
    roof = {"traffic": None}
    bench.attach_ncu_static(roof, a, 10000000)
    assert abs(roof["traffic"] - 2.62e9) < 1e3 and roof["ncu_static"]["fp64_pipe_pct"] == 53.1
    roof = {"traffic": None}
    bench.attach_ncu_static(roof, a, 2000000)                        # another launch size: evidence kept, traffic not claimed
    assert roof["traffic"] is None and roof["ncu_static"]["rays_of_profiled_launch"] == 10000000
    monkeypatch.setattr(bench, "source_sha16", lambda: "0" * 16)      # the kernel source changed
    roof = {"traffic": None}
    bench.attach_ncu_static(roof, a, 10000000)
    assert roof["traffic"] is None and roof["ncu_static"] == {"stale": True, "source": os.path.join("profiles", "r2_c2_k_propagate_ncu_full.json")}


def test_bench_parity_helpers_and_lattice():
    """bench.parity_check's ingredients that can be checked without a GPU: the per-row scale of the relative error, NaN
    pattern handling, and -- the point of the parity block -- that the oracle is stepped on the SAME fixed-step lattice
    (h, n_steps) that propagator._params hands to the kernel for every workload."""
    import bench
    from synthpy_b200 import domain as Dm, propagator as P
    a = np.array([[1e-3, -2e-3, 1e-12], [0.02, 1e-9, -0.03]])
    b = a * (1 + 1e-10)
    s = bench._row_scale(a)
    assert np.allclose(s, np.sqrt((a ** 2).mean(axis=1)))
    assert abs(bench._rel(b, a, s) - 1e-10) < 1e-13                       # tiny entries are measured against the row scale
    assert bench._rel(b, a, 1e-30) > 9e-11
    c = a.copy(); c[0, 1] = np.nan
    assert bench._rel(c, a, s) == float("inf")                            # NaN patterns must coincide
    for w in ("C1", "C2", "C3", "C5"):
        args = bench.parse(["--workload", w])
        dom = Dm.ScalarDomain(bench.LENGTHS, 16)                          # cell size only depends on lengths / dims
        dom.dims = np.array([args.grid] * 3)
        prm = P._params(dom, bench.EXTENT, bench.LWL, "rk4", None, args.ds_frac * dom.cell_size(), None, None, "fp64", True, False,
                        False, True, "current", None)
        h, n = bench.rk4_lattice(args)
        assert prm.h == h and prm.n_steps == n, w


def test_bench_dump_outputs_budget_and_sample(tmp_path):
    """bench.dump_outputs: float64 files within the byte budget, small arrays whole, a larger one as a fixed seeded sample
    whose index file says where every value came from; the same arrays always give the same files."""
    import bench
    big = np.random.default_rng(1).integers(0, 50, size=(300, 500))
    stats = np.arange(6)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"img": big, "stats": stats}, budget=600_000)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["img.npy", "img_index.npy", "stats.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 600_000
    got = {f: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert got[f].dtype == np.float64 and np.array_equal(got[f], np.load(tmp_path / "b" / f))
    idx = got["img_index.npy"].astype(np.int64)
    assert len(idx) > 30_000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(got["img.npy"], big.ravel()[idx]) and np.array_equal(got["stats.npy"], stats)
    bench.dump_outputs(str(tmp_path / "c"), {"img": big, "stats": stats})
    assert np.array_equal(np.load(tmp_path / "c" / "img.npy"), big)         # fits the default budget: written whole
    assert sorted(os.listdir(tmp_path / "c")) == ["img.npy", "stats.npy"]


def test_bench_rejects_step_counts_below_one_and_dumps_of_the_reference_arm():
    import bench
    import pytest
    assert bench.parse(["--steps", "7"]).steps == 7
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        with pytest.raises(SystemExit):
            bench.parse(argv)


def test_numa_binding_is_best_effort():
    """distributed.bind_to_local_numa never raises: without a GPU (or without sysfs NUMA information, as inside the GPU
    pool's containers: numa_node = -1) it reports that nothing was bound and the run proceeds unbound."""
    from synthpy_b200 import distributed as D
    before = os.sched_getaffinity(0)
    r = D.bind_to_local_numa(0)
    assert isinstance(r, dict) and r.get("bound") in (False, True)
    if not r["bound"]:
        assert os.sched_getaffinity(0) == before
    else:
        os.sched_setaffinity(0, before)
