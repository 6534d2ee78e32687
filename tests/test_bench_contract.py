"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) runs the CPU
restatement on the host cores and prints ONE JSON line with the keys of the result.  The product
arm's --steps / --dump-outputs check needs one."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--ref-cells", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1
    for k in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "GDoF/s" and d["value"] > 0 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"]


def test_default_arm_fails_loudly_without_gpu():
    """No CPU fallback: without a CUDA device the product arm must exit non-zero, not print a number."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1",
                        "--cells", "4", "--no-cpu-baseline", "--no-rk4"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not any(l.startswith("{") and '"value"' in l for l in r.stdout.splitlines())


def test_reference_arm_is_independent_of_the_product_library():
    """The CPU arm must not import the product package: it runs with the library path pointing
    nowhere (capi raises on import when libwavefx.so is missing), under torch.distributed.run's
    OMP_NUM_THREADS=1, and still uses the host cores it may run on."""
    env = dict(os.environ, WFX_LIB="/nonexistent/libwavefx.so", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--ref-cells", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["cpu_baseline"]["cores"] == max(1, min(len(os.sched_getaffinity(0)), 32))


def _bench(args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])


def _oracle_kv(cells, P, perturb, x):
    """kv = M^-1 (-c0^2 K x) on bench.py's cells^3 mesh, by the CPU oracle"""
    import numpy as np
    sys.path.insert(0, ROOT)
    from oracle import oracle, refmesh
    mesh = refmesh.box(cells, P, (0.1, 0.1, 0.1), perturb=perturb)
    G, detJ = oracle.precompute_geometric_data(mesh, P)
    m, b = np.zeros(mesh.ndofs), np.zeros(mesh.ndofs)
    oracle.mass_apply(mesh, P, detJ, np.ones(mesh.ndofs), m)
    oracle.stiffness_apply(mesh, P, G, x, b, dense=False)
    return b / m


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs DIR: the reference arm writes the kv of its last timed step to DIR/kv.npy."""
    import numpy as np
    d = _bench(["--impl", "reference", "--steps", "2", "--warmup", "0", "--ref-cells", "3",
                "--dump-outputs", str(tmp_path)])
    assert d["steps"] == 2
    kv = np.load(tmp_path / "kv.npy")
    want = _oracle_kv(3, 4, 0.0, np.random.default_rng(42).standard_normal(kv.size))
    assert kv.dtype == np.float64 and kv.shape == want.shape
    assert np.linalg.norm(kv - want) <= 1e-12 * np.linalg.norm(want)


def test_dump_sample_is_fixed_and_bounded():
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = bench.DUMP_MAX_VALUES
    assert bench.dump_sample_index(n) is None
    a, b = bench.dump_sample_index(n + 5), bench.dump_sample_index(n + 5)
    assert np.array_equal(a, b) and a.size == n and np.all(np.diff(a) > 0) and a[-1] < n + 5
    assert n * 8 <= 32 * 2 ** 20  # one float64 array stays far below the 64 MB a dump may take


@pytest.mark.gpu
def test_b200_arm_dumps_its_last_timed_step(tmp_path):
    """--steps K: the timed windows hold K applies in all, and their device time grows with K (45 applies take
    well over 5x the time of 3).  --dump-outputs writes the kv of the timed applies (every apply gets the same
    seeded x, so the last one's kv is also every one's): it equals the oracle's kv on that x and is the same,
    bit for bit, for another number of steps."""
    import numpy as np
    import torch
    common = ["--cells", "4", "--warmup", "1", "--no-cpu-baseline", "--no-rk4", "--no-strong", "--no-affine",
              "--sustain-s", "0"]
    d3 = _bench([*common, "--steps", "3", "--dump-outputs", str(tmp_path / "a")])
    assert d3["steps"] == 3 and d3["window_steps"] == [3]
    d = _bench([*common, "--steps", "45", "--dump-outputs", str(tmp_path / "b")])
    assert d["steps"] == 45 and d["window_steps"] == [23, 22]
    assert 5 * sum(d3["windows_ms"]) < sum(d["windows_ms"]) < 45 * sum(d3["windows_ms"])
    kv = np.load(tmp_path / "a" / "kv.npy")
    assert kv.dtype == np.float64 and np.array_equal(kv, np.load(tmp_path / "b" / "kv.npy"))
    g = torch.Generator(device="cuda:0").manual_seed(42)
    x = torch.randn(kv.size, dtype=torch.float64, device="cuda:0", generator=g).cpu().numpy()
    want = _oracle_kv(4, 4, 0.15, x)
    assert np.linalg.norm(kv - want) <= 1e-12 * np.linalg.norm(want)


def test_oracle_mesh_generator_matches_the_product_generator(wfx):
    """oracle/refmesh.py (numpy + the oracle's permutation) and wave-fenics_b200/mesh.py (libwavefx's
    permutation) are independent and produce the same DOLFINx-layout arrays."""
    import numpy as np
    sys.path.insert(0, ROOT)
    from oracle import refmesh
    for n, P, pert in (((3, 4, 5), 3, 0.1), (4, 4, 0.15), (2, 7, 0.0)):
        a = wfx.create_box_hex(n, P, (0.1, 0.2, 0.3), perturb=pert)
        b = refmesh.box(n, P, (0.1, 0.2, 0.3), perturb=pert)
        assert np.array_equal(a.x, b.x) and np.array_equal(a.xdofs, b.xdofs) and np.array_equal(a.dofmap, b.dofmap)
        assert a.ndofs == b.ndofs
