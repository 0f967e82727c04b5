"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys and never
loads the product library; our arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_reference_arm_line_and_independence_from_the_product_library():
    # any attempt to load the product library would fail: the path does not exist
    env = dict(os.environ, WRFB200_LIB="/nonexistent/libwrfb200.so")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                        "--steps", "3", "--warmup", "3"], capture_output=True, text=True, cwd=ROOT, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must carry exactly one JSON line"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "advance_mu_t grid-points/s" and d["unit"] == "grid-points/s"
    assert d["steps"] == 3 and d["warmup"] == 3 and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    # the printed ms_per_step is the TIMED one: value x time per step = the points one small step updates
    from oracle import synth_np
    from wrf_model_cuda_sample_b200.advance_mu_t import Grid
    n3, _ = synth_np.updated_points(Grid.from_shape(74, 61, 28, halo=5))
    assert abs(d["value"] * d["ms_per_step"] * 1e-3 / n3 - 1.0) < 1e-6
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "grid-points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.skipif(_have_gpu(), reason="GPU present")
def test_our_arm_refuses_to_run_without_a_gpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "1"],
                       capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.strip().startswith("{")], "no JSON line may be printed"


def _bench(*argv, **kw):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                          cwd=ROOT, timeout=600, **kw)


def _oracle_steps(fields, g, scalars, n):
    from oracle import loader
    for _ in range(n):
        loader.oracle_c(fields, g, scalars)
    return fields


def test_reference_arm_dumps_its_last_step(tmp_path):
    """Wiring of the CPU arm: --dump-outputs writes the seven output fields after the timed steps, --steps and
    --warmup set how many small steps ran, the same arguments give the same files.  The expected values come from
    our C oracle; without oracle/_ref the arm runs that same oracle, so this is no check against the reference
    (the golden vectors are)."""
    from oracle import synth_np
    from tests import cases
    from wrf_model_cuda_sample_b200.advance_mu_t import Grid
    runs = []
    for d in ("a", "b"):
        r = _bench("--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1",
                   "--dump-outputs", str(tmp_path / d))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 2
        runs.append({n: np.load(tmp_path / d / f"{n}.npy") for n in cases.OUTPUTS})
    assert sorted(os.listdir(tmp_path / "a")) == sorted(f"{n}.npy" for n in cases.OUTPUTS)
    g = Grid.from_shape(74, 61, 28, halo=5)
    want = _oracle_steps(synth_np.synth_fields(g), g, cases.SCALARS_12KM, 3)
    for got in runs:
        assert all(got[n].dtype == np.float32 for n in got)
        cases.assert_bit_equal(got, want)


def test_dump_samples_large_fields_at_fixed_positions(tmp_path):
    """A field above its share of the 64 MB budget is cut to one value from each of equal runs of its flattened
    array, at positions that do not change between runs; a smaller field is written whole."""
    import bench
    big = np.arange(3_000_000, dtype=np.float32).reshape(30, 100, 1000)
    fields = {n: np.full((7, 5), i, dtype=np.float32) for i, n in enumerate(bench.OUTPUTS)}
    fields["t"] = big
    bench.dump_outputs(str(tmp_path / "a"), fields)
    bench.dump_outputs(str(tmp_path / "b"), fields)
    a, b = np.load(tmp_path / "a" / "t.npy"), np.load(tmp_path / "b" / "t.npy")
    cap = a.size
    assert a.shape == (cap,) and cap < big.size and np.array_equal(a, b)
    assert np.array_equal(a.astype(np.int64) // (big.size // cap), np.arange(cap))
    assert np.array_equal(np.load(tmp_path / "a" / "mu.npy"), fields["mu"])


@pytest.mark.parametrize("share", [1, 4])
def test_dump_stays_within_64_mb_when_every_field_is_sampled(tmp_path, share):
    """The budget counts whole files, headers included, over all writers of a run (one per rank)."""
    import bench
    big = np.arange(3_000_000, dtype=np.float32).reshape(30, 100, 1000)
    fields = {n: big for n in bench.OUTPUTS}
    for rank in range(share):
        bench.dump_outputs(str(tmp_path), fields, prefix=f"rank{rank}_" if share > 1 else "", share=share)
    files = os.listdir(tmp_path)
    assert len(files) == share * len(bench.OUTPUTS)
    assert all(np.load(tmp_path / f).size < big.size for f in files)
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64_000_000


@pytest.mark.gpu
def test_our_arm_dumps_its_last_step(tmp_path):
    """The timed path's own result: warmup + steps small steps of the device-resident loop, bit for bit the oracle's."""
    import wrf_model_cuda_sample_b200 as wrf
    from tests import cases
    r = _bench("--workload", "tiny", "--steps", "2", "--warmup", "3", "--no-extras", "--no-e2e", "--no-cpu",
               "--no-ref-cuda", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    got = {n: np.load(tmp_path / f"{n}.npy") for n in cases.OUTPUTS}
    g = wrf.Grid.from_shape(74, 61, 28, halo=5)
    want = _oracle_steps(wrf.synth_fields(g), g, cases.SCALARS_12KM, 5)
    cases.assert_bit_equal(got, want)
