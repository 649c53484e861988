"""bench.py's JSON contract on what can run without a GPU: the reference arm (the reference algorithm on the host cores)
on the tiny workload, and the bookkeeping helpers behind the roofline numbers; and what --dump-outputs writes, for the
reference arm and (on a GPU) for the timed paths."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


import pytest


@pytest.mark.parametrize("kind,workload", [("port", "tiny"), ("auto", "tiny"), ("auto", "tiny_3fold")])
def test_reference_arm_prints_one_contract_line(kind, workload):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload,
                          "--steps", "1", "--warmup", "1", "--cpu-sample", "2", "--cpu-kind", kind],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "gblup_fitness_evals_per_sec" and d["unit"] == "evals/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["config"]["workload"] == workload and d["config"]["pop_is"] == "per_gpu"
    from oracle import stage_ref
    have_ref = stage_ref.ref_path() is not None
    assert d["cpu_baseline"]["kind"] == ("reference" if kind == "auto" and have_ref else "port")
    assert d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


def _run_bench(*args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_dumps_the_same_last_step_every_run(tmp_path):
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        out = _run_bench("--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1", "--cpu-sample", "3",
                         "--cpu-kind", "port", "--dump-outputs", str(tmp_path / run))
        assert out.returncode == 0, out.stderr[-2000:]
        assert sorted(os.listdir(tmp_path / run)) == ["fitness.npy"]
        dumps.append(np.load(tmp_path / run / "fitness.npy"))
    assert dumps[0].dtype == np.float64 and dumps[0].shape == (3, 1) and np.all(np.isfinite(dumps[0]))
    assert np.array_equal(dumps[0], dumps[1])
    # the last timed step scored genomes 6..8 of the seeded draw (warmup 1 + steps 2, 3 genomes per step)
    sys.path.insert(0, ROOT)
    import bench
    from oracle import gblup_oracle as O
    from tblup_b200 import synth
    wl = bench.WORKLOADS["tiny"]
    x, y = synth.synth_dataset(wl["n"], wl["m"], h2=bench.H2, seed=0)
    tr, va, _ = synth.split_indices(wl["n"], seed=0)
    flat, off = synth.random_genomes(3 * 3, wl["m"], wl["k"], seed=100)
    want = [O.exact_fitness_rowsets(flat[off[i]:off[i + 1]], [(tr, va)], x, y, bench.H2)[0] for i in range(6, 9)]
    assert np.abs(dumps[0][:, 0] - want).max() < 1e-9


@pytest.mark.gpu
def test_gpu_arm_dumps_what_the_timed_paths_returned(tmp_path):
    """With one timed step both timed paths score the first seeded batch: each dump equals the engine's fitness for it
    and the exact oracle's to the parity bar."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from tblup_b200 import GblupEngine, MODE_AUTO, synth
    out = _run_bench("--workload", "tiny", "--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-sustained-peaks",
                     "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    wl = bench.WORKLOADS["tiny"]
    x, y = synth.synth_dataset(wl["n"], wl["m"], h2=bench.H2, seed=0)
    tr, va, te = synth.split_indices(wl["n"], seed=0)
    flat, off = synth.random_genomes(wl["pop"], wl["m"], wl["k"], seed=1000)
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        eng.set_rowset(0, tr, va)
        eng.set_precision("mixed")
        want = eng.evaluate_packed(flat, off, [0], bench.H2, MODE_AUTO)
    from oracle import gblup_oracle as O
    exact = np.array([O.exact_blup(flat[off[i]:off[i + 1]], tr, va, x, y, bench.H2) for i in range(wl["pop"])])
    for name in ("fitness", "fitness_e2e"):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float64 and got.shape == (wl["pop"], 1), name
        assert np.abs(got - want).max() < 1e-9, name
        assert np.abs(got[:, 0] - exact).max() < bench.PARITY_BAR, name


def test_steps_below_one_are_refused():
    out = _run_bench("--impl", "reference", "--workload", "tiny", "--steps", "0", timeout=60)
    assert out.returncode != 0 and "--steps must be at least 1" in out.stderr


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                          "--gpus", "2", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120,
                         cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_algorithmic_work_formulas():
    sys.path.insert(0, ROOT)
    import bench
    # Cholesky update flops: sum over block columns equals n^3/3 to leading order
    n = 3200
    assert abs(bench.chol_update_flops(n, 64) / (n ** 3 / 3) - 1) < 0.05
    assert abs(bench.chol_update_flops(n, 256) / (n ** 3 / 3) - 1) < 0.15
    # update traffic: 8 B read-modify-write per entry below the first block column + the fp16 row operand
    b = bench.chol_update_bytes(n, 256)
    rmw = sum((n - c0) * min(256, n - c0) * 8 for c0 in range(256, n, 256))
    assert b > rmw and abs(b / 80.2e6 - 1) < 0.01
    # block column formed from int16 cross-products (2 B read + 4 B written per entry), and with t16 the rows below the
    # diagonal block of every full-width block column written as halves (2 + 2 B): the figures quoted in DESIGN.md §5
    assert abs(bench.chol_update_bytes(n, 256, 2) / 70.8e6 - 1) < 0.01
    b16 = bench.chol_update_bytes(n, 256, 2, True)
    below = sum((n - c0 - 256) * 256 for c0 in range(256, n, 256) if c0 + 256 < n)
    assert b16 == bench.chol_update_bytes(n, 256, 2) - 2 * below and abs(b16 / 62.9e6 - 1) < 0.01
