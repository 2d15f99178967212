"""CPU (-m "not gpu"): the reference arm of bench.py runs without a GPU (it times the oracle port
on the host cores) -- check the one-JSON-line contract and its keys on a tiny grid.  GPU: the
outputs --dump-outputs writes for the timed arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "12",
                          "--steps", "1", "--warmup", "1", "--ref-iters", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout                  # exactly one line on stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "iterations/s" and d["value"] > 0
    assert d["dtype"] == "f64" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("CPU-only check")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--grid", "12", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0                           # no CPU fallback: the product path needs the GPU
    assert out.stdout.strip() == ""                      # and never prints a number it did not measure


def test_traffic_stamps_match_the_kernel_sources():
    """profiles/traffic.json holds ncu-measured DRAM bytes per launch; bench.py echoes an entry as
    `roofline.traffic` only while it is stamped with the fingerprint of the device headers its kernel
    class is compiled from.  A header edited after the capture (even a comment) makes the bench line
    report `traffic: null` -- this test says so before the round ends."""
    sys.path.insert(0, ROOT)
    import bench
    from new_cg_variants_b200 import build as b
    t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    assert "pr_fused" in t and "csr_sp_pr" in t
    for cls, ent in t.items():
        assert ent["kernel_sources_sha"] == b.kernel_fingerprint(cls), f"{cls}: captured for other kernel sources"
        assert all(os.path.exists(os.path.join(b.CSRC, f)) for p, lst in b.KERNEL_SOURCES.items() if cls.startswith(p) for f in lst)
    val, note = bench.read_traffic("pr_fused")
    assert val == t["pr_fused"]["dram_bytes_per_launch"] and "ncu" in note
    assert bench.read_traffic("no_such_kernel")[0] is None
    # a class's stamp ignores headers its kernel is not compiled from
    assert b.kernel_fingerprint("pr_fused") != b.kernel_fingerprint("csr_sp_pr") != b.kernel_fingerprint()


def test_dump_outputs_sample_is_fixed_and_other_arms_refuse_it(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    n = bench.DUMP_MAX_ENTRIES + 1000
    x = np.arange(n, dtype=np.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), x)
    sa, sb = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "b" / "x.npy")
    assert sa.dtype == np.float64 and sa.shape == (bench.DUMP_MAX_ENTRIES,)
    assert np.array_equal(sa, sb) and np.all(np.diff(sa) > 0)      # same entries, in index order
    bench.dump_outputs(str(tmp_path / "small"), x[:100])
    assert np.array_equal(np.load(tmp_path / "small" / "x.npy"), x[:100])
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "12",
                          "--dump-outputs", str(tmp_path / "ref")], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and out.stdout.strip() == "" and not (tmp_path / "ref").exists()


@pytest.mark.gpu
def test_dump_outputs_hold_the_solution_of_the_timed_steps(tmp_path):
    """--dump-outputs writes x of the last timed step: bit for bit what a direct Session run of the
    same workload returns, whatever --steps is; --steps sets the number of timed solves."""
    sys.path.insert(0, ROOT)
    import bench
    from new_cg_variants_b200 import Session
    runs = {}
    for steps in (2, 3):
        d = tmp_path / f"steps{steps}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--grid", "12", "--iters", "20",
                              "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert sorted(os.listdir(d)) == ["x.npy"]
        runs[steps] = (json.loads(out.stdout), np.load(d / "x.npy"))
    assert runs[2][0]["steps"] == 2 and runs[3][0]["steps"] == 3
    assert 2 * runs[3][0]["gpu_launches"] == 3 * runs[2][0]["gpu_launches"]
    S, b, x0, x_true, dinv = bench.build_problem(12)
    with Session(S, dinv=dinv) as s:
        s.load_problem(b, x0, None)
        s.run("pr", 21, histories=(), path="auto")
        x = s.fetch(want_hist=False)[0]
    for _, dumped in runs.values():
        assert dumped.dtype == np.float64 and np.array_equal(dumped, x)
