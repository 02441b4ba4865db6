"""bench.py's reference arm (the CPU restatement through `--impl reference`) needs no GPU: its one JSON line must
carry the keys the driver's contract names, with the arm's own value repeated under cpu_baseline and e2e."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--circuit", "synthetic"],
                         capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"].startswith("proofs/sec") and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "threads" in d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_dumps_the_proof_of_its_last_step(tmp_path):
    import numpy as np

    import bench
    from oracle import cref

    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0", "--circuit", "synthetic",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["proofs.npy"]
    got = np.load(tmp_path / "proofs.npy")
    assert got.dtype == np.float32 and got.shape == (1, 1008)
    arrays, _ = bench.build_workload("synthetic")
    srs = cref.srs_from_secret(bench.SRS_POINTS, bench.SRS_X, bench.SRS_G)
    want = cref.CrefProver(bench.LABEL, arrays, srs).prove(bench.blinders_for(1001))  # step 2 of 2
    assert got.astype(np.uint8).tobytes() == want and (got == got.astype(np.uint8)).all()


def test_other_ranks_of_the_reference_arm_do_no_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
