"""bench.py --dump-outputs on the GPU path: the proofs of the last timed step of every timed region, one per proof
in flight, equal the CPU restatement's proofs of the same circuit under the same seeded blinders."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_proofs_of_its_last_timed_step(tmp_path):
    import numpy as np

    import bench
    from oracle import cref

    inflight, steps = 2, 2
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--inflight", str(inflight), "--steps", str(steps), "--warmup", "0",
                          "--no-cpu-baseline", "--no-msm-sweep", "--no-proof20", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    names = ["proofs", "proofs_e2e", "proofs_e2e_with_synthesis"]
    assert sorted(os.listdir(tmp_path)) == [n + ".npy" for n in names]
    dumps = [np.load(tmp_path / (n + ".npy")) for n in names]
    for d in dumps:
        assert d.dtype == np.float32 and d.shape == (inflight, 1008)
        assert (d == dumps[0]).all()  # every region's last step proves with the same blinders
    arrays, _ = bench.build_workload("bench")
    srs = cref.srs_from_secret(bench.SRS_POINTS, bench.SRS_X, bench.SRS_G)
    prover = cref.CrefProver(bench.LABEL, arrays, srs)
    last = 1000 + steps - 1
    for slot in range(inflight):
        assert dumps[0][slot].astype(np.uint8).tobytes() == prover.prove(bench.blinders_for(last * inflight + slot)), slot
