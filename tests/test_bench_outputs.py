"""bench.py --dump-outputs: the proof of the last timed step lands in DIR/proof.npy, and it is the proof of the seeded batch."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def run_bench(args, out_dir):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--num-tx", "2", "--dump-outputs", str(out_dir)] + args,
                         capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(ln) for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return lines[0]


def oracle_proof(csg, oracle):
    trace, pub = csg.TransactionBatch(seed=1000, num_tx=2).transaction_trace()      # bench.py's batch of rank 0
    return oracle.prove(oracle.AIR_TRANSACTION, trace, pub, oracle.options())


def load_proof(path):
    got = np.load(path)
    assert got.dtype == np.float32 and got.ndim == 1
    return got.astype(np.uint8).tobytes()


def test_reference_arm_dumps_its_last_proof(csg, oracle, tmp_path):
    run_bench(["--impl", "reference", "--steps", "1", "--warmup", "0"], tmp_path)
    assert load_proof(tmp_path / "proof.npy") == oracle_proof(csg, oracle)


@pytest.mark.gpu
def test_gpu_bench_dumps_the_proof_of_its_last_timed_step(csg, oracle, tmp_path):
    line = run_bench(["--steps", "2", "--warmup", "1", "--no-cpu-baseline"], tmp_path)
    assert line["steps"] == 2 and line["n_gpus"] == 1
    assert load_proof(tmp_path / "proof.npy") == oracle_proof(csg, oracle)
    assert sorted(p.name for p in tmp_path.iterdir()) == ["proof.npy"]
