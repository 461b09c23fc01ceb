"""CPU: the reference arm of bench.py (`--impl reference`) -- the reference's own
AsyncEnvPool compiled into oracle/_ref, timed on the host cores -- prints one JSON line with
the keys of our arm's line.  Where oracle/_ref has not been built (it is compiled from a
reference checkout), the arm times the scalar C port of the oracle instead and says so."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line(engine_built):
    built = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libenvpool_ref.so"))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"]
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert "CartPole-v1" in d["config"]["workload"] and "65536" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if built else "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
