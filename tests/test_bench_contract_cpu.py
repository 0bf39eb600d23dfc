"""CPU: the reference arm of bench.py (`--impl reference`: the reference's CPU path - the unmodified
reference when a checkout is reachable, else the oracle port - timed on the host cores) prints ONE
JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--files", "8",
                          "--seconds", "6", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "audio_seconds_fingerprinted_per_sec"
    assert d["unit"] == "audio-s/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    # the unmodified reference where a checkout is reachable, the oracle port otherwise
    refs = (os.environ.get("AFP_REFERENCE"), os.path.join(ROOT, "baseline", "_ref"))
    want_kind = "reference" if any(d and os.path.isfile(os.path.join(d, "audfprint_analyze.py")) for d in refs) else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["host_cores"]["used"] == d["cpu_baseline"]["cores"]
    assert d["config0"]["cores"] == 1 and d["config0"]["median_s"] > 0 and d["config0"]["runs"] >= 5
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None
