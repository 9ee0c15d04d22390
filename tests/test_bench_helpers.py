"""CPU: the parts of bench.py that do not need a GPU -- argument defaults, the CPU-baseline
object, the clock sampler's degraded path and the reference arm's JSON line and output dump."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_defaults_and_cpu_baseline_object(oracle):
    import bench
    old = sys.argv
    sys.argv = ["bench.py"]
    try:
        a = bench.parse_args()
    finally:
        sys.argv = old
    assert a.gpus == 1 and a.warmup >= 3 and a.steps >= 1 and a.recsize == 131072 and a.impl != "reference"
    s = oracle.synth_stream(64, recsize=131072, kind=oracle.PAYLOAD_PCG)
    cpu = bench.cpu_verify_baseline(oracle, s, 2)
    assert cpu["kind"] == "port" and cpu["cores"] == 2 and cpu["unit"] == "GiB/s"
    assert cpu["value"] > 0 and cpu["single_thread_value"] > 0 and "fletcher_4" in cpu["sample"]
    assert cpu["fletcher4"] in bench.SIMD_NAME.values()
    json.dumps(cpu)
    q = bench.cpu_quota()
    assert q is None or q > 0
    assert bench.host_threads() >= 1
    cs = bench.ClockSampler(0)                 # never started: the degraded answer, not an exception
    c = cs.stop()
    assert c["sm_mhz"] is None and c["reasons"]


def test_reference_arm_prints_the_contract_line(tmp_path):
    dump = str(tmp_path / "outputs")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--ref-gib", "0.25", "--dump-outputs", dump], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=280, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"] and d["gpu_launches"] == 0
    # --dump-outputs: the last step's output stream, sampled, as float arrays of at most 64 MB in all
    import numpy as np
    out = {f[:-4]: np.load(os.path.join(dump, f)) for f in os.listdir(dump)}
    assert sorted(out) == ["output_bytes", "output_sample", "output_sample_offsets"]
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    smp, n = out["output_sample"], int(out["output_bytes"][0])
    assert n > 0 and smp.size == out["output_sample_offsets"].size * 65536
    assert smp.min() >= 0 and smp.max() <= 255 and np.all(smp == np.round(smp))


def test_restated_plumbing_pump_pair_moves_the_stream_unchanged():
    """BASELINE.md row B0': tools/pump_pair.c (the reference's two pipes restated in C) between the
    fake zfs children -- SHA-256 at `zfs recv` == SHA-256 at `zfs send`."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_plumbing.py"), "0.03", "cpump"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])["plumbing"]["cpump"]
    assert d["identity"] is True and d["exit_codes"] == [0, 0, 0, 0] and d["stream_gibs"] > 0
